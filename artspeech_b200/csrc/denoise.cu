// Noise reduction for voice enrollment (artspeech_b200/frontend.py step 2b states the semantics; header: as_denoise):
// a stationary-noise spectral suppressor on 24 kHz rows, before the trim and the log-mel.  Three launches:
//   1. STFT: grid (8 frames, row), one warp per frame.  The centred, zero-padded, Hann-windowed 512-sample frame goes
//      to shared memory in bit-reversed order, fft_radix2<9, 32> (fft.cuh) transforms it, and bins 0 .. 256 go to the
//      workspace's X plane.
//   2. Noise profile and gain: grid (32 consecutive bins, row), 8 warps.  The r-th smallest P of each bin over the
//      row's frames is found by a radix select on the fp32 bit patterns (P >= 0, so they order as unsigned integers):
//      four 8-bit passes, each a shared-memory histogram of integer counts per (digit, bin) over the frames whose
//      higher digits match, read coalesced (lane = bin, warps stride the frames).  The counts do not depend on the
//      order the frames are counted in, so the selected value does not depend on scheduling.  Then warp 0 runs the
//      decision-directed gain as one lane per bin: a sequential fp64 scan over the frames whose loop-carried chain
//      holds two multiplies, two adds and one divide; gamma and max(gamma - 1, 0) of the next frames, and the loads
//      of the frames after those, are issued off that chain.
//   3. Synthesis: grid (13 blocks of 128 output samples, row), one warp per covering frame (16).  Each warp forms
//      G X as a Hermitian 512-point spectrum (imaginary parts of the DC and Nyquist bins dropped, as irfft does),
//      transforms it with fft_radix2<9, 32> and the conjugate twiddle table, and the CTA gathers the <= 4 windowed
//      frames covering each sample in ascending frame order.  Samples at and beyond n are written as zeros.
// No atomics on floating-point data, no host synchronisation; every value of a row follows from its own samples and
// its own frame count, so the output does not depend on B, S, the row strides or the batch-mates.
#include <cmath>

#include "common.cuh"
#include "fft.cuh"

namespace asb {

constexpr int kDnN = 512, kDnLog2 = 9, kDnHop = 128, kDnBins = AS_DENOISE_BINS;
constexpr int kDnStftFrames = 8, kDnStftThreads = 32 * kDnStftFrames;
constexpr int kDnGroup = 32, kDnGainThreads = 256, kDnGainWarps = kDnGainThreads / 32;
constexpr int kDnGroups = (kDnBins + kDnGroup - 1) / kDnGroup;
constexpr int kDnScanChunk = 8;
constexpr int kDnSynBlocks = 13, kDnSynFrames = kDnSynBlocks + 3, kDnSynThreads = 32 * kDnSynFrames;
constexpr size_t kDnSynSmem = (size_t)kDnSynFrames * kDnN * sizeof(float2);
static_assert(kDnSynFrames == 16, "one warp per frame covering 13 hops of output");
static_assert(kDnGainWarps == 8, "the digit partial sums assume 8 warps of 32 digits");

__device__ __forceinline__ float dn_power(float2 x) { return __fadd_rn(__fmul_rn(x.x, x.x), __fmul_rn(x.y, x.y)); }

__device__ __forceinline__ int dn_len(const int* lens, int b, int S) { return lens ? min(max(lens[b], 0), S) : S; }

// Launch 1: X[b, f, k] for f < F_b = 1 + n_b / 128.
__global__ void __launch_bounds__(kDnStftThreads) denoise_stft_kernel(
    const float* __restrict__ y, long long y_ld, int S, const int* __restrict__ lens, const float* __restrict__ window,
    const float2* __restrict__ twiddle, float2* __restrict__ X, int F_max) {
  pdl_wait();
  __shared__ float2 buf[kDnStftFrames][kDnN];
  __shared__ float2 tw[kDnN / 2];
  const int b = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n = dn_len(lens, b, S), F = 1 + n / kDnHop;
  if ((int)blockIdx.x * kDnStftFrames >= F) return;      // the whole CTA is beyond this row's frames
  for (int i = tid; i < kDnN / 2; i += kDnStftThreads) tw[i] = twiddle[i];
  const int f = blockIdx.x * kDnStftFrames + warp;
  const float* yb = y + (long long)b * y_ld;
  const int s0 = f * kDnHop - kDnN / 2;
  for (int i = lane; i < kDnN; i += 32) {
    const int s = s0 + i;
    const float v = (f < F && s >= 0 && s < n) ? __fmul_rn(yb[s], window[i]) : 0.f;
    buf[warp][fft_slot<kDnLog2>(i)] = make_float2(v, 0.f);
  }
  __syncthreads();
  fft_radix2<kDnLog2, 32>(buf[warp], tw, lane);
  if (f < F) {
    float2* Xf = X + ((long long)b * F_max + f) * kDnBins;
    for (int k = lane; k < kDnBins; k += 32) Xf[k] = buf[warp][k];
  }
}

// Launch 2: lambda[b, k] and G[b, f, k].
__global__ void __launch_bounds__(kDnGainThreads) denoise_gain_kernel(
    const float2* __restrict__ X, int F_max, int S, const int* __restrict__ lens, double c, double g_min,
    double alpha, double one_minus_alpha, double* __restrict__ lambda, float* __restrict__ G) {
  pdl_wait();
  __shared__ unsigned hist[256][kDnGroup];
  __shared__ unsigned part[kDnGainWarps][kDnGroup];
  __shared__ unsigned prefix_s[kDnGroup], rank_s[kDnGroup];
  const int b = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int k = blockIdx.x * kDnGroup + lane;
  const bool valid = k < kDnBins;
  const int n = dn_len(lens, b, S), F = 1 + n / kDnHop;
  const float2* Xb = X + (long long)b * F_max * kDnBins + (valid ? k : 0);
  if (tid < kDnGroup) { prefix_s[tid] = 0u; rank_s[tid] = (unsigned)(F / 10); }
#pragma unroll 1
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int i = tid; i < 256 * kDnGroup; i += kDnGainThreads) (&hist[0][0])[i] = 0u;
    __syncthreads();
    const unsigned pre = prefix_s[lane], mask = shift == 24 ? 0u : 0xFFFFFFFFu << (shift + 8);
    if (valid) {
      for (int f = warp; f < F; f += kDnGainWarps) {
        const unsigned u = __float_as_uint(dn_power(Xb[(long long)f * kDnBins]));
        if ((u & mask) == pre) atomicAdd(&hist[(u >> shift) & 255u][lane], 1u);
      }
    }
    __syncthreads();
    unsigned s = 0;
#pragma unroll 8
    for (int d = 0; d < 32; ++d) s += hist[32 * warp + d][lane];
    part[warp][lane] = s;
    __syncthreads();
    if (warp == 0) {                                       // the digit holding the rank-th key of this bin
      unsigned r = rank_s[lane];
      int w = 0;
      while (w < kDnGainWarps - 1 && r >= part[w][lane]) r -= part[w++][lane];
      int d = 32 * w;
      while (d < 32 * w + 31 && r >= hist[d][lane]) r -= hist[d++][lane];
      prefix_s[lane] |= (unsigned)d << shift;
      rank_s[lane] = r;
    }
    __syncthreads();
  }
  if (warp != 0 || !valid) return;
  const double lam = fmax(1e-20, __ddiv_rn((double)__uint_as_float(prefix_s[lane]), c));
  lambda[(long long)b * kDnBins + k] = lam;
  float* Gb = G + (long long)b * F_max * kDnBins + k;
  float2 cur[kDnScanChunk], nxt[kDnScanChunk];
#pragma unroll
  for (int e = 0; e < kDnScanChunk; ++e) cur[e] = e < F ? Xb[(long long)e * kDnBins] : make_float2(0.f, 0.f);
  double A = 0.0;
  for (int f0 = 0; f0 < F; f0 += kDnScanChunk) {
#pragma unroll
    for (int e = 0; e < kDnScanChunk; ++e) {              // the next chunk's loads, in flight during this chunk
      const int f = f0 + kDnScanChunk + e;
      nxt[e] = f < F ? Xb[(long long)f * kDnBins] : make_float2(0.f, 0.f);
    }
    double gam[kDnScanChunk], m[kDnScanChunk];
#pragma unroll
    for (int e = 0; e < kDnScanChunk; ++e) {
      gam[e] = __ddiv_rn((double)dn_power(cur[e]), lam);
      m[e] = fmax(__dadd_rn(gam[e], -1.0), 0.0);
    }
#pragma unroll
    for (int e = 0; e < kDnScanChunk; ++e) {
      const int f = f0 + e;
      if (f < F) {
        const double xi = f == 0 ? m[e] : __dadd_rn(__dmul_rn(alpha, A), __dmul_rn(one_minus_alpha, m[e]));
        const double W = __ddiv_rn(xi, __dadd_rn(1.0, xi));
        A = __dmul_rn(__dmul_rn(W, W), gam[e]);
        Gb[(long long)f * kDnBins] = __double2float_rn(fmax(W, g_min));
      }
    }
#pragma unroll
    for (int e = 0; e < kDnScanChunk; ++e) cur[e] = nxt[e];
  }
}

// Launch 3: out[b, t] for t in the CTA's 13 hops.
__global__ void __launch_bounds__(kDnSynThreads) denoise_synth_kernel(
    const float2* __restrict__ X, const float* __restrict__ G, int F_max, int S, const int* __restrict__ lens,
    const float* __restrict__ window, const float2* __restrict__ itwiddle, float* __restrict__ out, long long out_ld) {
  pdl_wait();
  extern __shared__ float2 fbuf[];                         // [kDnSynFrames][kDnN]
  __shared__ float2 tw[kDnN / 2];
  __shared__ float win[kDnN];
  const int b = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n = dn_len(lens, b, S), F = 1 + n / kDnHop;
  const int m0 = blockIdx.x * kDnSynBlocks, t0 = m0 * kDnHop, t1 = min(S, t0 + kDnSynBlocks * kDnHop);
  float* ob = out + (long long)b * out_ld;
  if (t0 >= n) {
    for (int t = t0 + tid; t < t1; t += kDnSynThreads) ob[t] = 0.f;
    return;
  }
  for (int i = tid; i < kDnN / 2; i += kDnSynThreads) tw[i] = itwiddle[i];
  for (int i = tid; i < kDnN; i += kDnSynThreads) win[i] = window[i];
  const int fa = max(0, m0 - 1), f = fa + warp;            // frames m0 - 1 .. m0 + 14 cover the CTA's samples
  float2* buf = fbuf + warp * kDnN;
  if (f < F && f <= m0 + kDnSynBlocks + 1) {
    const float2* Xf = X + ((long long)b * F_max + f) * kDnBins;
    const float* Gf = G + ((long long)b * F_max + f) * kDnBins;
    for (int k = lane; k < kDnBins; k += 32) {
      const float2 x = Xf[k];
      const float g = Gf[k];
      float2 v = make_float2(__fmul_rn(g, x.x), __fmul_rn(g, x.y));
      if (k == 0 || k == kDnN / 2) v.y = 0.f;
      buf[fft_slot<kDnLog2>(k)] = v;
      if (k > 0 && k < kDnN / 2) buf[fft_slot<kDnLog2>(kDnN - k)] = make_float2(v.x, -v.y);
    }
  } else {
    for (int i = lane; i < kDnN; i += 32) buf[i] = make_float2(0.f, 0.f);
  }
  __syncthreads();
  fft_radix2<kDnLog2, 32>(buf, tw, lane);
  for (int t = t0 + tid; t < t1; t += kDnSynThreads) {
    float v = 0.f;
    if (t < n) {
      const int f_lo = t >= kDnN / 2 ? (t - kDnN / 2) / kDnHop + 1 : 0;
      const int f_hi = min(F - 1, (t + kDnN / 2) / kDnHop);
      float num = 0.f, den = 0.f;
      for (int ff = f_lo; ff <= f_hi; ++ff) {
        const int j = t - ff * kDnHop + kDnN / 2;
        const float w = win[j];
        num = fmaf(w, fbuf[(ff - fa) * kDnN + j].x, num);
        den = fmaf(w, w, den);
      }
      v = (num * (1.f / kDnN)) / den;
    }
    ob[t] = v;
  }
}

static size_t dn_align(size_t v) { return (v + 255) & ~(size_t)255; }

static size_t dn_plane(int32_t B, int32_t S, size_t elem) {
  return dn_align((size_t)B * (size_t)(1 + S / kDnHop) * kDnBins * elem);
}

}  // namespace asb

using namespace asb;

extern "C" size_t as_denoise_workspace_bytes(int32_t B, int32_t S) {
  if (B <= 0 || S < 0) return 0;
  return dn_plane(B, S, sizeof(float2)) + dn_plane(B, S, sizeof(float)) +
         dn_align((size_t)B * kDnBins * sizeof(double));
}

extern "C" int as_denoise(const float* y, int64_t y_ld, int32_t B, int32_t S, const int32_t* lens, double reduction_db,
                          const float* window, const float* twiddle, const float* itwiddle, double c, double g_min,
                          double alpha, double one_minus_alpha, void* workspace, size_t workspace_bytes, float* out,
                          int64_t out_ld, void* stream) {
  if (B == 0 || S == 0) return AS_OK;
  ASB_REQUIRE(B > 0 && B <= 65535 && S > 0 && y && out && y_ld >= S && out_ld >= S && window && twiddle && itwiddle,
              AS_ERR_SHAPE, "as_denoise: bad argument");
  ASB_REQUIRE((const void*)y != (const void*)out, AS_ERR_SHAPE, "as_denoise: out must not alias y");
  ASB_REQUIRE(reduction_db >= 0.0 && reduction_db <= 60.0, AS_ERR_SHAPE,
              "as_denoise: reduction_db must be in [0, 60], got %g", reduction_db);
  ASB_REQUIRE(std::fabs(g_min - std::pow(10.0, -reduction_db / 20.0)) <= 1e-12 * g_min, AS_ERR_SHAPE,
              "as_denoise: g_min %.17g is not 10^(-reduction_db / 20) for reduction_db %g", g_min, reduction_db);
  ASB_REQUIRE(c > 0.0 && std::isfinite(c) && alpha > 0.0 && alpha < 1.0 && one_minus_alpha == 1.0 - alpha,
              AS_ERR_SHAPE, "as_denoise: bad constants (c > 0, 0 < alpha < 1, one_minus_alpha = 1 - alpha)");
  ASB_REQUIRE(workspace && workspace_bytes >= as_denoise_workspace_bytes(B, S), AS_ERR_WORKSPACE,
              "as_denoise: workspace of %zu bytes, %zu needed", workspace_bytes, as_denoise_workspace_bytes(B, S));
  ASB_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, AS_ERR_ALIGN,
              "as_denoise: the workspace must be 256-byte aligned");
  if (int rc = check_arch()) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int F_max = 1 + S / kDnHop;
  char* ws = static_cast<char*>(workspace);
  float2* X = reinterpret_cast<float2*>(ws);
  float* G = reinterpret_cast<float*>(ws + dn_plane(B, S, sizeof(float2)));
  double* lambda = reinterpret_cast<double*>(ws + dn_plane(B, S, sizeof(float2)) + dn_plane(B, S, sizeof(float)));
  const float2* tw = reinterpret_cast<const float2*>(twiddle);
  ASB_CUDA(launch_k(denoise_stft_kernel, dim3((unsigned)((F_max + kDnStftFrames - 1) / kDnStftFrames), (unsigned)B),
                    dim3(kDnStftThreads), 0, st, y, (long long)y_ld, (int)S, lens, window, tw, X, F_max));
  ASB_CUDA(launch_k(denoise_gain_kernel, dim3((unsigned)kDnGroups, (unsigned)B), dim3(kDnGainThreads), 0, st,
                    (const float2*)X, F_max, (int)S, lens, c, g_min, alpha, one_minus_alpha, lambda, G));
  ASB_SMEM_OPT_IN((int)kDnSynSmem, denoise_synth_kernel);
  const int n_tiles = (S + kDnSynBlocks * kDnHop - 1) / (kDnSynBlocks * kDnHop);
  ASB_CUDA(launch_k(denoise_synth_kernel, dim3((unsigned)n_tiles, (unsigned)B), dim3(kDnSynThreads), kDnSynSmem, st,
                    (const float2*)X, (const float*)G, F_max, (int)S, lens, window,
                    reinterpret_cast<const float2*>(itwiddle), out, (long long)out_ld));
  return AS_OK;
}
