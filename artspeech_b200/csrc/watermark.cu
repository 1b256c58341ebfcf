// Synthesis watermark (artspeech_b200/audio.py, header: as_watermark_embed / as_watermark_detect; the detector's input
// decoder as_audio_decode is in audio_in.cu):
// a keyed, band-limited, periodic spread-spectrum pattern added to the vocoder's 24 kHz waveform under its own
// envelope, and a detector that finds it at 8 kHz at any circular lag (so cropped excerpts need no search).
//
// Embed: one launch, grid (tile of 32 frames of 240 samples, utterance).  A CTA stages its tile plus one frame of
// halo on each side (16-byte loads, zero at and beyond n), computes the RMS of those 34 frames (one warp per frame,
// lane-strided squares then a butterfly: the same order in every CTA, so a frame shared by two tiles has the same
// bits in both), and writes y = x + (alpha e(t)) c[t mod 12288] with 16-byte pattern loads (L2-resident: 48 KB read
// by every CTA) and 16-byte stores, zeros beyond n.
//
// Detect: two launches.
//   1. grid (period of 4096 samples, utterance), 512 threads: frame RMS of the 80-sample frames covering the period,
//      envelope-normalised samples into shared memory in bit-reversed order, a 4096-point fp32 FFT (fft.cuh), and
//      the 1587 in-band bins written to the workspace.
//   2. one CTA per utterance: A(k) and S(k) summed over the utterance's periods in index order, G = A / S, then for
//      each of the three patterns the real part of sum_k G(k) e^{-j phi_i(k)} e^{j 2 pi k tau / 4096} at every lag,
//      as one forward FFT of the conjugated spectrum; argmax and RMS of r_0 and the two symbol searches are
//      reductions of a fixed shape (per-thread strided, warp butterfly, warps in index order).
// No atomics, no host synchronisation, and every sum's shape depends only on the utterance's own length, so the
// results do not depend on B, S, the row strides or the batch-mates.
#include "common.cuh"
#include "fft.cuh"

namespace asb {

constexpr int kWmThreads = 256;
constexpr int kEmbHop = 240, kEmbFrames = 32, kEmbTile = kEmbHop * kEmbFrames;   // 7680 samples a CTA
constexpr int kEmbWin = kEmbTile + 2 * kEmbHop;                                  // staged: tile + halo frames
constexpr int kDetHop = 80, kDetLog2 = 12, kDetN = 1 << kDetLog2, kDetThreads = 512;
constexpr int kDetEnv = 64;                              // frames covering a period (at most 54)
static_assert(AS_WM_PERIOD == kDetN, "detection period");
static_assert(AS_WM_PERIOD_24K % 4 == 0 && kEmbTile % 4 == 0 && kEmbHop % 4 == 0, "16-byte access");

// e(t) of hop H from the frame RMS values env[f - fbase]: linear between the centres H f + (H - 1) / 2, held before
// the first and after the last (nf frames).  The caller guarantees the frames it reads are in env.
template <int H>
__device__ __forceinline__ float wm_env_at(const float* env, int fbase, int t, int nf) {
  const int u = 2 * t - (H - 1);                         // 2 (t - centre_0)
  if (u <= 0) return env[-fbase];
  const int f = u / (2 * H);
  if (f >= nf - 1) return env[nf - 1 - fbase];
  const float w = (float)(u - 2 * H * f) / (float)(2 * H);
  const float a = env[f - fbase], b = env[f + 1 - fbase];
  return fmaf(w, b - a, a);
}

// RMS of frame (hop H) from its H samples s(i), one warp: lane-strided fma of squares, then a butterfly.
template <int H, typename Ld>
__device__ __forceinline__ float wm_frame_rms(Ld s, int lane) {
  float acc = 0.f;
#pragma unroll
  for (int i = lane; i < H; i += 32) {
    const float v = s(i);
    acc = fmaf(v, v, acc);
  }
  return sqrtf(warp_sum(acc) / (float)H);
}

__global__ void __launch_bounds__(kWmThreads) wm_embed_kernel(
    const float* __restrict__ x, long long x_ld, int S, const int* __restrict__ lens,
    const float* __restrict__ pattern, float alpha, float* __restrict__ out, long long out_ld, int vec_in,
    int vec_out) {
  pdl_wait();
  __shared__ __align__(16) float xs[kEmbWin];
  __shared__ float env[kEmbFrames + 2];
  const int b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int t0 = blockIdx.x * kEmbTile;
  const int nt = min(kEmbTile, S - t0);                 // outputs of this tile
  const int n = lens ? min(max(lens[b], 0), S) : S;
  const float* xb = x + (long long)b * x_ld;
  float* ob = out + (long long)b * out_ld;
  if (t0 < n) {
    const int w0 = t0 - kEmbHop;
    for (int q = tid; q < kEmbWin / 4; q += kWmThreads) {
      const int i = w0 + 4 * q;
      float4 v;
      if (vec_in && i >= 0 && i + 3 < n) {
        v = __ldg(reinterpret_cast<const float4*>(xb + i));
      } else {
        v.x = i >= 0 && i < n ? xb[i] : 0.f;
        v.y = i + 1 >= 0 && i + 1 < n ? xb[i + 1] : 0.f;
        v.z = i + 2 >= 0 && i + 2 < n ? xb[i + 2] : 0.f;
        v.w = i + 3 >= 0 && i + 3 < n ? xb[i + 3] : 0.f;
      }
      reinterpret_cast<float4*>(xs)[q] = v;
    }
    __syncthreads();
    const int F0 = t0 / kEmbHop, nf = (n + kEmbHop - 1) / kEmbHop;
    for (int j = warp; j < kEmbFrames + 2; j += kWmThreads / 32) {
      const float* fr = xs + j * kEmbHop;               // frame F0 - 1 + j (zeros outside [0, n))
      const float e = wm_frame_rms<kEmbHop>([fr](int i) { return fr[i]; }, lane);
      if (lane == 0) env[j] = e;
    }
    __syncthreads();
    for (int q = tid; 4 * q < nt; q += kWmThreads) {
      const int t = t0 + 4 * q;
      const float4 c = __ldg(reinterpret_cast<const float4*>(pattern + t % AS_WM_PERIOD_24K));
      const float4 xv = reinterpret_cast<const float4*>(xs + kEmbHop)[q];
      const float cc[4] = {c.x, c.y, c.z, c.w}, xx[4] = {xv.x, xv.y, xv.z, xv.w};
      float y[4];
#pragma unroll
      for (int e = 0; e < 4; ++e)
        y[e] = t + e < n ? fmaf(alpha * wm_env_at<kEmbHop>(env, F0 - 1, t + e, nf), cc[e], xx[e]) : 0.f;
      if (vec_out && 4 * q + 3 < nt) {
        *reinterpret_cast<float4*>(ob + t) = make_float4(y[0], y[1], y[2], y[3]);
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (4 * q + e < nt) ob[t + e] = y[e];
      }
    }
  } else {
    for (int i = tid; i < nt; i += kWmThreads) ob[t0 + i] = 0.f;
  }
}

// Launch 1: the in-band spectrum of each period of the envelope-normalised utterance.
__global__ void __launch_bounds__(kDetThreads) wm_spectra_kernel(
    const float* __restrict__ x, long long x_ld, int S, const int* __restrict__ lens,
    const float2* __restrict__ twiddle, float2* __restrict__ ws, int nper_max) {
  pdl_wait();
  __shared__ float2 buf[kDetN];
  __shared__ float env[kDetEnv];
  const int p = blockIdx.x, b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = lens ? min(max(lens[b], 0), S) : S;
  if (p >= (n + kDetN - 1) / kDetN) return;             // beyond the utterance: not read by launch 2
  const float* xb = x + (long long)b * x_ld;
  const int t0 = p * kDetN, nf = (n + kDetHop - 1) / kDetHop;
  const int f_lo = max(0, (2 * t0 - (kDetHop - 1)) / (2 * kDetHop));
  const int f_hi = min(nf - 1, (2 * (t0 + kDetN - 1) - (kDetHop - 1)) / (2 * kDetHop) + 1);
  for (int j = warp; j <= f_hi - f_lo; j += kDetThreads / 32) {
    const int s0 = (f_lo + j) * kDetHop;
    const float e = wm_frame_rms<kDetHop>([=](int i) { return s0 + i < n ? xb[s0 + i] : 0.f; }, lane);
    if (lane == 0) env[j] = e;
  }
  __syncthreads();
  for (int i = tid; i < kDetN; i += kDetThreads) {
    const int t = t0 + i;
    float z = 0.f;
    if (t < n) {
      const float e = wm_env_at<kDetHop>(env, f_lo, t, nf);
      if (e >= 1e-4f) z = xb[t] / e;
    }
    buf[fft_slot<kDetLog2>(i)] = make_float2(z, 0.f);
  }
  __syncthreads();
  fft_radix2<kDetLog2, kDetThreads>(buf, twiddle, tid);
  float2* w = ws + ((long long)b * nper_max + p) * AS_WM_BINS_LD;
  for (int k = tid; k < AS_WM_BINS; k += kDetThreads) w[k] = buf[AS_WM_K_LO + k];
}

// Largest v, lowest index on ties, across a warp (every lane gets the result).
__device__ __forceinline__ void wm_warp_argmax(float& v, int& i) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int oi = __shfl_xor_sync(0xffffffffu, i, o);
    if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
  }
}

// Launch 2: whitening, the three correlations and the decisions, one CTA per utterance.
__global__ void __launch_bounds__(kDetThreads) wm_correlate_kernel(
    const float2* __restrict__ ws, int nper_max, int S, const int* __restrict__ lens,
    const float2* __restrict__ spectra, const float2* __restrict__ twiddle, float threshold,
    float* __restrict__ score, int* __restrict__ lag, int* __restrict__ message, unsigned char* __restrict__ detected) {
  pdl_wait();
  __shared__ float2 buf[kDetN];
  __shared__ float2 G[AS_WM_BINS];
  __shared__ float red_v[kDetThreads / 32], red_s[kDetThreads / 32];
  __shared__ int red_i[kDetThreads / 32];
  __shared__ int tau_s;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = lens ? min(max(lens[b], 0), S) : S;
  const int nper = (n + kDetN - 1) / kDetN;
  const float2* wb = ws + (long long)b * nper_max * AS_WM_BINS_LD;
  for (int k = tid; k < AS_WM_BINS; k += kDetThreads) {
    float ar = 0.f, ai = 0.f, s = 0.f;
    for (int p = 0; p < nper; ++p) {
      const float2 z = wb[(long long)p * AS_WM_BINS_LD + k];
      ar += z.x;
      ai += z.y;
      s = fmaf(z.y, z.y, fmaf(z.x, z.x, s));
    }
    G[k] = s > 0.f ? make_float2(ar / s, ai / s) : make_float2(0.f, 0.f);
  }
  float sc = 0.f;
  int tau = 0, sym[2] = {0, 0};
  for (int pat = 0; pat < 3; ++pat) {
    __syncthreads();                                     // G complete; the previous transform is consumed
    const float2* sp = spectra + pat * AS_WM_BINS_LD;
    for (int m = tid; m < kDetN; m += kDetThreads) {
      float2 v = make_float2(0.f, 0.f);
      if (m >= AS_WM_K_LO && m < AS_WM_K_LO + AS_WM_BINS) {
        const float2 g = G[m - AS_WM_K_LO], e = sp[m - AS_WM_K_LO];
        v = make_float2(g.x * e.x - g.y * e.y, -(g.x * e.y + g.y * e.x));   // conj(G e^{-j phi})
      }
      buf[fft_slot<kDetLog2>(m)] = v;
    }
    __syncthreads();
    fft_radix2<kDetLog2, kDetThreads>(buf, twiddle, tid);   // buf[tau].x = r_pat[tau]
    float best = -1.f, ss = 0.f;
    int bi = 0;
    if (pat == 0) {
#pragma unroll
      for (int j = 0; j < kDetN / kDetThreads; ++j) {
        const float r = buf[tid + j * kDetThreads].x;
        ss = fmaf(r, r, ss);
        if (fabsf(r) > best) { best = fabsf(r); bi = tid + j * kDetThreads; }
      }
      ss = warp_sum(ss);
    } else if (tid < AS_WM_SYMBOLS) {
      best = fabsf(buf[(tau + (kDetN / AS_WM_SYMBOLS) * tid) & (kDetN - 1)].x);
      bi = tid;
    }
    wm_warp_argmax(best, bi);
    if (lane == 0) { red_v[warp] = best; red_i[warp] = bi; red_s[warp] = ss; }
    __syncthreads();
    if (tid == 0) {
      float v = red_v[0], s = red_s[0];
      int i = red_i[0];
      for (int w = 1; w < kDetThreads / 32; ++w) {
        if (red_v[w] > v || (red_v[w] == v && red_i[w] < i)) { v = red_v[w]; i = red_i[w]; }
        s += red_s[w];
      }
      if (pat == 0) {
        const float ms = s / (float)kDetN;
        sc = ms > 0.f ? v / sqrtf(ms) : 0.f;
        tau_s = i;
      } else {
        sym[pat - 1] = i;
      }
    }
    __syncthreads();
    tau = tau_s;
  }
  if (tid == 0) {
    score[b] = sc;
    lag[b] = tau;
    message[b] = sym[0] | (sym[1] << 8);
    detected[b] = sc >= threshold ? 1 : 0;
  }
}

static size_t wm_align(size_t v) { return (v + 255) & ~(size_t)255; }

}  // namespace asb

using namespace asb;

extern "C" int as_watermark_embed(const float* x, int64_t x_ld, int32_t B, int32_t S, const int32_t* lens,
                                  const float* pattern, float alpha, float* out, int64_t out_ld, void* stream) {
  if (B == 0 || S == 0) return AS_OK;
  ASB_REQUIRE(x && pattern && out && B > 0 && S > 0 && x_ld >= S && out_ld >= S, AS_ERR_SHAPE,
              "as_watermark_embed: bad argument");
  ASB_REQUIRE((reinterpret_cast<uintptr_t>(pattern) & 15) == 0, AS_ERR_ALIGN,
              "as_watermark_embed: the pattern must be 16-byte aligned");
  ASB_REQUIRE((const void*)x != (const void*)out, AS_ERR_SHAPE, "as_watermark_embed: out must not alias x");
  ASB_REQUIRE(B <= 65535, AS_ERR_SHAPE, "as_watermark_embed: B %d above 65535", (int)B);
  if (int rc = check_arch()) return rc;
  const int vec_in = (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (x_ld & 3) == 0;
  const int vec_out = (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (out_ld & 3) == 0;
  dim3 grid((unsigned)((S + kEmbTile - 1) / kEmbTile), (unsigned)B);
  ASB_CUDA(launch_k(wm_embed_kernel, grid, dim3(kWmThreads), 0, static_cast<cudaStream_t>(stream), x,
                    (long long)x_ld, (int)S, lens, pattern, alpha, out, (long long)out_ld, vec_in, vec_out));
  return AS_OK;
}

extern "C" size_t as_watermark_workspace_bytes(int32_t B, int32_t S) {
  if (B <= 0 || S <= 0) return 0;
  const size_t nper = ((size_t)S + kDetN - 1) / kDetN;
  return wm_align((size_t)B * nper * AS_WM_BINS_LD * sizeof(float2));
}

extern "C" int as_watermark_detect(const float* x, int64_t x_ld, int32_t B, int32_t S, const int32_t* lens,
                                   const float* spectra, const float* twiddles, float threshold, void* workspace,
                                   size_t workspace_bytes, float* score, int32_t* lag, int32_t* message,
                                   uint8_t* detected, void* stream) {
  if (B == 0) return AS_OK;
  ASB_REQUIRE(B > 0 && S >= 0 && x_ld >= S && (S == 0 || x) && spectra && twiddles && score && lag && message &&
                  detected,
              AS_ERR_SHAPE, "as_watermark_detect: bad argument");
  ASB_REQUIRE(workspace_bytes >= as_watermark_workspace_bytes(B, S) && (S == 0 || workspace), AS_ERR_SHAPE,
              "as_watermark_detect: workspace of %zu bytes, %zu needed", workspace_bytes,
              as_watermark_workspace_bytes(B, S));
  ASB_REQUIRE(((reinterpret_cast<uintptr_t>(spectra) | reinterpret_cast<uintptr_t>(twiddles) |
                reinterpret_cast<uintptr_t>(workspace)) & 7) == 0,
              AS_ERR_ALIGN, "as_watermark_detect: spectra, twiddles and workspace must be 8-byte aligned");
  const int nper_max = (int)(((long long)S + kDetN - 1) / kDetN);
  ASB_REQUIRE(B <= 65535 || nper_max == 0, AS_ERR_SHAPE, "as_watermark_detect: B %d above 65535", (int)B);
  if (int rc = check_arch()) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float2* tw = reinterpret_cast<const float2*>(twiddles);
  float2* ws = static_cast<float2*>(workspace);
  if (nper_max > 0)
    ASB_CUDA(launch_k(wm_spectra_kernel, dim3((unsigned)nper_max, (unsigned)B), dim3(kDetThreads), 0, st, x,
                      (long long)x_ld, (int)S, lens, tw, ws, nper_max));
  ASB_CUDA(launch_k(wm_correlate_kernel, dim3((unsigned)B), dim3(kDetThreads), 0, st, ws, nper_max, (int)S, lens,
                    reinterpret_cast<const float2*>(spectra), tw, threshold, score, lag, message, detected));
  return AS_OK;
}
