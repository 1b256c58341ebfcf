// Voice enrollment input stage (artspeech_b200/frontend.py states the semantics; header: as_audio_to_mono,
// as_audio_decode, as_trim_bounds): the steps the reference applies to a reference recording before its log-mel
// (test.py:100-108: librosa.load(sr=24000), librosa.effects.trim(top_db=30)).
//
// Downmix: one launch, grid (tile of 1024 output samples, utterance).  A CTA stages the tile's C interleaved channels
// into shared memory (16-byte loads when the row allows, element loads for the tail), then each thread decodes and
// averages 4 outputs (fp32 sum in channel order, one fp32 divide) and stores them as one float4 where aligned.
// as_audio_decode is the C = 1 case.
//
// Trim: two launches.
//   1. grid (8 blocks of 512 samples, utterance): one warp per block, lane-strided fp64 sums of squares in a fixed
//      order (lane l owns samples 4 (l + 32 k) + e, k then e), a warp butterfly, q_j to the workspace.
//   2. one CTA per utterance: p_f = (((q_{f-2} + q_{f-1}) + q_f) + q_{f+1}) / 2048, P = max p_f, the decision in dB,
//      and the first / last non-silent frame (min / max reductions, exact in any order).
// No atomics; every sum's shape depends only on the utterance's own samples, so the bounds do not depend on B, S,
// the row stride or the batch-mates.
#include <cmath>

#include "common.cuh"

namespace asb {

constexpr int kMonoTile = 1024, kMonoThreads = 256, kMonoMaxC = AS_AUDIO_MAX_CHANNELS;
constexpr int kTrimBlock = 512, kTrimFrame = 2048, kTrimBlocksPerCta = 8, kTrimThreads = 256;
static_assert(kTrimBlocksPerCta * 32 == kTrimThreads, "one warp per block");
static_assert(kTrimBlock == 32 * 4 * 4, "a lane owns 4 float4 of a block");

// CPython audioop.ulaw2lin / alaw2lin, width 2 (st_ulaw2linear16 / st_alaw2linear16)
__device__ __forceinline__ int ulaw2lin(unsigned u) {
  u = ~u & 0xFFu;
  int t = (int)(((u & 0xFu) << 3) + 0x84u);
  t <<= (u & 0x70u) >> 4;
  return (u & 0x80u) ? 0x84 - t : t - 0x84;
}

__device__ __forceinline__ int alaw2lin(unsigned a) {
  a ^= 0x55u;
  int t = (int)((a & 0xFu) << 4);
  const int seg = (int)((a & 0x70u) >> 4);
  if (seg == 0) t += 8;
  else if (seg == 1) t += 0x108;
  else t = (t + 0x108) << (seg - 1);
  return (a & 0x80u) ? t : -t;
}

template <typename T, int ENC>
__device__ __forceinline__ float decode_sample(T v) {
  if constexpr (ENC == AS_AUDIO_F32) return v;
  else if constexpr (ENC == AS_AUDIO_PCM16) return (float)v * (1.f / 32768.f);
  else if constexpr (ENC == AS_AUDIO_MULAW) return (float)ulaw2lin(v) * (1.f / 32768.f);
  else return (float)alaw2lin(v) * (1.f / 32768.f);
}

// out[b, t] = (x_0[t] + ... + x_{C-1}[t]) / C for t < n_b, 0 for n_b <= t < S; nothing at or beyond n_b is read.
template <typename T, int ENC>
__global__ void __launch_bounds__(kMonoThreads) audio_to_mono_kernel(
    const T* __restrict__ in, long long in_ld, int S, int C, const int* __restrict__ lens, float* __restrict__ out,
    long long out_ld, int vec_in, int vec_out) {
  pdl_wait();
  constexpr int kVec = 16 / sizeof(T);
  __shared__ __align__(16) T xs[kMonoTile * kMonoMaxC];
  const int b = blockIdx.y, tid = threadIdx.x;
  const int t0 = blockIdx.x * kMonoTile;
  const int nt = min(kMonoTile, S - t0);
  const int n = lens ? min(max(lens[b], 0), S) : S;
  const int nv = max(0, min(nt, n - t0));               // valid outputs of this tile
  const T* src = in + (long long)b * in_ld + (long long)t0 * C;
  const int ne = nv * C;                                 // staged elements
  const int nvec = vec_in ? ne / kVec : 0;
  for (int q = tid; q < nvec; q += kMonoThreads)
    reinterpret_cast<int4*>(xs)[q] = __ldg(reinterpret_cast<const int4*>(src) + q);
  for (int i = nvec * kVec + tid; i < ne; i += kMonoThreads) xs[i] = src[i];
  __syncthreads();
  float* ob = out + (long long)b * out_ld + t0;
  const float fc = (float)C;
  for (int i = 4 * tid; i < nt; i += 4 * kMonoThreads) {
    float y[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float s = 0.f;
      if (i + e < nv) {
        const T* p = xs + (i + e) * C;
        s = decode_sample<T, ENC>(p[0]);
        for (int c = 1; c < C; ++c) s += decode_sample<T, ENC>(p[c]);
        s = s / fc;
      }
      y[e] = s;
    }
    if (vec_out && i + 3 < nt) {
      *reinterpret_cast<float4*>(ob + i) = make_float4(y[0], y[1], y[2], y[3]);
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (i + e < nt) ob[i + e] = y[e];
    }
  }
}

// Launch 1 of the trim: q_j = sum of y^2 over block j (fp64), for the blocks j < ceil(n_b / 512).
__global__ void __launch_bounds__(kTrimThreads) trim_blocks_kernel(const float* __restrict__ y, long long y_ld, int S,
                                                                   const int* __restrict__ lens,
                                                                   double* __restrict__ q, int nblk_max, int vec) {
  pdl_wait();
  const int b = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int j = blockIdx.x * kTrimBlocksPerCta + warp;
  const int n = lens ? min(max(lens[b], 0), S) : S;
  if (j >= (n + kTrimBlock - 1) / kTrimBlock) return;
  const float* yb = y + (long long)b * y_ld + (long long)j * kTrimBlock;
  const int m = min(kTrimBlock, n - j * kTrimBlock);     // samples of this block below n
  double acc = 0.0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int i = 4 * (lane + 32 * k);
    float4 v;
    if (vec && m == kTrimBlock) {
      v = __ldg(reinterpret_cast<const float4*>(yb + i));
    } else {
      v.x = i < m ? yb[i] : 0.f;
      v.y = i + 1 < m ? yb[i + 1] : 0.f;
      v.z = i + 2 < m ? yb[i + 2] : 0.f;
      v.w = i + 3 < m ? yb[i + 3] : 0.f;
    }
    acc = fma((double)v.x, (double)v.x, acc);
    acc = fma((double)v.y, (double)v.y, acc);
    acc = fma((double)v.z, (double)v.z, acc);
    acc = fma((double)v.w, (double)v.w, acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) q[(long long)b * nblk_max + j] = acc;
}

__device__ __forceinline__ double trim_frame_power(const double* qb, int nblk, int f) {
  double s = 0.0;
#pragma unroll
  for (int d = -2; d <= 1; ++d) {
    const int j = f + d;
    s += (j >= 0 && j < nblk) ? qb[j] : 0.0;
  }
  return s / (double)kTrimFrame;
}

// Launch 2 of the trim: one CTA per utterance.
__global__ void __launch_bounds__(kTrimThreads) trim_decide_kernel(const double* __restrict__ q, int nblk_max, int S,
                                                                   const int* __restrict__ lens, double top_db,
                                                                   int* __restrict__ bounds) {
  pdl_wait();
  __shared__ double red_p[kTrimThreads / 32];
  __shared__ int red_lo[kTrimThreads / 32], red_hi[kTrimThreads / 32];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = lens ? min(max(lens[b], 0), S) : S;
  if (n == 0) {
    if (tid == 0) { bounds[2 * b] = 0; bounds[2 * b + 1] = 0; }
    return;
  }
  const int nblk = (n + kTrimBlock - 1) / kTrimBlock, F = 1 + n / kTrimBlock;
  const double* qb = q + (long long)b * nblk_max;
  double pm = 0.0;
  for (int f = tid; f < F; f += kTrimThreads) pm = fmax(pm, trim_frame_power(qb, nblk, f));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) pm = fmax(pm, __shfl_xor_sync(0xffffffffu, pm, o));
  if (lane == 0) red_p[warp] = pm;
  __syncthreads();
  double P = red_p[0];
  for (int w = 1; w < kTrimThreads / 32; ++w) P = fmax(P, red_p[w]);
  const double ref_db = 10.0 * log10(fmax(1e-10, P));
  int lo = F, hi = -1;
  for (int f = tid; f < F; f += kTrimThreads) {
    const double db = 10.0 * log10(fmax(1e-10, trim_frame_power(qb, nblk, f))) - ref_db;
    if (db > -top_db) { lo = min(lo, f); hi = max(hi, f); }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if (lane == 0) { red_lo[warp] = lo; red_hi[warp] = hi; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < kTrimThreads / 32; ++w) { lo = min(lo, red_lo[w]); hi = max(hi, red_hi[w]); }
    // the frame holding P is always non-silent (0 dB > -top_db), so lo <= hi
    bounds[2 * b] = lo * kTrimBlock;
    bounds[2 * b + 1] = (int)min((long long)n, (long long)(hi + 1) * kTrimBlock);
  }
}

static size_t trim_align(size_t v) { return (v + 255) & ~(size_t)255; }

template <typename T, int ENC>
static int launch_to_mono(const void* in, int64_t in_ld, int32_t B, int32_t S, int32_t C, const int32_t* lens,
                          float* out, int64_t out_ld, cudaStream_t st) {
  const int vec_in = (reinterpret_cast<uintptr_t>(in) & 15) == 0 && ((in_ld * (int64_t)sizeof(T)) & 15) == 0;
  const int vec_out = (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (out_ld & 3) == 0;
  dim3 grid((unsigned)((S + kMonoTile - 1) / kMonoTile), (unsigned)B);
  ASB_CUDA(launch_k(audio_to_mono_kernel<T, ENC>, grid, dim3(kMonoThreads), 0, st, static_cast<const T*>(in),
                    (long long)in_ld, (int)S, (int)C, lens, out, (long long)out_ld, vec_in, vec_out));
  return AS_OK;
}

}  // namespace asb

using namespace asb;

extern "C" int as_audio_to_mono(const void* in, int64_t in_ld, int32_t B, int32_t S, int32_t C, int32_t encoding,
                                const int32_t* lens, float* out, int64_t out_ld, void* stream) {
  if (B == 0 || S == 0) return AS_OK;
  ASB_REQUIRE(in && out && B > 0 && S > 0 && C >= 1 && C <= kMonoMaxC && in_ld >= (int64_t)S * C && out_ld >= S &&
                  B <= 65535,
              AS_ERR_SHAPE, "as_audio_to_mono: bad argument (C must be 1..%d)", kMonoMaxC);
  ASB_REQUIRE((const void*)in != (const void*)out, AS_ERR_SHAPE, "as_audio_to_mono: out must not alias in");
  if (int rc = check_arch()) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (encoding) {
    case AS_AUDIO_F32: return launch_to_mono<float, AS_AUDIO_F32>(in, in_ld, B, S, C, lens, out, out_ld, st);
    case AS_AUDIO_PCM16: return launch_to_mono<int16_t, AS_AUDIO_PCM16>(in, in_ld, B, S, C, lens, out, out_ld, st);
    case AS_AUDIO_MULAW: return launch_to_mono<uint8_t, AS_AUDIO_MULAW>(in, in_ld, B, S, C, lens, out, out_ld, st);
    case AS_AUDIO_ALAW: return launch_to_mono<uint8_t, AS_AUDIO_ALAW>(in, in_ld, B, S, C, lens, out, out_ld, st);
    default:
      set_error("as_audio_to_mono: encoding %d is not F32, PCM16, mu-law or A-law", (int)encoding);
      return AS_ERR_DTYPE;
  }
}

extern "C" int as_audio_decode(const void* in, int64_t in_ld, int32_t B, int32_t S, int32_t encoding, float* out,
                               int64_t out_ld, void* stream) {
  if (B == 0 || S == 0) return AS_OK;
  ASB_REQUIRE(encoding == AS_AUDIO_PCM16 || encoding == AS_AUDIO_MULAW || encoding == AS_AUDIO_ALAW, AS_ERR_DTYPE,
              "as_audio_decode: encoding %d is not PCM16, mu-law or A-law", (int)encoding);
  return as_audio_to_mono(in, in_ld, B, S, 1, encoding, nullptr, out, out_ld, stream);
}

extern "C" size_t as_trim_workspace_bytes(int32_t B, int32_t S) {
  if (B <= 0 || S <= 0) return 0;
  const size_t nblk = ((size_t)S + kTrimBlock - 1) / kTrimBlock;
  return trim_align((size_t)B * nblk * sizeof(double));
}

extern "C" int as_trim_bounds(const float* y, int64_t y_ld, int32_t B, int32_t S, const int32_t* lens, double top_db,
                              void* workspace, size_t workspace_bytes, int32_t* bounds, void* stream) {
  if (B == 0) return AS_OK;
  ASB_REQUIRE(B > 0 && B <= 65535 && S >= 0 && y_ld >= S && (S == 0 || y) && bounds, AS_ERR_SHAPE,
              "as_trim_bounds: bad argument");
  ASB_REQUIRE(top_db > 0.0 && std::isfinite(top_db), AS_ERR_SHAPE, "as_trim_bounds: top_db must be finite and positive");
  ASB_REQUIRE(workspace_bytes >= as_trim_workspace_bytes(B, S) && (S == 0 || workspace), AS_ERR_WORKSPACE,
              "as_trim_bounds: workspace of %zu bytes, %zu needed", workspace_bytes, as_trim_workspace_bytes(B, S));
  ASB_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 7) == 0, AS_ERR_ALIGN,
              "as_trim_bounds: the workspace must be 8-byte aligned");
  if (int rc = check_arch()) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int nblk_max = (int)(((long long)S + kTrimBlock - 1) / kTrimBlock);
  double* q = static_cast<double*>(workspace);
  if (nblk_max > 0) {
    const int vec = (reinterpret_cast<uintptr_t>(y) & 15) == 0 && (y_ld & 3) == 0;
    dim3 grid((unsigned)((nblk_max + kTrimBlocksPerCta - 1) / kTrimBlocksPerCta), (unsigned)B);
    ASB_CUDA(launch_k(trim_blocks_kernel, grid, dim3(kTrimThreads), 0, st, y, (long long)y_ld, (int)S, lens, q,
                      nblk_max, vec));
  }
  ASB_CUDA(launch_k(trim_decide_kernel, dim3((unsigned)B), dim3(kTrimThreads), 0, st, (const double*)q, nblk_max,
                    (int)S, lens, top_db, bounds));
  return AS_OK;
}
