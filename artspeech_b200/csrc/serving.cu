// Small device-side glue of the serving path: everything the reference does on the host between the duration
// predictor and the length regulator (models.py:361-366: round, clamp, cumulative frame counts) stays on the
// device, so the whole pass is capturable in a CUDA graph with durations as a graph INPUT.  The per-utterance
// prosody controls (artspeech_b200/prosody.py) are graph inputs the same way: a duration scale applied before the
// rounding, and edits of the predicted F0 / energy / EMA tracks before the decoder.
#include "common.cuh"

namespace asb {

// One warp per utterance: dur[b,t] = max(1, rint(pred[b,t] * s)) for t < lens[b], else 0 (torch.round is
// round-half-to-even = rintf in the default rounding mode); sum[b] = total half-rate frames of the utterance.
// s = 1 when scale is NULL, scale[b * scale_ld + t] otherwise (scale_ld == 0: scale[b], one value per utterance).
__global__ void round_durations_kernel(const float* __restrict__ pred, long long pred_ld, int B, int Tt,
                                       const int* __restrict__ lens, const float* __restrict__ scale,
                                       long long scale_ld, int* __restrict__ dur, int* __restrict__ sum) {
  pdl_wait();
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  const int n = lens ? min(max(lens[b], 0), Tt) : Tt;
  int acc = 0;
  for (int t = lane; t < Tt; t += 32) {
    int d = 0;
    if (t < n) {
      float p = pred[(long long)b * pred_ld + t];
      if (scale) p *= scale_ld ? scale[(long long)b * scale_ld + t] : scale[b];
      const float r = rintf(p);
      d = r >= 1.f ? (r > 2147483000.f ? 2147483000 : (int)r) : 1;     // clamp(min=1); NaN -> 1
    }
    dur[(long long)b * Tt + t] = d;
    acc += d;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0 && sum) sum[b] = acc;
}

constexpr int kProsodyThreads = 512;
constexpr int kEma = 10;
constexpr int kSums = 2 + kEma;               // sum ln hz, voiced count, EMA channel sums
constexpr float kVoicingFloorHz = 50.f;       // prosody.VOICING_FLOOR_HZ

// One CTA per utterance (grid = B).  Thread i visits frames i, i + 512, ... below the utterance's length, so the
// partial sums, and the fixed shuffle / warp-order reduction after them, depend on the utterance's own frames only:
// not on B, the bucket's Tm or the grid.  An utterance's edited tracks are therefore bit-identical whatever it is
// batched with.  Arithmetic is fp64 with one rounding to fp32 per written value (the tracks are 48 bytes a frame;
// fp64 costs nothing here and keeps the result within an ulp of an exact evaluation).
__global__ void __launch_bounds__(kProsodyThreads) prosody_apply_kernel(
    float* __restrict__ f0, long long f0_ld, float* __restrict__ nrg, long long n_ld, float* __restrict__ ema,
    long long ema_ld, int Tm, const int* __restrict__ lens, const float* __restrict__ ctrl, double pitch_mean,
    double pitch_std, double energy_std) {
  pdl_wait();
  const int b = blockIdx.x;
  const float* c = ctrl + (long long)b * AS_PROSODY_CTRL;
  const float shift = c[0], range = c[1], db = c[2];
  // identity tracks are not written (CTA-uniform)
  const bool do_f0 = shift != 0.f || range != 1.f;
  const bool do_n = db != 0.f;
  bool do_ema = false;
#pragma unroll
  for (int k = 0; k < kEma; ++k) do_ema |= c[4 + k] != 1.f || c[4 + kEma + k] != 0.f;
  if (!(do_f0 || do_n || do_ema)) return;
  const int len = lens ? min(max(lens[b], 0), Tm) : Tm;
  f0 += (long long)b * Tm * f0_ld;
  nrg += (long long)b * Tm * n_ld;
  ema += (long long)b * Tm * ema_ld;

  // pass 1: sum of ln hz and count over the voiced frames, EMA channel sums over all valid frames
  double s[kSums];
#pragma unroll
  for (int k = 0; k < kSums; ++k) s[k] = 0.0;
  for (int t = threadIdx.x; t < len; t += kProsodyThreads) {
    if (do_f0) {
      const double hz = (double)f0[t * f0_ld] * pitch_std + pitch_mean;
      if (hz >= kVoicingFloorHz) { s[0] += log(hz); s[1] += 1.0; }
    }
    if (do_ema) {
#pragma unroll
      for (int k = 0; k < kEma; ++k) s[2 + k] += (double)ema[t * ema_ld + k];
    }
  }
  __shared__ double red[kProsodyThreads / 32][kSums];
  __shared__ double tot[kSums];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < kSums; ++k) {
    double v = s[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < kSums) {
    double v = 0.0;
    for (int w = 0; w < kProsodyThreads / 32; ++w) v += red[w][threadIdx.x];
    tot[threadIdx.x] = v;
  }
  __syncthreads();

  // pass 2: the edits
  const bool edit_f0 = do_f0 && tot[1] > 0.0;                     // no voiced frame: F0 unchanged
  const double mu = edit_f0 ? tot[0] / tot[1] : 0.0;
  const double lift = (double)shift * (0.69314718055994531 / 12.0);
  const double dn = (double)db * (2.302585092994046 / 10.0) / energy_std;
  double m[kEma];
#pragma unroll
  for (int k = 0; k < kEma; ++k) m[k] = len > 0 ? tot[2 + k] / (double)len : 0.0;
  for (int t = threadIdx.x; t < len; t += kProsodyThreads) {
    if (edit_f0) {
      const float v = f0[t * f0_ld];
      const double hz = (double)v * pitch_std + pitch_mean;
      if (hz >= kVoicingFloorHz) {
        const double hz2 = exp(mu + (double)range * (log(hz) - mu) + lift);
        f0[t * f0_ld] = (float)((double)v + (hz2 - hz) / pitch_std);
      }
    }
    if (do_n) nrg[t * n_ld] = (float)((double)nrg[t * n_ld] + dn);
    if (do_ema) {
#pragma unroll
      for (int k = 0; k < kEma; ++k) {
        float* p = ema + t * ema_ld + k;
        *p = (float)(m[k] + (double)c[4 + k] * ((double)*p - m[k]) + (double)c[4 + kEma + k]);
      }
    }
  }
}

}  // namespace asb

using namespace asb;

static int round_durations_launch(const float* pred, int64_t pred_ld, int32_t B, int32_t Tt, const int32_t* lens,
                                  const float* scale, int64_t scale_ld, int32_t* dur, int32_t* sum, void* stream) {
  if (int rc = check_arch()) return rc;
  const int warps = 4;
  ASB_CUDA(launch_k(round_durations_kernel, dim3((B + warps - 1) / warps), dim3(32 * warps), 0,
                    static_cast<cudaStream_t>(stream), pred, (long long)pred_ld, B, Tt, lens, scale,
                    (long long)scale_ld, dur, sum));
  return AS_OK;
}

extern "C" int as_round_durations(const float* pred, int64_t pred_ld, int32_t B, int32_t Tt, const int32_t* lens,
                                  int32_t* dur, int32_t* sum, void* stream) {
  if (B == 0) return AS_OK;
  ASB_REQUIRE(pred && dur && B > 0 && Tt >= 0 && pred_ld >= Tt, AS_ERR_SHAPE, "as_round_durations: bad argument");
  return round_durations_launch(pred, pred_ld, B, Tt, lens, nullptr, 0, dur, sum, stream);
}

extern "C" int as_round_durations_scaled(const float* pred, int64_t pred_ld, int32_t B, int32_t Tt,
                                         const int32_t* lens, const float* scale, int64_t scale_ld, int32_t* dur,
                                         int32_t* sum, void* stream) {
  if (B == 0) return AS_OK;
  ASB_REQUIRE(pred && dur && scale && B > 0 && Tt >= 0 && pred_ld >= Tt && (scale_ld == 0 || scale_ld >= Tt),
              AS_ERR_SHAPE, "as_round_durations_scaled: bad argument");
  return round_durations_launch(pred, pred_ld, B, Tt, lens, scale, scale_ld, dur, sum, stream);
}

extern "C" int as_prosody_apply(float* f0, int64_t f0_ld, float* n, int64_t n_ld, float* ema, int64_t ema_ld,
                                int32_t B, int32_t Tm, const int32_t* lens, const float* ctrl, double pitch_mean,
                                double pitch_std, double energy_std, void* stream) {
  if (B == 0 || Tm == 0) return AS_OK;
  ASB_REQUIRE(f0 && n && ema && ctrl && B > 0 && Tm > 0 && f0_ld >= 1 && n_ld >= 1 && ema_ld >= kEma,
              AS_ERR_SHAPE, "as_prosody_apply: bad argument");
  ASB_REQUIRE(pitch_std > 0.0 && energy_std > 0.0, AS_ERR_SHAPE,
              "as_prosody_apply: pitch_std and energy_std must be positive");
  if (int rc = check_arch()) return rc;
  ASB_CUDA(launch_k(prosody_apply_kernel, dim3(B), dim3(kProsodyThreads), 0, static_cast<cudaStream_t>(stream), f0,
                    (long long)f0_ld, n, (long long)n_ld, ema, (long long)ema_ld, (int)Tm, lens, ctrl, pitch_mean,
                    pitch_std, energy_std));
  return AS_OK;
}
