// Log-mel front-end (the step before the synthesis path, SURVEY.md §8f rank 1): the reference's
// torchaudio MelSpectrogram(n_mels 80, n_fft 2048, win 1200, hop 300) + log(1e-5 + .) + (x + 4) / 4
// (test.py:40-47, meldataset.py:42-49) for a batch of reference recordings, one launch.
//
// One CTA per frame: reflect-padded, windowed 2048-sample frame -> shared memory in bit-reversed order
// -> in-place radix-2 FFT (fft.cuh: fp32, twiddles from a host-computed table, 11 stages x 4 butterflies
// per thread) -> power spectrum -> triangular mel filters over each filter's own bin range -> log ->
// normalise -> [B, n_mels, n_frames] (the reference's channels-first mel layout).  fp32 throughout: a
// tensor-core DFT in 16-bit operands would bury the bins 60 dB below the frame's peak, which the log brings up.
#include "common.cuh"
#include "fft.cuh"

namespace asb {

constexpr int FE_NFFT = 2048, FE_LOG2 = 11, FE_THREADS = 256;

__global__ void __launch_bounds__(FE_THREADS)
log_mel_kernel(const float* __restrict__ wave, long long wave_ld, const int* __restrict__ lens,
               const int* __restrict__ starts, int N,
               const float* __restrict__ window, const float2* __restrict__ twiddle, const float* __restrict__ fb,
               const int2* __restrict__ fb_range, int hop, int n_mels, float log_eps, float mean, float inv_std,
               float* __restrict__ out, int n_frames) {
  pdl_wait();
  __shared__ float2 buf[FE_NFFT];
  __shared__ float power[FE_NFFT / 2 + 1];
  const int f = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const int st = starts ? starts[b] : 0;                 // first sample of the recording's span in its row
  const int nb = lens ? min(lens[b], N - st) : N - st;
  const int frames_b = nb > 0 ? 1 + nb / hop : 0;
  float* ob = out + (long long)b * n_mels * n_frames;
  if (f >= frames_b) {                                   // padding frame of a shorter recording
    for (int m = tid; m < n_mels; m += FE_THREADS) ob[(long long)m * n_frames + f] = 0.f;
    return;
  }
  const float* wb = wave + (long long)b * wave_ld + st;
  const int s0 = f * hop - FE_NFFT / 2;
  for (int i = tid; i < FE_NFFT; i += FE_THREADS) {
    int s = s0 + i;
    if (s < 0) s = -s;                                   // reflect padding (torch.stft centre = True)
    if (s >= nb) s = 2 * (nb - 1) - s;
    const float v = (s >= 0 && s < nb) ? wb[s] * window[i] : 0.f;
    buf[fft_slot<FE_LOG2>(i)] = make_float2(v, 0.f);
  }
  __syncthreads();
  fft_radix2<FE_LOG2, FE_THREADS>(buf, twiddle, tid);
  for (int i = tid; i <= FE_NFFT / 2; i += FE_THREADS) power[i] = buf[i].x * buf[i].x + buf[i].y * buf[i].y;
  __syncthreads();
  for (int m = tid; m < n_mels; m += FE_THREADS) {
    const int2 r = fb_range[m];                          // first bin, number of bins with a non-zero weight
    float acc = 0.f;
    for (int i = 0; i < r.y; ++i) acc += power[r.x + i] * fb[(long long)(r.x + i) * n_mels + m];
    ob[(long long)m * n_frames + f] = (logf(log_eps + acc) - mean) * inv_std;
  }
}

static int log_mel_launch(const float* wave, int64_t wave_ld, const int32_t* lens, const int32_t* starts, int32_t B,
                          int32_t N, const float* window, const float* twiddle, const float* fb, const int32_t* fb_range,
                          int32_t n_fft, int32_t hop, int32_t n_mels, float log_eps, float mean, float std, float* out,
                          int32_t n_frames, void* stream, const char* name) {
  if (B == 0 || n_frames == 0) return AS_OK;
  ASB_REQUIRE(wave && window && twiddle && fb && fb_range && out, AS_ERR_SHAPE, "%s: null pointer", name);
  ASB_REQUIRE(n_fft == FE_NFFT, AS_ERR_SHAPE, "%s: n_fft=%d unsupported (2048 only)", name, n_fft);
  ASB_REQUIRE(B > 0 && N > n_fft / 2 && hop > 0 && n_mels > 0 && std != 0.f, AS_ERR_SHAPE,
              "%s: bad argument (N must exceed n_fft/2 for reflect padding)", name);
  int rc = check_arch();
  if (rc != AS_OK) return rc;
  dim3 grid((unsigned)n_frames, (unsigned)B);
  ASB_CUDA(launch_k(log_mel_kernel, grid, FE_THREADS, 0, reinterpret_cast<cudaStream_t>(stream), wave, (long long)wave_ld, lens, starts, N, window,
                    reinterpret_cast<const float2*>(twiddle), fb, reinterpret_cast<const int2*>(fb_range), hop, n_mels, log_eps,
                    mean, 1.0f / std, out, n_frames));
  return AS_OK;
}

}  // namespace asb

using namespace asb;

extern "C" int as_log_mel(const float* wave, int64_t wave_ld, const int32_t* lens, int32_t B, int32_t N,
                          const float* window, const float* twiddle, const float* fb, const int32_t* fb_range,
                          int32_t n_fft, int32_t hop, int32_t n_mels, float log_eps, float mean, float std,
                          float* out, int32_t n_frames, void* stream) {
  return log_mel_launch(wave, wave_ld, lens, nullptr, B, N, window, twiddle, fb, fb_range, n_fft, hop, n_mels, log_eps,
                        mean, std, out, n_frames, stream, "as_log_mel");
}

extern "C" int as_log_mel_span(const float* wave, int64_t wave_ld, const int32_t* starts, const int32_t* lens,
                               int32_t B, int32_t N, const float* window, const float* twiddle, const float* fb,
                               const int32_t* fb_range, int32_t n_fft, int32_t hop, int32_t n_mels, float log_eps,
                               float mean, float std, float* out, int32_t n_frames, void* stream) {
  ASB_REQUIRE(B == 0 || n_frames == 0 || (starts && lens), AS_ERR_SHAPE, "as_log_mel_span: starts and lens are required");
  return log_mel_launch(wave, wave_ld, lens, starts, B, N, window, twiddle, fb, fb_range, n_fft, hop, n_mels, log_eps,
                        mean, std, out, n_frames, stream, "as_log_mel_span");
}
