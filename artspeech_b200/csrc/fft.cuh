// In-place radix-2 FFT of 2^kLog2 complex fp32 points in shared memory, shared by the log-mel front-end
// (frontend.cu, 2048 points) and the watermark detector (watermark.cu, 4096 points).
#pragma once
#include "common.cuh"

namespace asb {

// Bit-reversed position of element i of a 2^kLog2-point transform: the caller writes its input there.
template <int kLog2>
__device__ __forceinline__ int fft_slot(int i) {
  return (int)(__brev((unsigned)i) >> (32 - kLog2));
}

// X[k] = sum_i x[i] e^{-2 pi j i k / N}, N = 2^kLog2, from buf holding x in bit-reversed order (fft_slot) to buf
// holding X in natural order.  twiddle[m] = (cos, -sin)(2 pi m / N), m < N/2.  Every thread of the block calls it
// with kThreads threads (N/2 a multiple of kThreads); buf must be complete (synchronised) on entry, and is on exit.
// Each butterfly is the same fp32 expression in every call, so a transform's bits depend only on its input.
template <int kLog2, int kThreads>
__device__ __forceinline__ void fft_radix2(float2* buf, const float2* __restrict__ twiddle, int tid) {
  constexpr int kN = 1 << kLog2;
  static_assert((kN / 2) % kThreads == 0, "fft_radix2: N/2 must be a multiple of the thread count");
#pragma unroll 1
  for (int st = 0; st < kLog2; ++st) {
    const int half = 1 << st;
    const int tw_step = (kN / 2) >> st;
#pragma unroll
    for (int j = 0; j < kN / 2 / kThreads; ++j) {
      const int k = tid + j * kThreads;
      const int pos = k & (half - 1);
      const int i0 = ((k >> st) << (st + 1)) + pos, i1 = i0 + half;
      const float2 w = twiddle[pos * tw_step];           // (cos, -sin)(2 pi pos / (2 half))
      const float2 a = buf[i0], c = buf[i1];
      const float2 t = make_float2(c.x * w.x - c.y * w.y, c.x * w.y + c.y * w.x);
      buf[i0] = make_float2(a.x + t.x, a.y + t.y);
      buf[i1] = make_float2(a.x - t.x, a.y - t.y);
    }
    __syncthreads();
  }
}

}  // namespace asb
