// FLAC output for synthesis (artspeech_b200/audio.py states the format; header: as_flac_encode): one complete
// RFC 9639 stream per utterance of int16 samples, 4096-sample blocks, mono, 16 bits.  Three launches:
//   1. Analysis: grid (block, row), 256 threads.  The block is staged in shared memory; the int64 autocorrelation
//      at lags 0..8 is a per-thread strided sum reduced in a fixed shape (integer, so exact); lane 0 of warp 0 runs
//      the fp64 Levinson recursion and the precision-12 quantisation with __dmul_rn / __dsub_rn / __ddiv_rn.  Each
//      predictor candidate (FIXED 0..4, LPC 1..8) is evaluated in turn: sum (u >> k), k = 0..14, per partition at the
//      finest partition order (each thread owns a run of one partition, integer atomics only where several threads
//      share one), then one pass per coarser order sums pairs of partitions (ping-pong buffers) while the per-order
//      cost is reduced per warp.  The smallest candidate wins, earlier on ties.  The decision record and the frame's
//      byte count go to the workspace.
//   2. Layout: one CTA per row.  An exclusive scan of the frame sizes gives the frame offsets and the byte count; the
//      CTA writes the 42-byte header (fLaC + STREAMINFO with min / max frame size) and zeroes the row past its end.
//   3. Emit: grid (block, row), 256 threads.  The chosen residual is recomputed, the Rice parameters re-derived at the
//      chosen partition order, per-sample code lengths are scanned across the block, and every field is OR-ed into
//      a shared-memory copy of the frame (integer atomicOr on 32-bit words, so the result does not depend on order).
//      CRC-16 is computed as per-thread CRCs of byte runs, each moved to the frame's end by a multiplication with
//      x^(8 L) mod P and XOR-reduced.  The frame is stored with 16-byte stores between byte-wise ends.
// No floating-point atomics, no host synchronisation; every byte of a row follows from its own samples and length, so
// the output does not depend on B, S, the row strides or the batch-mates.  Samples at or beyond n_b are never read.
#include <climits>
#include <cmath>

#include "common.cuh"

namespace asb {

constexpr int kFlBlock = AS_FLAC_BLOCK, kFlThreads = 256, kFlWarps = kFlThreads / 32;
constexpr int kFlMaxLpc = 8, kFlMaxPorder = 8, kFlKs = 15, kFlPrecision = 12;
constexpr int kFlParts = 1 << kFlMaxPorder;                 // partitions at order 8
constexpr int kFlFrameWords = 2064;                         // > 8210 bytes, the largest frame, plus one word
constexpr int kFlRecInts = 16;                              // kind, order, porder, shift, coef[8], bytes, pad
constexpr int kFlPerThread = kFlBlock / kFlThreads;
static_assert(kFlPerThread == 16 && kFlParts == kFlThreads, "one thread per order-8 partition of a full block");

enum { kFlConstant = 0, kFlFixed = 1, kFlLpc = 2, kFlVerbatim = 3 };

__device__ __forceinline__ long long fl_len(const int* lens, int b, long long S) {
  return lens ? min(max((long long)lens[b], 0LL), S) : S;
}

__device__ __forceinline__ int fl_utf8_len(unsigned v) {
  return v < 0x80u ? 1 : v < 0x800u ? 2 : v < 0x10000u ? 3 : v < 0x200000u ? 4 : v < 0x4000000u ? 5 : 6;
}

__device__ __forceinline__ int fl_rate_code(int rate) {
  switch (rate) {
    case 8000: return 4;
    case 16000: return 5;
    case 22050: return 6;
    case 24000: return 7;
    case 32000: return 8;
    case 44100: return 9;
    case 48000: return 10;
    default: return 13;                                     // 16-bit rate in Hz follows
  }
}

__device__ __forceinline__ int fl_header_bytes(unsigned f, int bs, int rate) {
  return 4 + fl_utf8_len(f) + (bs != kFlBlock ? 2 : 0) + (fl_rate_code(rate) == 13 ? 2 : 0) + 1;
}

__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void fl_fixed_coefs(int order, int* c) {
  const int t[5][4] = {{0, 0, 0, 0}, {1, 0, 0, 0}, {2, -1, 0, 0}, {3, -3, 1, 0}, {4, -6, 4, -1}};
#pragma unroll
  for (int j = 0; j < kFlMaxLpc; ++j) c[j] = j < 4 ? t[order][j] : 0;
}

// Zigzag value of the residual x[i] - ((sum_{j=1}^{order} c_j x[i-j]) >> shift); sets *big when |r| >= 2^31.
__device__ __forceinline__ unsigned long long fl_residual(const int* xs, int i, int order, const int* c, int shift,
                                                          bool& big) {
  long long acc = 0;
#pragma unroll
  for (int j = 1; j <= kFlMaxLpc; ++j)
    if (j <= order) acc += (long long)c[j - 1] * xs[i - j];
  const long long r = (long long)xs[i] - (acc >> shift);
  if (r >= (1LL << 31) || r <= -(1LL << 31)) big = true;
  return r >= 0 ? 2ull * (unsigned long long)r : 2ull * (unsigned long long)(-r) - 1ull;
}

// sums[k * ld + p] = sum of (u_i >> k) over the residual samples i >= order of partition p < 2^o.  The caller zeroes
// sums (when several threads share a partition) and synchronises after.
__device__ void fl_partition_sums(const int* xs, int bs, int order, const int* c, int shift, int o,
                                  unsigned long long* sums, int ld, int* overflow) {
  const int P = 1 << o, m = bs >> o, g = kFlThreads / P, t = threadIdx.x, p = t / g, j = t % g;
  unsigned long long s[kFlKs];
#pragma unroll
  for (int k = 0; k < kFlKs; ++k) s[k] = 0;
  bool big = false;
  for (int i = p * m + j; i < (p + 1) * m; i += g) {
    if (i < order) continue;
    const unsigned long long u = fl_residual(xs, i, order, c, shift, big);
#pragma unroll
    for (int k = 0; k < kFlKs; ++k) s[k] += u >> k;
  }
  if (big) *overflow = 1;
  if (g == 1) {
#pragma unroll
    for (int k = 0; k < kFlKs; ++k) sums[k * ld + p] = s[k];
  } else {
#pragma unroll
    for (int k = 0; k < kFlKs; ++k)
      if (s[k]) atomicAdd(&sums[k * ld + p], s[k]);
  }
}

// ---- launch 1: analysis ------------------------------------------------------------------------------------------
struct FlAnalysisSmem {
  int x[kFlBlock];
  unsigned long long sa[kFlKs * kFlParts];                  // partition sums, even passes
  unsigned long long sb[kFlKs * kFlParts / 2];              // odd passes
  long long wsum[(kFlMaxPorder + 1) * kFlWarps];
  long long wr[kFlWarps][kFlMaxLpc + 1];
  int q[kFlMaxLpc][kFlMaxLpc];                              // quantised predictor of order p + 1
  int shift[kFlMaxLpc], ok[kFlMaxLpc];
  int overflow, differ;
  int best_kind, best_order, best_porder, best_shift, best_coef[kFlMaxLpc];
  long long best_bits;
};

// Quantise the fp64 predictor a[1..p] at precision 12 into q; false when it is not a candidate.
__device__ bool fl_quantize(const double* a, int p, int* q, int* shift_out) {
  double cmax = 0.0;
  for (int j = 1; j <= p; ++j) {
    if (!isfinite(a[j])) return false;                    // any a_j not finite: no candidate
    cmax = fmax(cmax, fabs(a[j]));
  }
  int e = 0;
  frexp(cmax, &e);
  int shift = kFlPrecision - 1 - e;
  if (shift < 0) return false;
  shift = min(shift, 15);
  const double scale = ldexp(1.0, shift);
  double err = 0.0;
  for (int j = 1; j <= p; ++j) {
    err = __dadd_rn(err, __dmul_rn(a[j], scale));
    const long long r = llround(err);
    const int qi = (int)min(max(r, -(1LL << (kFlPrecision - 1))), (1LL << (kFlPrecision - 1)) - 1);
    err = __dsub_rn(err, (double)qi);
    q[j - 1] = qi;
  }
  *shift_out = shift;
  return true;
}

__global__ void __launch_bounds__(kFlThreads) flac_analysis_kernel(
    const int16_t* __restrict__ x, long long x_ld, long long S, const int* __restrict__ lens, int rate,
    int* __restrict__ recs, int F_max) {
  pdl_wait();
  extern __shared__ __align__(16) unsigned char fl_smem[];
  FlAnalysisSmem& sm = *reinterpret_cast<FlAnalysisSmem*>(fl_smem);
  const int b = blockIdx.y, f = blockIdx.x, t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const long long n = fl_len(lens, b, S);
  if ((long long)f * kFlBlock >= n) return;
  const int bs = (int)min((long long)kFlBlock, n - (long long)f * kFlBlock);
  const int16_t* xb = x + (long long)b * x_ld + (long long)f * kFlBlock;
  for (int i = t; i < bs; i += kFlThreads) sm.x[i] = xb[i];
  if (t == 0) sm.differ = 0;
  __syncthreads();

  // exact autocorrelation and the constant test
  long long R[kFlMaxLpc + 1];
#pragma unroll
  for (int l = 0; l <= kFlMaxLpc; ++l) R[l] = 0;
  bool differ = false;
  const int x0 = sm.x[0];
  for (int i = t; i < bs; i += kFlThreads) {
    const long long v = sm.x[i];
    differ |= sm.x[i] != x0;
#pragma unroll
    for (int l = 0; l <= kFlMaxLpc; ++l)
      if (i >= l) R[l] += v * sm.x[i - l];
  }
  if (differ) sm.differ = 1;
#pragma unroll
  for (int l = 0; l <= kFlMaxLpc; ++l) {
    const long long v = warp_sum_ll(R[l]);
    if (lane == 0) sm.wr[warp][l] = v;
  }
  __syncthreads();
  if (t == 0) {
    double Rd[kFlMaxLpc + 1], a[kFlMaxLpc + 1], na[kFlMaxLpc + 1];
    for (int l = 0; l <= kFlMaxLpc; ++l) {
      long long s = 0;
      for (int w = 0; w < kFlWarps; ++w) s += sm.wr[w][l];
      Rd[l] = (double)s;
      a[l] = 0.0;
    }
    for (int p = 0; p < kFlMaxLpc; ++p) sm.ok[p] = 0;
    double E = Rd[0];
    for (int m = 1; m <= kFlMaxLpc; ++m) {
      if (!(E > 0.0)) break;
      double acc = Rd[m];
      for (int j = 1; j < m; ++j) acc = __dsub_rn(acc, __dmul_rn(a[j], Rd[m - j]));
      const double k = __ddiv_rn(acc, E);
      if (!isfinite(k)) break;
      for (int j = 1; j < m; ++j) na[j] = __dsub_rn(a[j], __dmul_rn(k, a[m - j]));
      for (int j = 1; j < m; ++j) a[j] = na[j];
      a[m] = k;
      E = __dmul_rn(E, __dsub_rn(1.0, __dmul_rn(k, k)));
      sm.ok[m - 1] = bs > m && fl_quantize(a, m, sm.q[m - 1], &sm.shift[m - 1]);
    }
    sm.best_kind = kFlVerbatim;
    sm.best_order = sm.best_porder = sm.best_shift = 0;
    sm.best_bits = LLONG_MAX;
    if (!sm.differ) {                                       // CONSTANT is first in the order: it wins any tie
      sm.best_kind = kFlConstant;
      sm.best_bits = 8 + 16;
    }
  }
  __syncthreads();

  int omax = 0;
  while (omax < kFlMaxPorder && bs % (2 << omax) == 0) ++omax;
  for (int cand = 0; cand < 5 + kFlMaxLpc; ++cand) {
    const bool lpc = cand >= 5;
    const int order = lpc ? cand - 4 : cand;
    if (bs <= order || (lpc && !sm.ok[order - 1])) continue;   // block-uniform
    int c[kFlMaxLpc], shift = 0;
    if (lpc) {
#pragma unroll
      for (int j = 0; j < kFlMaxLpc; ++j) c[j] = sm.q[order - 1][j];
      shift = sm.shift[order - 1];
    } else {
      fl_fixed_coefs(order, c);
    }
    for (int i = t; i < kFlKs * kFlParts; i += kFlThreads) sm.sa[i] = 0;
    if (t == 0) sm.overflow = 0;
    __syncthreads();
    fl_partition_sums(sm.x, bs, order, c, shift, omax, sm.sa, kFlParts, &sm.overflow);
    __syncthreads();
    for (int o = omax, it = 0; o >= 0; --o, ++it) {
      const unsigned long long* cur = (it & 1) ? sm.sb : sm.sa;
      unsigned long long* nxt = (it & 1) ? sm.sa : sm.sb;
      const int ldc = (it & 1) ? kFlParts / 2 : kFlParts, ldn = (it & 1) ? kFlParts : kFlParts / 2;
      const int P = 1 << o;
      long long cost = 0;
      if (t < P) {
        const long long cnt = (bs >> o) - (t == 0 ? order : 0);
        long long best = LLONG_MAX;
#pragma unroll
        for (int k = 0; k < kFlKs; ++k) {
          const long long v = (long long)cur[k * ldc + t] + cnt * (1 + k);
          if (v < best) best = v;
        }
        cost = 4 + best;
      }
      cost = warp_sum_ll(cost);
      if (lane == 0) sm.wsum[o * kFlWarps + warp] = cost;
      if (t < P / 2) {
#pragma unroll
        for (int k = 0; k < kFlKs; ++k) nxt[k * ldn + t] = cur[k * ldc + 2 * t] + cur[k * ldc + 2 * t + 1];
      }
      __syncthreads();
    }
    if (t == 0 && !sm.overflow) {
      long long rice = LLONG_MAX;
      int porder = 0;
      for (int o = 0; o <= omax; ++o) {
        if ((bs >> o) <= order) continue;
        long long v = 2 + 4;
        for (int w = 0; w < kFlWarps; ++w) v += sm.wsum[o * kFlWarps + w];
        if (v < rice) { rice = v; porder = o; }
      }
      const long long bits = 8 + 16LL * order + (lpc ? 4 + 5 + (long long)kFlPrecision * order : 0) + rice;
      if (rice != LLONG_MAX && bits < sm.best_bits) {
        sm.best_bits = bits;
        sm.best_kind = lpc ? kFlLpc : kFlFixed;
        sm.best_order = order;
        sm.best_porder = porder;
        sm.best_shift = shift;
        for (int j = 0; j < kFlMaxLpc; ++j) sm.best_coef[j] = c[j];
      }
    }
    // the next candidate's first barrier orders thread 0's reads of wsum / overflow before they are rewritten
  }
  if (t == 0) {
    if (8 + 16LL * bs < sm.best_bits) {                     // VERBATIM is last: it wins no tie
      sm.best_kind = kFlVerbatim;
      sm.best_bits = 8 + 16LL * bs;
    }
    int* rec = recs + ((long long)b * F_max + f) * kFlRecInts;
    const bool pred = sm.best_kind == kFlFixed || sm.best_kind == kFlLpc;
    rec[0] = sm.best_kind;
    rec[1] = sm.best_order;
    rec[2] = sm.best_porder;
    rec[3] = sm.best_shift;
    for (int j = 0; j < kFlMaxLpc; ++j) rec[4 + j] = pred ? sm.best_coef[j] : 0;
    rec[12] = fl_header_bytes((unsigned)f, bs, rate) + (int)((sm.best_bits + 7) / 8) + 2;
  }
}

// ---- byte stores -------------------------------------------------------------------------------------------------
// dst[0 .. len) = byte(i), with 16-byte stores where dst is 16-byte aligned; the CTA's threads share the work.
template <typename ByteAt, typename Word4At>
__device__ void fl_store(uint8_t* dst, long long len, ByteAt byte_at, Word4At word4_at) {
  const int t = threadIdx.x;
  const long long head = min(len, (long long)((16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15));
  for (long long i = t; i < head; i += kFlThreads) dst[i] = byte_at(i);
  const long long chunks = (len - head) / 16;
  for (long long c = t; c < chunks; c += kFlThreads) {
    const long long s = head + 16 * c;
    *reinterpret_cast<uint4*>(dst + s) = make_uint4(word4_at(s), word4_at(s + 4), word4_at(s + 8), word4_at(s + 12));
  }
  for (long long i = head + 16 * chunks + t; i < len; i += kFlThreads) dst[i] = byte_at(i);
}

// ---- launch 2: layout --------------------------------------------------------------------------------------------
__device__ __forceinline__ long long fl_block_excl_scan(long long v, long long* wbuf, long long* total) {
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  long long inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long u = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += u;
  }
  if (lane == 31) wbuf[warp] = inc;
  __syncthreads();
  long long before = 0, all = 0;
  for (int w = 0; w < kFlWarps; ++w) {
    if (w < warp) before += wbuf[w];
    all += wbuf[w];
  }
  __syncthreads();
  *total = all;
  return before + inc - v;
}

__global__ void __launch_bounds__(kFlThreads) flac_layout_kernel(
    long long S, const int* __restrict__ lens, int rate, const int* __restrict__ recs, long long* __restrict__ offs,
    int F_max, uint8_t* __restrict__ out, long long out_ld, long long row_bytes, long long* __restrict__ out_bytes) {
  pdl_wait();
  __shared__ long long wbuf[kFlWarps];
  __shared__ int mn_s[kFlWarps], mx_s[kFlWarps];
  const int b = blockIdx.x, t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const long long n = fl_len(lens, b, S);
  const int F = (int)((n + kFlBlock - 1) / kFlBlock);
  long long carry = 0;
  int mn = INT_MAX, mx = 0;
  for (int f0 = 0; f0 < F; f0 += kFlThreads) {
    const int f = f0 + t;
    const int sz = f < F ? recs[((long long)b * F_max + f) * kFlRecInts + 12] : 0;
    if (f < F) { mn = min(mn, sz); mx = max(mx, sz); }
    long long tot;
    const long long ex = fl_block_excl_scan(sz, wbuf, &tot);
    if (f < F) offs[(long long)b * F_max + f] = carry + ex;
    carry += tot;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if (lane == 0) { mn_s[warp] = mn; mx_s[warp] = mx; }
  __syncthreads();
  const long long total = 42 + carry;
  uint8_t* row = out + (long long)b * out_ld;
  if (t == 0) {
    for (int w = 1; w < kFlWarps; ++w) { mn = min(mn, mn_s[w]); mx = max(mx, mx_s[w]); }
    if (F == 0) mn = mx = 0;
    out_bytes[b] = total;
    uint8_t h[42];
    const uint8_t magic[8] = {'f', 'L', 'a', 'C', 0x80, 0, 0, 34};
    for (int i = 0; i < 8; ++i) h[i] = magic[i];
    h[8] = h[10] = kFlBlock >> 8;
    h[9] = h[11] = kFlBlock & 255;
    for (int i = 0; i < 3; ++i) {
      h[12 + i] = (uint8_t)(mn >> (16 - 8 * i));
      h[15 + i] = (uint8_t)(mx >> (16 - 8 * i));
    }
    const unsigned long long v = ((unsigned long long)rate << 44) | (15ull << 36) | (unsigned long long)n;
    for (int i = 0; i < 8; ++i) h[18 + i] = (uint8_t)(v >> (56 - 8 * i));
    for (int i = 26; i < 42; ++i) h[i] = 0;
    for (int i = 0; i < 42; ++i) row[i] = h[i];
  }
  fl_store(row + total, max(0LL, row_bytes - total), [](long long) { return (uint8_t)0; }, [](long long) { return 0u; });
}

// ---- launch 3: emit ----------------------------------------------------------------------------------------------
struct FlEmitSmem {
  int x[kFlBlock];
  unsigned long long sums[kFlKs * kFlParts];
  unsigned w[kFlFrameWords];
  unsigned short crc_tab[256];
  long long wbuf[kFlWarps];
  unsigned wx[kFlWarps];
  unsigned char kpar[kFlParts];
  int overflow;
};

// OR the low nbits (<= 32) of v into the frame at bit position pos (MSB first).
__device__ __forceinline__ void fl_put(unsigned* w, long long pos, unsigned v, int nbits) {
  if (nbits <= 0) return;
  const unsigned long long vv = (unsigned long long)(nbits == 32 ? v : (v & ((1u << nbits) - 1u)))
                                << (64 - nbits - (int)(pos & 31));
  const long long i = pos >> 5;
  if (vv >> 32) atomicOr(&w[i], (unsigned)(vv >> 32));
  if ((unsigned)vv) atomicOr(&w[i + 1], (unsigned)vv);
}

__device__ __forceinline__ unsigned fl_byte(const unsigned* w, long long i) {
  return (w[i >> 2] >> (24 - 8 * (int)(i & 3))) & 255u;
}

// a * b mod (x^16 + x^15 + x^2 + 1), a, b < 2^16
__device__ __forceinline__ unsigned fl_gf_mul(unsigned a, unsigned b) {
  unsigned r = 0;
  for (int i = 15; i >= 0; --i) {
    r <<= 1;
    if (r & 0x10000u) r ^= 0x18005u;
    if ((b >> i) & 1u) r ^= a;
  }
  return r;
}

// CRC-16 register c after L more zero bytes: c x^(8 L) mod P
__device__ unsigned fl_crc16_shift(unsigned c, long long L) {
  unsigned p = 0x100u;                                      // x^8
  while (L) {
    if (L & 1) c = fl_gf_mul(c, p);
    p = fl_gf_mul(p, p);
    L >>= 1;
  }
  return c;
}

__global__ void __launch_bounds__(kFlThreads) flac_emit_kernel(
    const int16_t* __restrict__ x, long long x_ld, long long S, const int* __restrict__ lens, int rate,
    const int* __restrict__ recs, const long long* __restrict__ offs, int F_max, uint8_t* __restrict__ out,
    long long out_ld) {
  pdl_wait();
  extern __shared__ __align__(16) unsigned char fl_smem[];
  FlEmitSmem& sm = *reinterpret_cast<FlEmitSmem*>(fl_smem);
  const int b = blockIdx.y, f = blockIdx.x, t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const long long n = fl_len(lens, b, S);
  if ((long long)f * kFlBlock >= n) return;
  const int bs = (int)min((long long)kFlBlock, n - (long long)f * kFlBlock);
  const int* rec = recs + ((long long)b * F_max + f) * kFlRecInts;
  const int kind = rec[0], order = rec[1], porder = rec[2], shift = rec[3], bytes = rec[12];
  int c[kFlMaxLpc];
#pragma unroll
  for (int j = 0; j < kFlMaxLpc; ++j) c[j] = rec[4 + j];
  const int16_t* xb = x + (long long)b * x_ld + (long long)f * kFlBlock;
  for (int i = t; i < bs; i += kFlThreads) sm.x[i] = xb[i];
  for (int i = t; i < kFlFrameWords; i += kFlThreads) sm.w[i] = 0u;
  for (int i = t; i < kFlKs * kFlParts; i += kFlThreads) sm.sums[i] = 0;
  {
    unsigned r = (unsigned)t << 8;                          // CRC-16 table: t x^16 mod P
    for (int i = 0; i < 8; ++i) r = (r & 0x8000u) ? ((r << 1) ^ 0x8005u) & 0xFFFFu : (r << 1) & 0xFFFFu;
    sm.crc_tab[t] = (unsigned short)r;
  }
  if (t == 0) sm.overflow = 0;
  __syncthreads();

  const int hbytes = fl_header_bytes((unsigned)f, bs, rate);
  const long long sub = 8LL * hbytes;
  const bool pred = kind == kFlFixed || kind == kFlLpc;
  if (t == 0) {
    uint8_t h[16];
    const int rc = fl_rate_code(rate);
    h[0] = 0xFF;
    h[1] = 0xF8;
    h[2] = (uint8_t)(((bs == kFlBlock ? 12 : 7) << 4) | rc);
    h[3] = 0x08;
    int k = 4;
    const unsigned fn = (unsigned)f;
    const int nb = fl_utf8_len(fn);
    if (nb == 1) {
      h[k++] = (uint8_t)fn;
    } else {
      h[k++] = (uint8_t)(((0xFF00u >> nb) & 0xFFu) | (fn >> (6 * (nb - 1))));
      for (int i = nb - 2; i >= 0; --i) h[k++] = (uint8_t)(0x80u | ((fn >> (6 * i)) & 0x3Fu));
    }
    if (bs != kFlBlock) { h[k++] = (uint8_t)((bs - 1) >> 8); h[k++] = (uint8_t)((bs - 1) & 255); }
    if (rc == 13) { h[k++] = (uint8_t)(rate >> 8); h[k++] = (uint8_t)(rate & 255); }
    unsigned crc = 0;
    for (int i = 0; i < k; ++i) {
      crc ^= h[i];
      for (int j = 0; j < 8; ++j) crc = (crc & 0x80u) ? ((crc << 1) ^ 0x07u) & 0xFFu : (crc << 1) & 0xFFu;
    }
    h[k++] = (uint8_t)crc;
    for (int i = 0; i < k; ++i) fl_put(sm.w, 8LL * i, h[i], 8);
    const unsigned type = kind == kFlConstant ? 0u : kind == kFlVerbatim ? 1u
                          : kind == kFlFixed ? (8u | (unsigned)order) : (32u | (unsigned)(order - 1));
    fl_put(sm.w, sub, type << 1, 8);
    if (kind == kFlConstant) fl_put(sm.w, sub + 8, (unsigned)(sm.x[0] & 0xFFFF), 16);
    if (kind == kFlLpc) {
      const long long p0 = sub + 8 + 16LL * order;
      fl_put(sm.w, p0, kFlPrecision - 1, 4);
      fl_put(sm.w, p0 + 4, (unsigned)shift, 5);
      for (int j = 0; j < order; ++j) fl_put(sm.w, p0 + 9 + kFlPrecision * j, (unsigned)c[j], kFlPrecision);
    }
  }
  if (kind == kFlVerbatim) {
    for (int i = t; i < bs; i += kFlThreads) fl_put(sm.w, sub + 8 + 16LL * i, (unsigned)(sm.x[i] & 0xFFFF), 16);
  } else if (pred) {
    for (int i = t; i < order; i += kFlThreads) fl_put(sm.w, sub + 8 + 16LL * i, (unsigned)(sm.x[i] & 0xFFFF), 16);
    const long long res0 = sub + 8 + 16LL * order + (kind == kFlLpc ? 4 + 5 + (long long)kFlPrecision * order : 0);
    if (t == 0) fl_put(sm.w, res0, (unsigned)porder, 6);      // method 00, then the 4-bit partition order
    fl_partition_sums(sm.x, bs, order, c, shift, porder, sm.sums, kFlParts, &sm.overflow);
    __syncthreads();
    const int P = 1 << porder, m = bs >> porder;
    if (t < P) {
      const long long cnt = m - (t == 0 ? order : 0);
      long long best = LLONG_MAX;
      int kb = 0;
      for (int k = 0; k < kFlKs; ++k) {
        const long long v = (long long)sm.sums[k * kFlParts + t] + cnt * (1 + k);
        if (v < best) { best = v; kb = k; }
      }
      sm.kpar[t] = (unsigned char)kb;
    }
    __syncthreads();
    // this thread's run of samples [16 t, 16 t + 16): code lengths, then their block-wide offsets
    unsigned long long u[kFlPerThread];
    long long mine = 0;
    bool big = false;
#pragma unroll
    for (int e = 0; e < kFlPerThread; ++e) {
      const int i = kFlPerThread * t + e;
      u[e] = 0;
      if (i >= order && i < bs) {
        u[e] = fl_residual(sm.x, i, order, c, shift, big);
        const int k = sm.kpar[i / m];
        mine += (long long)(u[e] >> k) + 1 + k;
      }
    }
    long long tot;
    long long pos = fl_block_excl_scan(mine, sm.wbuf, &tot);
    const long long codes = res0 + 6;
    if (t == 0) fl_put(sm.w, codes, sm.kpar[0], 4);
#pragma unroll
    for (int e = 0; e < kFlPerThread; ++e) {
      const int i = kFlPerThread * t + e;
      if (i >= order && i < bs) {
        const int p = i / m, k = sm.kpar[p];
        const long long at = codes + 4LL * (p + 1) + pos;
        if (p > 0 && i == p * m) fl_put(sm.w, at - 4, (unsigned)k, 4);
        const unsigned long long q = u[e] >> k;
        fl_put(sm.w, at + (long long)q, (1u << k) | (unsigned)(u[e] & ((1ull << k) - 1ull)), k + 1);
        pos += (long long)q + 1 + k;
      }
    }
  }
  __syncthreads();

  // CRC-16 over bytes [0, L): per-thread runs, moved to the end and XOR-ed together
  const long long L = bytes - 2;
  const long long run = (L + kFlThreads - 1) / kFlThreads, lo = min(L, run * t), hi = min(L, lo + run);
  unsigned crc = 0;
  for (long long i = lo; i < hi; ++i) crc = ((crc << 8) & 0xFFFFu) ^ sm.crc_tab[(crc >> 8) ^ fl_byte(sm.w, i)];
  crc = fl_crc16_shift(crc, L - hi);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) crc ^= __shfl_xor_sync(0xffffffffu, crc, o);
  if (lane == 0) sm.wx[warp] = crc;
  __syncthreads();
  if (t == 0) {
    unsigned all = 0;
    for (int w = 0; w < kFlWarps; ++w) all ^= sm.wx[w];
    fl_put(sm.w, 8 * L, all, 16);
  }
  __syncthreads();
  uint8_t* dst = out + (long long)b * out_ld + 42 + offs[(long long)b * F_max + f];
  const unsigned* w = sm.w;
  fl_store(dst, bytes, [w](long long i) { return (uint8_t)fl_byte(w, i); },
           [w](long long s) {
             const long long i = s >> 2;
             const int r = (int)(s & 3);
             const unsigned be = r ? (w[i] << (8 * r)) | (w[i + 1] >> (32 - 8 * r)) : w[i];
             return __byte_perm(be, 0u, 0x0123);
           });
}

static size_t fl_align(size_t v) { return (v + 255) & ~(size_t)255; }

}  // namespace asb

using namespace asb;

extern "C" size_t as_flac_workspace_bytes(int32_t B, int64_t S) {
  if (B <= 0 || S <= 0) return 0;
  const size_t frames = (size_t)B * (size_t)((S + kFlBlock - 1) / kFlBlock);
  return fl_align(frames * kFlRecInts * sizeof(int)) + fl_align(frames * sizeof(long long));
}

extern "C" int64_t as_flac_max_bytes(int64_t n) {
  if (n < 0) return 0;
  return 42 + 2 * n + 18 * ((n + kFlBlock - 1) / kFlBlock);
}

extern "C" int as_flac_encode(const int16_t* x, int64_t x_ld, int32_t B, int64_t S, const int32_t* lens,
                              int32_t sample_rate, void* workspace, size_t workspace_bytes, uint8_t* out,
                              int64_t out_ld, int64_t* out_bytes, void* stream) {
  if (B == 0) return AS_OK;
  const int64_t row = as_flac_max_bytes(S);
  ASB_REQUIRE(B > 0 && B <= 65535 && S >= 0 && S < (1LL << 31) && out && out_bytes && out_ld >= row &&
              (S == 0 || (x && x_ld >= S)), AS_ERR_SHAPE, "as_flac_encode: bad argument");
  ASB_REQUIRE(sample_rate >= 1 && sample_rate <= 65535, AS_ERR_SHAPE,
              "as_flac_encode: sample_rate %d outside 1 .. 65535 Hz", sample_rate);
  ASB_REQUIRE(S == 0 || (workspace && workspace_bytes >= as_flac_workspace_bytes(B, S)), AS_ERR_WORKSPACE,
              "as_flac_encode: workspace of %zu bytes, %zu needed", workspace_bytes, as_flac_workspace_bytes(B, S));
  ASB_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, AS_ERR_ALIGN,
              "as_flac_encode: the workspace must be 256-byte aligned");
  if (int rc = check_arch()) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int F_max = (int)((S + kFlBlock - 1) / kFlBlock);
  char* ws = static_cast<char*>(workspace);
  int* recs = reinterpret_cast<int*>(ws);
  long long* offs = reinterpret_cast<long long*>(ws + fl_align((size_t)B * F_max * kFlRecInts * sizeof(int)));
  const dim3 grid((unsigned)max(F_max, 1), (unsigned)B);   // S = 0: every CTA returns at once (42-byte rows)
  ASB_SMEM_OPT_IN((int)sizeof(FlAnalysisSmem), flac_analysis_kernel);
  ASB_CUDA(launch_k(flac_analysis_kernel, grid, dim3(kFlThreads), sizeof(FlAnalysisSmem), st, x, (long long)x_ld,
                    (long long)S, lens, (int)sample_rate, recs, F_max));
  ASB_CUDA(launch_k(flac_layout_kernel, dim3((unsigned)B), dim3(kFlThreads), 0, st, (long long)S, lens,
                    (int)sample_rate, (const int*)recs, offs, F_max, out, (long long)out_ld, (long long)row,
                    reinterpret_cast<long long*>(out_bytes)));
  ASB_SMEM_OPT_IN((int)sizeof(FlEmitSmem), flac_emit_kernel);
  ASB_CUDA(launch_k(flac_emit_kernel, grid, dim3(kFlThreads), sizeof(FlEmitSmem), st, x, (long long)x_ld,
                    (long long)S, lens, (int)sample_rate, (const int*)recs, (const long long*)offs, F_max, out,
                    (long long)out_ld));
  return AS_OK;
}
