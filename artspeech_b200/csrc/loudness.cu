// Loudness meter (artspeech_b200/audio.py, header: as_loudness_measure): ITU-R BS.1770 integrated loudness with
// K-weighting and two-stage gating, the 4x oversampled true peak, and the normalisation gain, per utterance, on the
// device, so the output-format stage can apply the gain before it quantises (audio_out.cu).
//
// K-weighting is a linear recurrence on a 4-dimensional state v (two transposed direct-form-II biquads, fp64):
// v' = M v + (input terms).  Over a run of c samples the state is v_end = M^c v_start + f, where f is the run
// filtered from zero state, so the recurrence is a scan of affine maps whose matrices are powers of M.  The powers
// M^(c 2^i), M^(g 2^i), M^(8 g 2^i) (c: samples per lane, g: samples per 100 ms segment) are computed on the host in
// fp64 and passed by value.  Three launches:
//   1. grid (tile, utterance), 8 warps, one warp per segment, lane k filters the sub-chunk [k c, (k+1) c) of its
//      segment from zero state.  A Hillis-Steele scan over lanes (M^(c 2^i)) and over the 8 warps (M^(g 2^i)) gives
//      each lane's start state relative to the tile, and the tile's end state from zero (its aggregate).  The same
//      pass reads the samples for the 4x true peak (21 fp32 taps per phase) and writes the tile's peak.
//   2. same grid: the tile's true start state is the sum over earlier tiles u of M^(8 g (t-1-u)) agg_u (binary
//      powers, a fixed-shape tree), propagated to each lane by the binary powers of its warp and lane index; each
//      lane re-filters its sub-chunk from that state and the warp sums y^2 into the segment energy.
//   3. one CTA per utterance: block energies, the two gates, the peak and the gain, in fp64.
// No thread runs a chain longer than c samples (c = g / P with P the largest divisor of g up to 32: 75 at 24 kHz).
// Every sum has a shape fixed by the utterance's own sample and segment indices (no atomics), so the results do not
// depend on B, S, x_ld or the batch-mates.  Samples are staged per warp in rounds of 32 steps of every lane (rows of
// 32 + 2 * 10 samples with the true peak's halo, zero outside [0, n)), read column-wise without bank conflicts.
#include <math_constants.h>

#include "common.cuh"

namespace asb {

constexpr int kLdWarps = 8;                          // segments per CTA (a tile)
constexpr int kLdThreads = kLdWarps * 32;
constexpr int kLdSteps = 32;                         // samples per lane per staging round
constexpr int kLdHalo = 10;                          // true-peak taps reach x[q - 10 .. q + 10]
constexpr int kLdTaps = 21;
constexpr int kLdRow = kLdSteps + 2 * kLdHalo + 1;   // 53: odd, so a column read hits 32 distinct banks
constexpr int kLdTileBits = 12;                      // AS_LOUDNESS_MAX_TILES = 2^12
constexpr int kLdBatch = 8;                          // staging loads in flight per lane
constexpr size_t kLdSmem = sizeof(float) * kLdWarps * 32 * kLdRow;

struct LoudParams {
  double kw[10];                   // shelf b0 b1 b2 a1 a2, high-pass b0 b1 b2 a1 a2
  double p_lane[5][16];            // M^(c 2^i), row-major 4x4
  double p_seg[3][16];             // M^(g 2^i)
  double p_tile[kLdTileBits][16];  // M^(8 g 2^i)
  float tp[4][kLdTaps];            // 4x true-peak polyphase taps
  int seg, c, P;
};

__device__ __forceinline__ void ld_matvec(const double* m, double v[4]) {
  double o[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) o[r] = fma(m[4 * r], v[0], fma(m[4 * r + 1], v[1], fma(m[4 * r + 2], v[2], m[4 * r + 3] * v[3])));
#pragma unroll
  for (int r = 0; r < 4; ++r) v[r] = o[r];
}

__device__ __forceinline__ void ld_shfl_up(const double v[4], double o[4], int d) {
#pragma unroll
  for (int r = 0; r < 4; ++r) o[r] = __shfl_up_sync(0xffffffffu, v[r], d);
}

// one sample through both biquads (transposed direct form II); returns the K-weighted output
__device__ __forceinline__ double ld_step(const LoudParams& p, double x, double v[4]) {
  const double y1 = fma(p.kw[0], x, v[0]);
  v[0] = fma(p.kw[1], x, fma(-p.kw[3], y1, v[1]));
  v[1] = fma(p.kw[2], x, -p.kw[4] * y1);
  const double y2 = fma(p.kw[5], y1, v[2]);
  v[2] = fma(p.kw[6], y1, fma(-p.kw[8], y2, v[3]));
  v[3] = fma(p.kw[7], y1, -p.kw[9] * y2);
  return y2;
}

// Run lane `lane`'s sub-chunk of the segment starting at s0 through the filter from state v (kEnergy: returns the
// sum of y^2 in sample order; kPeak: the largest |x| and |y4| in *peak).  Rows are staged by the whole warp.
template <bool kPeak, bool kEnergy>
__device__ __forceinline__ double ld_chunk(const LoudParams& p, const float* __restrict__ xb, long long n,
                                           long long s0, int lane, float* row, double v[4], float* peak) {
  const int c = p.c, P = p.P;
  double acc = 0.0;
  float pk = 0.f;
  const long long q0 = s0 + (long long)lane * c;
  constexpr int halo = kPeak ? kLdHalo : 0;
  for (int r0 = 0; r0 < c; r0 += kLdSteps) {
    const int steps = min(kLdSteps, c - r0);
    __syncwarp();
    // P rows of wr samples, flattened over the warp; kLdBatch loads in flight per lane before their stores
    const int wr = steps + 2 * halo, total = P * wr;
    for (int i0 = 0; i0 < total; i0 += 32 * kLdBatch) {
      float val[kLdBatch];
#pragma unroll
      for (int u = 0; u < kLdBatch; ++u) {
        const int idx = i0 + u * 32 + lane;
        const int k = idx / wr;
        const long long i = s0 + (long long)k * c + r0 - halo + (idx - k * wr);
        val[u] = idx < total && i >= 0 && i < n ? __ldg(xb + i) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < kLdBatch; ++u) {
        const int idx = i0 + u * 32 + lane;
        const int k = idx / wr;
        if (idx < total) row[k * kLdRow + idx - k * wr] = val[u];
      }
    }
    __syncwarp();
    if (lane < P) {
      const float* w = row + lane * kLdRow + halo;
      const int m = (int)min((long long)steps, n - (q0 + r0));
      for (int t = 0; t < m; ++t) {
        const float xv = w[t];
        const double y = ld_step(p, (double)xv, v);
        if (kEnergy) acc = fma(y, y, acc);
        if (kPeak) {
          pk = fmaxf(pk, fabsf(xv));
#pragma unroll
          for (int ph = 0; ph < 4; ++ph) {
            float a = 0.f;
#pragma unroll
            for (int j = 0; j < kLdTaps; ++j) a = fmaf(p.tp[ph][j], w[t + kLdHalo - j], a);
            pk = fmaxf(pk, fabsf(a));
          }
        }
      }
    }
  }
  if (kPeak) *peak = pk;
  return acc;
}

__device__ __forceinline__ long long ld_len(const int* lens, int b, long long S) {
  return lens ? min((long long)max(lens[b], 0), S) : S;
}

__global__ void __launch_bounds__(kLdThreads) loudness_pass1_kernel(
    const float* __restrict__ x, long long x_ld, long long S, const int* __restrict__ lens, const LoudParams p,
    int tiles, double* __restrict__ lane_st, double* __restrict__ seg_in, double* __restrict__ agg,
    float* __restrict__ peak) {
  pdl_wait();
  extern __shared__ __align__(16) float ld_smem[];
  __shared__ double s_seg[kLdWarps][4];
  __shared__ float s_pk[kLdWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t = blockIdx.x, b = blockIdx.y;
  const long long n = ld_len(lens, b, S);
  const long long tile0 = (long long)t * kLdWarps * p.seg;
  if (tile0 >= n) return;
  const long long s0 = tile0 + (long long)warp * p.seg;
  double v[4] = {0.0, 0.0, 0.0, 0.0};
  float pk = 0.f;
  if (s0 < n)
    ld_chunk<true, false>(p, x + (long long)b * x_ld, n, s0, lane, ld_smem + warp * 32 * kLdRow, v, &pk);
  if (lane >= p.P) v[0] = v[1] = v[2] = v[3] = 0.0;
  // inclusive scan over the lanes: v_k = sum_{j <= k} M^(c (k - j)) f_j
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    double o[4];
    ld_shfl_up(v, o, 1 << i);
    if (lane >= (1 << i)) {
      ld_matvec(p.p_lane[i], o);
#pragma unroll
      for (int r = 0; r < 4; ++r) v[r] += o[r];
    }
  }
  double e[4];
  ld_shfl_up(v, e, 1);                                   // state at the start of the lane's sub-chunk
  const long long sidx = ((long long)b * tiles + t) * kLdWarps + warp;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const double agg_seg = __shfl_sync(0xffffffffu, v[r], p.P - 1);
    lane_st[(sidx * 32 + lane) * 4 + r] = lane == 0 ? 0.0 : e[r];
    if (lane == 0) s_seg[warp][r] = agg_seg;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) pk = fmaxf(pk, __shfl_xor_sync(0xffffffffu, pk, o));
  if (lane == 0) s_pk[warp] = pk;
  __syncthreads();
  if (warp == 0) {
    // scan over the segments: V_w = sum_{u <= w} M^(g (w - u)) F_u
    double V[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) V[r] = lane < kLdWarps ? s_seg[lane][r] : 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      double o[4];
      ld_shfl_up(V, o, 1 << i);
      if (lane >= (1 << i)) {
        ld_matvec(p.p_seg[i], o);
#pragma unroll
        for (int r = 0; r < 4; ++r) V[r] += o[r];
      }
    }
    double Vin[4];
    ld_shfl_up(V, Vin, 1);
    const long long tidx = (long long)b * tiles + t;
    if (lane < kLdWarps) {
#pragma unroll
      for (int r = 0; r < 4; ++r) seg_in[(tidx * kLdWarps + lane) * 4 + r] = lane == 0 ? 0.0 : Vin[r];
    }
    if (lane == kLdWarps - 1) {
#pragma unroll
      for (int r = 0; r < 4; ++r) agg[tidx * 4 + r] = V[r];
    }
    if (lane == 0) {
      float m = 0.f;
      for (int w = 0; w < kLdWarps; ++w) m = fmaxf(m, s_pk[w]);
      peak[tidx] = m;
    }
  }
}

__global__ void __launch_bounds__(kLdThreads, 1) loudness_pass2_kernel(
    const float* __restrict__ x, long long x_ld, long long S, const int* __restrict__ lens, const LoudParams p,
    int tiles, const double* __restrict__ lane_st, const double* __restrict__ seg_in, const double* __restrict__ agg,
    double* __restrict__ energy) {
  pdl_wait();
  extern __shared__ __align__(16) float ld_smem[];
  __shared__ double s_red[kLdWarps][4];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t = blockIdx.x, b = blockIdx.y;
  const long long n = ld_len(lens, b, S);
  const long long tile0 = (long long)t * kLdWarps * p.seg;
  if (tile0 >= n) return;
  // the tile's start state: sum over u < t of M^(8 g (t - 1 - u)) agg_u; thread i takes u = i, i + 256, ... in order
  const long long tb = (long long)b * tiles;
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  for (int u = threadIdx.x; u < t; u += kLdThreads) {
    double a[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) a[r] = agg[(tb + u) * 4 + r];
    const int ex = t - 1 - u;
#pragma unroll
    for (int i = 0; i < kLdTileBits; ++i)
      if ((ex >> i) & 1) ld_matvec(p.p_tile[i], a);
#pragma unroll
    for (int r = 0; r < 4; ++r) acc[r] += a[r];
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[r] += __shfl_down_sync(0xffffffffu, acc[r], o);
    if (lane == 0) s_red[warp][r] = acc[r];
  }
  __syncthreads();
  double G[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    double s = s_red[0][r];
    for (int w = 1; w < kLdWarps; ++w) s += s_red[w][r];
    G[r] = s;
  }
  const long long s0 = tile0 + (long long)warp * p.seg;
  if (s0 >= n) return;                                   // warp-uniform; no block-wide barrier follows
  // segment start state: seg_in_w + M^(g w) S_in; lane start state: lane_st + M^(c k) (segment start state)
  const long long sidx = (tb + t) * kLdWarps + warp;
#pragma unroll
  for (int i = 0; i < 3; ++i)
    if ((warp >> i) & 1) ld_matvec(p.p_seg[i], G);
#pragma unroll
  for (int r = 0; r < 4; ++r) G[r] += seg_in[sidx * 4 + r];
#pragma unroll
  for (int i = 0; i < 5; ++i)
    if ((lane >> i) & 1) ld_matvec(p.p_lane[i], G);
  double v[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) v[r] = G[r] + lane_st[(sidx * 32 + lane) * 4 + r];
  double e = ld_chunk<false, true>(p, x + (long long)b * x_ld, n, s0, lane, ld_smem + warp * 32 * kLdRow, v,
                                   nullptr);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) e += __shfl_down_sync(0xffffffffu, e, o);
  if (lane == 0) energy[sidx] = e;
}

// fixed-shape block reduction of (sum, count) over kLdThreads threads
__device__ __forceinline__ void ld_block_sum(double& s, int& cnt, double* rs, int* rc) {
  const int tid = threadIdx.x;
  rs[tid] = s;
  rc[tid] = cnt;
  __syncthreads();
  for (int h = kLdThreads / 2; h > 0; h >>= 1) {
    if (tid < h) {
      rs[tid] += rs[tid + h];
      rc[tid] += rc[tid + h];
    }
    __syncthreads();
  }
  s = rs[0];
  cnt = rc[0];
  __syncthreads();
}

__device__ __forceinline__ double ld_block_z(const double* E, long long j, double inv) {
  return (((E[j] + E[j + 1]) + E[j + 2]) + E[j + 3]) * inv;
}

__global__ void __launch_bounds__(kLdThreads) loudness_final_kernel(
    long long S, const int* __restrict__ lens, int seg, int tiles, const double* __restrict__ energy,
    const float* __restrict__ peak, double target, double ceiling, double* __restrict__ loud_out,
    double* __restrict__ tp_out, double* __restrict__ gdb_out, float* __restrict__ g_out) {
  pdl_wait();
  __shared__ double rs[kLdThreads];
  __shared__ int rc[kLdThreads];
  const int b = blockIdx.x, tid = threadIdx.x;
  const long long n = ld_len(lens, b, S);
  const double* E = energy + (long long)b * tiles * kLdWarps;
  const double ninf = -CUDART_INF;
  const long long nfull = n / seg;
  // blocks: j = 0 .. nfull - 4, or one block over all n samples when n < 4 g
  const long long nb = n == 0 ? 0 : nfull >= 4 ? nfull - 3 : 1;
  const bool single = n > 0 && nfull < 4;
  double z1 = 0.0;
  if (single) {
    const long long ns = (n + seg - 1) / seg;
    for (long long s = 0; s < ns; ++s) z1 += E[s];
    z1 /= (double)n;
  }
  const double inv = 1.0 / (4.0 * seg);
  double sa = 0.0;
  int ca = 0;
  for (long long j = tid; j < nb; j += kLdThreads) {
    const double z = single ? z1 : ld_block_z(E, j, inv);
    if (-0.691 + 10.0 * log10(z) > -70.0) { sa += z; ++ca; }
  }
  ld_block_sum(sa, ca, rs, rc);
  double L = ninf;
  if (ca > 0) {
    const double gate = -0.691 + 10.0 * log10(sa / ca) - 10.0;
    double sg = 0.0;
    int cg = 0;
    for (long long j = tid; j < nb; j += kLdThreads) {
      const double z = single ? z1 : ld_block_z(E, j, inv);
      const double Lj = -0.691 + 10.0 * log10(z);
      if (Lj > -70.0 && Lj > gate) { sg += z; ++cg; }
    }
    ld_block_sum(sg, cg, rs, rc);
    L = -0.691 + 10.0 * log10(sg / cg);
  }
  if (tid == 0) {
    const long long nt = (n + (long long)kLdWarps * seg - 1) / ((long long)kLdWarps * seg);
    float pk = 0.f;
    for (long long u = 0; u < nt; ++u) pk = fmaxf(pk, peak[(long long)b * tiles + u]);
    const double tp = pk > 0.f ? 20.0 * log10((double)pk) : ninf;
    const double gdb = L == ninf ? 0.0 : fmin(target - L, ceiling - tp);
    loud_out[b] = L;
    tp_out[b] = tp;
    if (gdb_out) gdb_out[b] = gdb;
    if (g_out) g_out[b] = (float)pow(10.0, gdb / 20.0);
  }
}

// ---- host side ----------------------------------------------------------------------------------------------------
static void ld_matmul(const double* a, const double* b, double* o) {
  double t[16];
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c) {
      double s = 0.0;
      for (int k = 0; k < 4; ++k) s += a[4 * r + k] * b[4 * k + c];
      t[4 * r + c] = s;
    }
  memcpy(o, t, sizeof(t));
}

static void ld_matpow(const double* m, long long e, double* o) {
  double r[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1}, b[16];
  memcpy(b, m, sizeof(b));
  for (; e > 0; e >>= 1) {
    if (e & 1) ld_matmul(r, b, r);
    ld_matmul(b, b, b);
  }
  memcpy(o, r, sizeof(r));
}

struct LdLayout {
  size_t lane_st, seg_in, agg, energy, peak, total;
};

static size_t ld_align(size_t v) { return (v + 255) & ~(size_t)255; }

static LdLayout ld_layout(long long B, long long tiles) {
  LdLayout l;
  const long long segs = B * tiles * kLdWarps;
  l.lane_st = 0;
  l.seg_in = l.lane_st + ld_align(sizeof(double) * segs * 32 * 4);
  l.agg = l.seg_in + ld_align(sizeof(double) * segs * 4);
  l.energy = l.agg + ld_align(sizeof(double) * B * tiles * 4);
  l.peak = l.energy + ld_align(sizeof(double) * segs);
  l.total = l.peak + ld_align(sizeof(float) * B * tiles);
  return l;
}

static long long ld_tiles(long long S, int fs) {
  const long long tile = (long long)kLdWarps * (fs / 10);
  return std::max(1LL, (S + tile - 1) / tile);
}

static bool ld_rate_ok(int fs) { return fs >= 8000 && fs <= 192000 && fs % 10 == 0; }

}  // namespace asb

using namespace asb;

extern "C" size_t as_loudness_workspace_bytes(int32_t B, int64_t S, int32_t fs) {
  if (B <= 0 || S < 0 || !ld_rate_ok(fs)) return 0;
  return ld_layout(B, ld_tiles(S, fs)).total;
}

extern "C" int as_loudness_measure(const float* x, int64_t x_ld, int32_t B, int64_t S, const int32_t* lens, int32_t fs,
                                   const double* kw, const float* tp_table, double target, double ceiling,
                                   void* workspace, size_t workspace_bytes, double* loudness_out,
                                   double* true_peak_out, double* gain_db_out, float* gain_out, void* stream) {
  if (B == 0) return AS_OK;
  ASB_REQUIRE(B > 0 && B <= 65535 && S >= 0 && x_ld >= S && (x || S == 0) && kw && tp_table && loudness_out &&
                  true_peak_out,
              AS_ERR_SHAPE, "as_loudness_measure: bad argument");
  ASB_REQUIRE(ld_rate_ok(fs), AS_ERR_SHAPE, "as_loudness_measure: fs %d Hz is not a multiple of 10 in [8000, 192000]",
              (int)fs);
  const long long tiles = ld_tiles(S, fs);
  ASB_REQUIRE(tiles <= AS_LOUDNESS_MAX_TILES, AS_ERR_SHAPE,
              "as_loudness_measure: %lld samples at %d Hz exceed %d tiles of 8 segments", (long long)S, (int)fs,
              AS_LOUDNESS_MAX_TILES);
  const LdLayout lay = ld_layout(B, tiles);
  ASB_REQUIRE(workspace && workspace_bytes >= lay.total, AS_ERR_WORKSPACE,
              "as_loudness_measure: workspace of %zu bytes, %zu needed", workspace_bytes, lay.total);
  ASB_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, AS_ERR_ALIGN,
              "as_loudness_measure: the workspace must be 256-byte aligned");
  if (int rc = check_arch()) return rc;

  LoudParams p;
  memset(&p, 0, sizeof(p));
  memcpy(p.kw, kw, sizeof(p.kw));
  p.seg = fs / 10;
  p.P = 1;
  for (int d = 32; d >= 1; --d)
    if (p.seg % d == 0) { p.P = d; break; }
  p.c = p.seg / p.P;
  // zero-input transition of the state (s1, s2, t1, t2) as ld_step updates it
  const double* k = p.kw;
  const double M[16] = {-k[3], 1.0, 0.0, 0.0,
                        -k[4], 0.0, 0.0, 0.0,
                        k[6] - k[8] * k[5], 0.0, -k[8], 1.0,
                        k[7] - k[9] * k[5], 0.0, -k[9], 0.0};
  ld_matpow(M, p.c, p.p_lane[0]);
  for (int i = 1; i < 5; ++i) ld_matmul(p.p_lane[i - 1], p.p_lane[i - 1], p.p_lane[i]);
  ld_matpow(M, p.seg, p.p_seg[0]);
  for (int i = 1; i < 3; ++i) ld_matmul(p.p_seg[i - 1], p.p_seg[i - 1], p.p_seg[i]);
  ld_matmul(p.p_seg[2], p.p_seg[2], p.p_tile[0]);                 // M^(8 g)
  for (int i = 1; i < kLdTileBits; ++i) ld_matmul(p.p_tile[i - 1], p.p_tile[i - 1], p.p_tile[i]);
  for (int r = 0; r < 4; ++r)
    for (int j = 0; j < kLdTaps; ++j) p.tp[r][j] = tp_table[r * AS_LOUDNESS_TP_LD + j];

  char* ws = static_cast<char*>(workspace);
  double* lane_st = reinterpret_cast<double*>(ws + lay.lane_st);
  double* seg_in = reinterpret_cast<double*>(ws + lay.seg_in);
  double* agg = reinterpret_cast<double*>(ws + lay.agg);
  double* energy = reinterpret_cast<double*>(ws + lay.energy);
  float* peak = reinterpret_cast<float*>(ws + lay.peak);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const dim3 grid((unsigned)tiles, (unsigned)B);
  ASB_SMEM_OPT_IN(kLdSmem, loudness_pass1_kernel);
  ASB_SMEM_OPT_IN(kLdSmem, loudness_pass2_kernel);
  ASB_CUDA(launch_k(loudness_pass1_kernel, grid, dim3(kLdThreads), kLdSmem, st, x, (long long)x_ld, (long long)S,
                    lens, p, (int)tiles, lane_st, seg_in, agg, peak));
  ASB_CUDA(launch_k(loudness_pass2_kernel, grid, dim3(kLdThreads), kLdSmem, st, x, (long long)x_ld, (long long)S,
                    lens, p, (int)tiles, (const double*)lane_st, (const double*)seg_in, (const double*)agg, energy));
  ASB_CUDA(launch_k(loudness_final_kernel, dim3((unsigned)B), dim3(kLdThreads), 0, st, (long long)S, lens,
                    (int)p.seg, (int)tiles, (const double*)energy, (const float*)peak, target, ceiling, loudness_out,
                    true_peak_out, gain_db_out, gain_out));
  return AS_OK;
}
