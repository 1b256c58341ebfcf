// Output audio formats (artspeech_b200/audio.py): polyphase resampling of the vocoder's 24 kHz fp32 waveforms to
// another rate and encoding to fp32 / 16-bit PCM / G.711 mu-law / A-law, in one HBM pass.  It runs after the
// synthesis graph, so a caller gets the bytes it will send (8 kHz mu-law is 1/4 of the fp32 24 kHz stream's bytes
// per second of audio, 1/12 of its size) without a device->host copy of the fp32 samples and a CPU resampler.
//
// One CTA per (utterance, tile of AS_AUDIO_TILE output samples), grid-stride beyond 16 waves.  The CTA stages the
// polyphase table once and, per tile, the input window the tile reads (16-byte loads, zero outside [0, n_in)),
// computes 4 outputs per thread (consecutive threads take consecutive outputs: the window reads are spread over
// the banks), encodes them into a shared-memory row and writes that row with 16-byte stores.  Each output is one
// fp32 fma chain over the taps j = 0..K-1 in that order, so its bits depend on its utterance's samples and its
// index only: not on B, S_in, the tile or the output offset m0 (batch invariance, chunked == one-shot output).
// With a per-utterance gain (loudness normalisation, loudness.cu) the value is multiplied by gain[b] once, in fp32,
// before it is encoded; the kernel is a template on whether there is a gain, so the gain-free path is unchanged.
#include "common.cuh"
#include "tc_util.cuh"

namespace asb {

constexpr int kAudioThreads = 256;
constexpr int kAudioTile = AS_AUDIO_TILE;
constexpr int kAudioPer = kAudioTile / kAudioThreads;       // outputs per thread per tile

// libsndfile's float -> PCM_16 as the vocoder's AS_PCM16 epilogue writes it (conv_cout1.cu): saturated lrint(32767 y)
__host__ __device__ __forceinline__ int audio_pcm16(float y) {
#ifdef __CUDA_ARCH__
  return max(-32768, min(32767, __float2int_rn(y * 32767.f)));
#else
  const float v = rintf(y * 32767.f);
  return v != v ? 0 : v < -32768.f ? -32768 : v > 32767.f ? 32767 : (int)v;
#endif
}

__host__ __device__ __forceinline__ int audio_bits(unsigned v) {       // position of the highest set bit + 1
#ifdef __CUDA_ARCH__
  return 32 - __clz((int)v);
#else
  int n = 0;
  while (v) { ++n; v >>= 1; }
  return n;
#endif
}

// ITU-T G.711 mu-law of a 16-bit sample (CPython audioop.lin2ulaw, width 2: st_14linear2ulaw(s >> 2)).  The segment
// search over {0x3F, 0x7F, ..., 0x1FFF} is the bit length of the biased magnitude minus 6.
__host__ __device__ __forceinline__ unsigned audio_ulaw(int s) {
  int v = s >> 2;
  unsigned mask = 0xFFu;
  if (v < 0) { v = -v; mask = 0x7Fu; }
  v = (v > 8159 ? 8159 : v) + 33;
  int seg = audio_bits((unsigned)v) - 6;
  seg = seg < 0 ? 0 : seg;
  if (seg >= 8) return 0x7Fu ^ mask;
  return ((unsigned)(seg << 4) | ((unsigned)(v >> (seg + 1)) & 0xFu)) ^ mask;
}

// ITU-T G.711 A-law (audioop.lin2alaw, width 2: st_linear2alaw(s >> 3)); segments {0x1F, ..., 0xFFF}.
__host__ __device__ __forceinline__ unsigned audio_alaw(int s) {
  int v = s >> 3;
  unsigned mask = 0xD5u;
  if (v < 0) { v = -v - 1; mask = 0x55u; }
  int seg = audio_bits((unsigned)v) - 5;
  seg = seg < 0 ? 0 : seg;
  if (seg >= 8) return 0x7Fu ^ mask;
  const unsigned q = (unsigned)(seg < 2 ? v >> 1 : v >> seg) & 0xFu;
  return ((unsigned)(seg << 4) | q) ^ mask;
}

__device__ __forceinline__ void audio_put(unsigned char* row, int r, float y, int enc) {
  switch (enc) {
    case AS_AUDIO_F32:   reinterpret_cast<float*>(row)[r] = y; break;
    case AS_AUDIO_PCM16: reinterpret_cast<int16_t*>(row)[r] = (int16_t)audio_pcm16(y); break;
    case AS_AUDIO_MULAW: row[r] = (unsigned char)audio_ulaw(audio_pcm16(y)); break;
    default:             row[r] = (unsigned char)audio_alaw(audio_pcm16(y)); break;
  }
}

template <bool kIdentity, bool kGain>
__global__ void __launch_bounds__(kAudioThreads) resample_encode_kernel(
    const float* __restrict__ x, long long x_ld, int S_in, const int* __restrict__ in_lens,
    const float* __restrict__ table, int table_ld, int up, int down, int K, int half_len, int m0, int S_out,
    unsigned char* __restrict__ out, long long out_ld, int enc, int* __restrict__ out_lens,
    const float* __restrict__ gain, int B, int tiles, int win_alloc, int vec_in, int vec_out) {
  pdl_wait();
  extern __shared__ __align__(16) float audio_smem[];
  float* tab = audio_smem;                                        // [up][table_ld]
  float* xw = tab + (kIdentity ? 0 : up * table_ld);              // [win_alloc] input window
  unsigned char* ys = reinterpret_cast<unsigned char*>(xw + win_alloc);   // [kAudioTile] encoded outputs
  const int tid = threadIdx.x;
  const int es = enc == AS_AUDIO_F32 ? 4 : enc == AS_AUDIO_PCM16 ? 2 : 1;
  if (!kIdentity)
    for (int i = tid; i < (up * table_ld) >> 2; i += kAudioThreads)
      reinterpret_cast<float4*>(tab)[i] = __ldg(reinterpret_cast<const float4*>(table) + i);
  // phase / input-index step between a thread's outputs (kAudioThreads apart): one division per thread
  const int si = (kAudioThreads * down) / up, sp = (kAudioThreads * down) % up;

  for (int w = blockIdx.x; w < B * tiles; w += gridDim.x) {
    const int b = w / tiles, r0 = (w - b * tiles) * kAudioTile;
    const int n_in = in_lens ? min(max(in_lens[b], 0), S_in) : S_in;
    const int n_out = (int)(((long long)n_in * up + down - 1) / down);
    if (r0 == 0 && tid == 0 && out_lens) out_lens[b] = n_out;
    const int nr = min(kAudioTile, S_out - r0);                   // outputs of this tile
    const int mt = m0 + r0;
    const int nv = max(0, min(nr, n_out - mt));                   // of which inside the utterance
    const float* xb = x + (long long)b * x_ld;
    const float g = kGain ? gain[b] : 1.f;
    __syncthreads();                                              // the previous tile's window / row are consumed
    int i_al = 0;
    if (nv > 0) {
      // input window [i_lo, i_hi] of the tile's outputs, from a multiple of 4 (16-byte loads)
      const int i_lo = kIdentity ? mt : (mt * down + half_len) / up - (K - 1);
      const int i_hi = kIdentity ? mt + nv - 1 : ((mt + nv - 1) * down + half_len) / up;
      i_al = i_lo & ~3;
      const int nq = ((i_hi - i_al) >> 2) + 1;
      for (int q = tid; q < nq; q += kAudioThreads) {
        const int i = i_al + 4 * q;
        float4 v;
        if (vec_in && i >= 0 && i + 3 < n_in) {
          v = __ldg(reinterpret_cast<const float4*>(xb + i));
        } else {
          v.x = i >= 0 && i < n_in ? xb[i] : 0.f;
          v.y = i + 1 >= 0 && i + 1 < n_in ? xb[i + 1] : 0.f;
          v.z = i + 2 >= 0 && i + 2 < n_in ? xb[i + 2] : 0.f;
          v.w = i + 3 >= 0 && i + 3 < n_in ? xb[i + 3] : 0.f;
        }
        reinterpret_cast<float4*>(xw)[q] = v;
      }
    }
    __syncthreads();
    if (kIdentity) {
#pragma unroll
      for (int o = 0; o < kAudioPer; ++o) {
        const int r = tid + o * kAudioThreads;
        if (r < nr) audio_put(ys, r, r < nv ? (kGain ? xw[mt + r - i_al] * g : xw[mt + r - i_al]) : 0.f, enc);
      }
    } else {
      const int n = (mt + tid) * down + half_len;
      int i0 = n / up, p = n - (n / up) * up;
#pragma unroll
      for (int o = 0; o < kAudioPer; ++o) {
        const int r = tid + o * kAudioThreads;
        if (r < nv) {
          const float* h = tab + p * table_ld;
          const float* xp = xw + (i0 - i_al);
          float acc = 0.f;
          int j = 0;
          for (; j + 4 <= K; j += 4) {
            const float4 h4 = *reinterpret_cast<const float4*>(h + j);
            acc = fmaf(h4.x, xp[-j], acc);
            acc = fmaf(h4.y, xp[-j - 1], acc);
            acc = fmaf(h4.z, xp[-j - 2], acc);
            acc = fmaf(h4.w, xp[-j - 3], acc);
          }
          for (; j < K; ++j) acc = fmaf(h[j], xp[-j], acc);
          audio_put(ys, r, kGain ? acc * g : acc, enc);
        } else if (r < nr) {
          audio_put(ys, r, 0.f, enc);                             // silence: the code of 0
        }
        i0 += si;
        p += sp;
        if (p >= up) { p -= up; ++i0; }
      }
    }
    __syncthreads();
    unsigned char* ob = out + ((long long)b * out_ld + r0) * es;
    const int nbytes = nr * es;
    int done = 0;
    if (vec_out) {
      const int n16 = nbytes >> 4;
      for (int q = tid; q < n16; q += kAudioThreads)
        reinterpret_cast<uint4*>(ob)[q] = reinterpret_cast<const uint4*>(ys)[q];
      done = n16 << 4;
    }
    for (int i = done / es + tid; i < nr; i += kAudioThreads) {   // the row's unaligned part, element by element
      if (es == 4) reinterpret_cast<float*>(ob)[i] = reinterpret_cast<const float*>(ys)[i];
      else if (es == 2) reinterpret_cast<int16_t*>(ob)[i] = reinterpret_cast<const int16_t*>(ys)[i];
      else ob[i] = ys[i];
    }
  }
}

// shared memory of a launch: table, input window, encoded row (audio.py smem_bytes restates this)
static size_t audio_window(int up, int down, int K) {
  const long long w = ((long long)(kAudioTile - 1) * down + up - 1) / up + K + 8;
  return (size_t)((w + 3) & ~3LL);
}

}  // namespace asb

using namespace asb;

extern "C" size_t as_resample_smem_bytes(int32_t up, int32_t down, int32_t K, int32_t table_ld) {
  if (up <= 0 || down <= 0 || K <= 0 || table_ld < K) return 0;
  const bool ident = up == 1 && down == 1;
  return sizeof(float) * ((ident ? 0 : (size_t)up * table_ld) + audio_window(up, down, ident ? 1 : K)) +
         (size_t)kAudioTile * 4;
}

template <bool kGain>
static int resample_encode_launch(const float* x, int64_t x_ld, int32_t B, int32_t S_in, const int32_t* in_lens,
                                  const float* table, int32_t table_ld, int32_t up, int32_t down, int32_t K,
                                  int32_t half_len, int32_t m0, int32_t S_out, void* out, int64_t out_ld,
                                  int32_t encoding, int32_t* out_lens, const float* gain, void* stream) {
  const bool ident = up == 1 && down == 1;
  const int tiles = S_out > 0 ? (S_out + kAudioTile - 1) / kAudioTile : 1;
  const size_t smem = as_resample_smem_bytes(up, down, ident ? 1 : K, ident ? 4 : table_ld);
  const int es = encoding == AS_AUDIO_F32 ? 4 : encoding == AS_AUDIO_PCM16 ? 2 : 1;
  const int vec_in = (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (x_ld & 3) == 0;
  const int vec_out = (reinterpret_cast<uintptr_t>(out) & 15) == 0 && ((out_ld * es) & 15) == 0;
  const long long work = (long long)B * tiles;
  const int grid = (int)std::min<long long>(work, (long long)num_sms() * 16);
  const int win = (int)audio_window(up, down, ident ? 1 : K);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned char* o = static_cast<unsigned char*>(out);
  if (ident) {
    ASB_SMEM_OPT_IN(AS_AUDIO_SMEM_MAX, resample_encode_kernel<true, kGain>);
    ASB_CUDA(launch_k(resample_encode_kernel<true, kGain>, dim3(grid), dim3(kAudioThreads), smem, st, x,
                      (long long)x_ld, (int)S_in, in_lens, table, 4, 1, 1, 1, 0, (int)m0, (int)S_out, o,
                      (long long)out_ld, (int)encoding, out_lens, gain, (int)B, tiles, win, vec_in, vec_out));
  } else {
    ASB_SMEM_OPT_IN(AS_AUDIO_SMEM_MAX, resample_encode_kernel<false, kGain>);
    ASB_CUDA(launch_k(resample_encode_kernel<false, kGain>, dim3(grid), dim3(kAudioThreads), smem, st, x,
                      (long long)x_ld, (int)S_in, in_lens, table, (int)table_ld, (int)up, (int)down, (int)K,
                      (int)half_len, (int)m0, (int)S_out, o, (long long)out_ld, (int)encoding, out_lens, gain,
                      (int)B, tiles, win, vec_in, vec_out));
  }
  return AS_OK;
}

extern "C" int as_resample_encode_gain(const float* x, int64_t x_ld, int32_t B, int32_t S_in,
                                       const int32_t* in_lens, const float* table, int32_t table_ld, int32_t up,
                                       int32_t down, int32_t K, int32_t half_len, int32_t m0, int32_t S_out,
                                       void* out, int64_t out_ld, int32_t encoding, int32_t* out_lens,
                                       const float* gain, void* stream) {
  if (B == 0) return AS_OK;
  ASB_REQUIRE(x && out && B > 0 && S_in >= 0 && S_out >= 0 && m0 >= 0 && x_ld >= S_in && out_ld >= S_out,
              AS_ERR_SHAPE, "as_resample_encode: bad argument");
  ASB_REQUIRE(encoding >= AS_AUDIO_F32 && encoding <= AS_AUDIO_ALAW, AS_ERR_DTYPE,
              "as_resample_encode: unknown encoding %d", (int)encoding);
  const bool ident = up == 1 && down == 1;
  ASB_REQUIRE(up > 0 && down > 0 && (ident || (table && K > 0 && table_ld >= K && (table_ld & 3) == 0 &&
                                               half_len >= 0)),
              AS_ERR_SHAPE, "as_resample_encode: bad filter (up %d, down %d, K %d, table_ld %d)", (int)up, (int)down,
              (int)K, (int)table_ld);
  ASB_REQUIRE(ident || (reinterpret_cast<uintptr_t>(table) & 15) == 0, AS_ERR_ALIGN,
              "as_resample_encode: the table must be 16-byte aligned");
  ASB_REQUIRE(!out_lens || (const void*)out_lens != (const void*)in_lens, AS_ERR_SHAPE,
              "as_resample_encode: out_lens must not alias in_lens");
  const int tiles = S_out > 0 ? (S_out + kAudioTile - 1) / kAudioTile : 1;
  // 32-bit indexing: m * down + half_len over every index a thread forms, and n_in * up
  const long long m_end = (long long)m0 + (long long)tiles * kAudioTile + kAudioThreads;
  ASB_REQUIRE(m_end * down + half_len + (long long)kAudioThreads * down < (1LL << 31) &&
                  (long long)S_in * up < (1LL << 31) && (long long)B * tiles < (1LL << 31),
              AS_ERR_SHAPE, "as_resample_encode: too many samples for 32-bit indexing");
  const size_t smem = as_resample_smem_bytes(up, down, ident ? 1 : K, ident ? 4 : table_ld);
  ASB_REQUIRE(smem <= AS_AUDIO_SMEM_MAX, AS_ERR_SHAPE,
              "as_resample_encode: %zu bytes of shared memory for up %d / down %d (at most %d)", smem, (int)up,
              (int)down, AS_AUDIO_SMEM_MAX);
  if (int rc = check_arch()) return rc;
  return gain ? resample_encode_launch<true>(x, x_ld, B, S_in, in_lens, table, table_ld, up, down, K, half_len, m0,
                                             S_out, out, out_ld, encoding, out_lens, gain, stream)
              : resample_encode_launch<false>(x, x_ld, B, S_in, in_lens, table, table_ld, up, down, K, half_len,
                                              m0, S_out, out, out_ld, encoding, out_lens, nullptr, stream);
}

extern "C" int as_resample_encode(const float* x, int64_t x_ld, int32_t B, int32_t S_in, const int32_t* in_lens,
                                  const float* table, int32_t table_ld, int32_t up, int32_t down, int32_t K,
                                  int32_t half_len, int32_t m0, int32_t S_out, void* out, int64_t out_ld,
                                  int32_t encoding, int32_t* out_lens, void* stream) {
  return as_resample_encode_gain(x, x_ld, B, S_in, in_lens, table, table_ld, up, down, K, half_len, m0, S_out, out,
                                 out_ld, encoding, out_lens, nullptr, stream);
}
