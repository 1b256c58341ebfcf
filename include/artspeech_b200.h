/*
 * artspeech_b200 — C ABI of the sm_100a (B200) kernels behind ArtSpeech's batched synthesis
 * forward pass and MAS.  The reference (Zhongxu-Wang/ArtSpeech) is pure Python/PyTorch and has no
 * FFI of its own (SURVEY.md §8b); each entry point below names the reference code whose
 * arithmetic it replaces.  The host side (artspeech_b200/*.py) binds these with ctypes and keeps
 * the reference's nn.Module constructors / state_dict / forward() signatures.
 *
 * Conventions
 *   - plain pointers + sizes only; every pointer is DEVICE memory owned by the caller unless the
 *     comment says "host".  The library never allocates or frees device memory, never
 *     synchronises the stream, and keeps no global mutable state besides the last-error string.
 *   - `stream` is a cudaStream_t passed as void*.
 *   - return 0 (AS_OK) or a negative as_status; as_last_error() gives a thread-local message.
 *   - no CPU fallback and no multi-arch dispatch: everything requires an sm_100 device.
 *   - activations are channels-last: 1-D features [B, T, C], images [B, T, F, C].
 */
#ifndef ARTSPEECH_B200_H_
#define ARTSPEECH_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum as_status {
  AS_OK = 0,
  AS_ERR_SHAPE = -1,
  AS_ERR_DTYPE = -2,
  AS_ERR_ALIGN = -3,
  AS_ERR_ARCH = -4,
  AS_ERR_CUDA = -5,
  AS_ERR_WORKSPACE = -6
} as_status;

/* AS_PCM16: output-only, accepted as y_act_dtype of a single-output-channel 1-D convolution (the vocoder's
 * conv_post + tanh, Vocoder/vocoder.py:113-115): int16 = rint(32767 * y), what soundfile.write(path, wav, 24000)
 * (test.py:119) stores for a float waveform. */
typedef enum as_dtype { AS_F16 = 0, AS_BF16 = 1, AS_F32 = 2, AS_PCM16 = 3 } as_dtype;

typedef enum as_act {
  AS_ACT_NONE = 0,
  AS_ACT_LRELU = 1, /* x > 0 ? x : slope * x */
  AS_ACT_RELU = 2,
  AS_ACT_TANH = 3,
  AS_ACT_SWISH = 4, /* x * sigmoid(x) */
  AS_ACT_ABS = 5
} as_act;

int as_version(void);
/* Persistent kernels launched after this call size their grids for at most n SMs (0: all SMs); returns the previous
 * limit.  The synthesis engine uses it to run the vocoder of one batch and the acoustic model of the next side by
 * side on disjoint SM shares instead of time-slicing the whole GPU (process-wide, host-side setting). */
int as_set_sm_limit(int32_t n);
const char* as_last_error(void);

/* ------------------------------------------------------------------------------------------
 * MAS — replaces S_monotonic_align.py:5-47 (maximum_path1), :50-95 (maximum_path2) and the
 * Triton kernel S_monotonic_align_Triton.py:7-71.
 *   value [B, Tx, Ty] fp32 row-major (not modified); x_len / y_len int32 [B];
 *   path  [B, Tx, Ty] fp32, fully overwritten with 0/1.
 *   tie_mode 0: stay on ties (maximum_path2 / Triton);  1: move to x-1 on ties (maximum_path1).
 *   workspace: as_mas_workspace_bytes() bytes (may be 0 → NULL allowed).
 * ------------------------------------------------------------------------------------------ */
size_t as_mas_workspace_bytes(int32_t B, int32_t Tx, int32_t Ty);
int as_mas_maximum_path(const float* value, const int32_t* x_len, const int32_t* y_len,
                        float* path, int32_t B, int32_t Tx, int32_t Ty, int32_t tie_mode,
                        void* workspace, size_t workspace_bytes, void* stream);

/* MAS plus the two reductions its training callers take of the path (train_second.py:181-187,
 * train_first.py:176-181, models.py:296,323-324), produced by the same back-track:
 *   durations      [B, Tx] int32 = path.sum(-1)                 (d_gt, train_second.py:182)
 *   token_of_frame [B, Ty] int32 = row of the path in column y, -1 for y >= y_len
 * so that `T_en @ s2s_attn_mono` becomes the gather as_expand_tokens below. */
int as_mas_align(const float* value, const int32_t* x_len, const int32_t* y_len, float* path,
                 int32_t* durations, int32_t* token_of_frame, int32_t B, int32_t Tx, int32_t Ty,
                 int32_t tie_mode, void* workspace, size_t workspace_bytes, void* stream);

/* out[b, c, y] = x[b, c, token_of_frame[b, y]] (0 where token_of_frame < 0): bit-identical to
 * `x @ path` for a 0/1 path with one 1 per column (models.py:296,323-324).  x [B, C, Tx] fp32
 * (reference layout, Tx contiguous), out [B, C, Ty] fp32. */
int as_expand_tokens(const float* x, const int32_t* token_of_frame, float* out, int32_t B, int32_t C,
                     int32_t Tx, int32_t Ty, void* stream);

/* ------------------------------------------------------------------------------------------
 * Implicit-GEMM convolution on tcgen05 tensor cores (TMA-fed, TMEM accumulators).
 * Replaces every dense torch Conv1d / ConvTranspose1d (polyphase-packed) / Conv2d / Linear on
 * the path: Vocoder/vocoder.py:35-42,100-116; models.py:189-202 (AdainResBlk1d convs),
 * :497-517 (Decoder), :596-621 (ArtsPredictor); Utils/RelTransformerEnc.py:127-136,261-269,
 * 316-325; Utils/JDC/model.py:102-137; Utils/EMA/conformer (Linear / pointwise convs).
 *
 *   acc[b,to,fo,co] = sum_{j<ntaps} sum_{ci<Cin} x[b, to+dt[j], fo+df[j], ci] * w[j][co][ci]
 *                     (out-of-range input coordinates read as zero: TMA OOB fill)
 *   v     = (acc + bias[co] + res1[row,co] + res2[row,co]) * out_scale,  row = (b*To+to)*Fo+fo
 *   v     = 0 where lens != NULL and to >= lens[b]
 *   y_raw[row*y_raw_ld + co] = v            (if y_raw)
 *   y_act[row*y_act_ld + co] = act(v)       (if y_act; act(0) = 0 for every supported act)
 *
 * x: 16-bit (AS_F16 or AS_BF16), rows of x_ld elements (x_ld % 8 == 0, base 16-byte aligned).
 * w: same dtype, packed [ntaps][CoutP][CinP], CinP % bk == 0 where bk = (Cin >= 64 ? 64 : 32),
 *    CoutP % tile_n == 0 (tile_n from as_conv_tile_n(Cout)); padding must be zero.
 * fp32 accumulation.  Output / residual dtypes: any of as_dtype.
 * ------------------------------------------------------------------------------------------ */
typedef struct as_conv_params {
  const void* x;
  int32_t x_dtype;
  int32_t B, T, F, Cin;
  int64_t x_ld;
  const void* w;
  int32_t ntaps, CinP, CoutP, Cout;
  const int32_t* tap_dt; /* host [ntaps] */
  const int32_t* tap_df; /* host [ntaps] */
  int32_t To, Fo;        /* output spatial size */
  const float* bias;     /* [Cout] fp32 or NULL */
  const void* res1;
  int32_t res1_dtype;
  int64_t res1_ld;
  const void* res2;
  int32_t res2_dtype;
  int64_t res2_ld;
  float out_scale;
  void* y_raw;
  int32_t y_raw_dtype;
  int64_t y_raw_ld;
  void* y_act;
  int32_t y_act_dtype;
  int64_t y_act_ld;
  int32_t act;
  float slope;
  const int32_t* lens; /* device [B] or NULL */
  /* optional fused instance-norm statistics of v (models.py:230-240): stats[b][co][0] += sum,
   * stats[b][co][1] += sum of squares over valid rows (fp32 atomics; caller zeroes it). */
  float* stats;
} as_conv_params;

int32_t as_conv_tile_n(int32_t Cout);
int as_conv_igemm(const as_conv_params* p, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused HiFi-GAN ResBlock1 pair — replaces one iteration of Vocoder/vocoder.py:36-41
 *     xt = c1(leaky_relu(x, slope)); xt = c2(leaky_relu(xt, slope)); x = xt + x
 * (c1: Conv1d(C, C, k, dilation=dil), c2: Conv1d(C, C, k), both 'same'-padded) in one launch; the
 * intermediate stays in shared memory / TMEM.  The residual stream is carried in ACTIVATED form:
 *
 *   x        [B, L, C] 16-bit channels-last holds a = leaky_relu(x_raw, slope); rows >= lens[b] are 0
 *   x_raw    = a < 0 ? a / slope : a
 *   t        = leaky_relu(conv1(a) + b1, slope), zero outside [0, lens[b])      (16-bit operand)
 *   v        = (conv2(t) + b2 + x_raw + res2 + res3) * out_scale ; v = 0 for rows >= lens[b]
 *   y        = out_act == AS_ACT_LRELU ? leaky_relu(v, out_slope) : v           (16-bit, [B, L, C])
 *
 * res2 / res3 (optional, 16-bit, raw) are the finished MRF branches summed by the last pair of a
 * stage (vocoder.py:105-111, with out_scale = 1 / num_kernels).
 * w1 / w2: packed [k][C][C] (tap, cout, cin) K-major like as_conv_igemm; C in {32, 64, 128};
 * k odd <= 15; (k-1)*dil <= 64; fp32 accumulation; 0 < slope <= 1.
 * ------------------------------------------------------------------------------------------ */
typedef struct as_resblock_pair_params {
  const void* x;
  int64_t x_ld;
  int32_t dtype; /* AS_F16 or AS_BF16: x, w1, w2, res2, res3, y */
  int32_t B, L, C, k, dil;
  const void* w1;
  const float* b1; /* [C] fp32 */
  const void* w2;
  const float* b2;
  float slope;
  const void* res2; /* or NULL */
  int64_t res2_ld;
  const void* res3; /* or NULL */
  int64_t res3_ld;
  float out_scale;
  int32_t out_act; /* AS_ACT_NONE or AS_ACT_LRELU */
  float out_slope;
  void* y;
  int64_t y_ld;
  const int32_t* lens; /* device [B] or NULL */
} as_resblock_pair_params;

int as_hifigan_resblock_pair(const as_resblock_pair_params* p, void* stream);


/* ------------------------------------------------------------------------------------------
 * Memory-bound / small kernels.  Unless stated otherwise `x` may be any as_dtype and is addressed
 * as rows of `*_ld` elements (channels-last, outer dims dense); `lens` (int32 [B], may be NULL)
 * gives the valid number of T positions per batch item and rows beyond it are written as zeros.
 * ------------------------------------------------------------------------------------------ */

/* emb(x) * scale (Utils/RelTransformerEnc.py:372-373); out32 fp32 and/or out16 (16-bit) [B,T,C].  Token ids
 * outside [0, n_vocab) read row 0 of the table. */
int as_embed(const int64_t* tokens, const float* table, int32_t n_vocab, int32_t B, int32_t T,
             int32_t C, float scale, const int32_t* lens, float* out32, void* out16,
             int32_t out16_dtype, void* stream);

/* LayerNorm over the channel axis of channels-last rows: custom LN (RelTransformerEnc.py:272-290,
 * eps 1e-4) and nn.LayerNorm (conformer, eps 1e-5).  y = act((x-mean)*rsqrt(var+eps)*gamma+beta).
 * rows = B*T; up to two outputs (e.g. fp32 + 16-bit operand). */
int as_layernorm(const void* x, int32_t x_dtype, int64_t x_ld, int32_t B, int32_t T, int32_t C,
                 const float* gamma, const float* beta, float eps, int32_t act, float slope,
                 const int32_t* lens, void* out_a, int32_t out_a_dtype, int64_t out_a_ld,
                 void* out_b, int32_t out_b_dtype, int64_t out_b_ld, void* stream);

/* Windowed relative-position multi-head self-attention (RelTransformerEnc.py:138-169, window 4,
 * E_k/E_v [2w+1, D] shared by the heads).  qkv fp32 [B,T,3*H*D] (q | k | v), keys >= lens[b] get
 * score -1e4 exactly like masked_fill; out [B,T,H*D]. */
int as_relpos_attention(const float* qkv, int64_t qkv_ld, const float* emb_rel_k,
                        const float* emb_rel_v, int32_t window, int32_t B, int32_t T, int32_t H,
                        int32_t D, const int32_t* lens, void* out, int32_t out_dtype,
                        int64_t out_ld, void* stream);

/* Conformer (Transformer-XL style) attention with the reference's view-based relative shift
 * (Utils/EMA/conformer/conformer/attention.py:72-113): score = ((q+u).k + shift((q+v).p)) /
 * sqrt(H*D); softmax over the valid keys of each item; . V.  q,k,v fp32 [B,T,H*D] rows of ld;
 * pos fp32 [T, H*D] = pos_proj(PE[0:T]); the shift uses each item's own length. */
int as_conformer_attention(const float* q, const float* k, const float* v, int64_t qkv_ld,
                           const float* pos, const float* u_bias, const float* v_bias, int32_t B,
                           int32_t T, int32_t H, int32_t D, const int32_t* lens, void* out,
                           int32_t out_dtype, int64_t out_ld, void* stream);

/* InstanceNorm1d statistics (models.py:230-240): stats[b][c] = {mean, rsqrt(biased var + eps)}
 * over t < lens[b]. */
int as_instnorm_stats(const void* x, int32_t x_dtype, int64_t x_ld, int32_t B, int32_t T,
                      int32_t C, const int32_t* lens, float eps, float* stats, void* stream);

/* AdaIN + LeakyReLU (+ optional depthwise ConvTranspose1d k3 s2 "pool", models.py:172,189-192):
 *   a[b,t,c] = lrelu(((x-mean)*rstd) * (1 + gamma[b,c]) + beta[b,c]),  gamma = gb[b*gb_ld + c],
 *   beta = gb[b*gb_ld + C + c];  up_w == NULL: out[b,t] = a[b,t];
 *   else out[b,2m] = a[m]*w[c][1] + up_b[c], out[b,2m+1] = a[m]*w[c][2] + a[m+1]*w[c][0] + up_b[c]
 *   (a[len] = 0), out has 2T rows and is masked with 2*lens. */
int as_adain_apply(const void* x, int32_t x_dtype, int64_t x_ld, int32_t B, int32_t T, int32_t C,
                   const float* stats, const float* gb, int64_t gb_ld, float slope,
                   const int32_t* lens, const float* up_w, const float* up_b, void* out,
                   int32_t out_dtype, int64_t out_ld, void* stream);

/* as_instnorm_stats + as_adain_apply in one launch: one read + one write of the tensor, exact two-pass
 * statistics from a shared-memory slab.  fp32 input up to 1750 frames: one CTA per (item, 32 channels), the
 * slab arrives by TMA bulk tensor copies; otherwise (16-bit input, up to 6144 frames) a cluster of 4 CTAs
 * splits the frames and exchanges partial sums through distributed shared memory; longer sequences run the
 * two separate passes.  `stats` fp32 [B, C, 2] receives {mean, rstd} (always required: it is the
 * workspace of the long path). */
int as_adain_norm_apply(const void* x, int32_t x_dtype, int64_t x_ld, int32_t B, int32_t T, int32_t C,
                        const float* gb, int64_t gb_ld, float eps, float slope, const int32_t* lens,
                        const float* up_w, const float* up_b, void* out, int32_t out_dtype,
                        int64_t out_ld, float* stats, void* stream);

/* out[b, r, :] = x[b, r / rep, :] for r < rep*lens[b] else 0 (nearest upsample, models.py:261-270) */
int as_repeat_rows(const void* x, int32_t x_dtype, int64_t x_ld, int32_t B, int32_t T, int32_t C,
                   int32_t rep, const int32_t* lens, void* out, int32_t out_dtype, int64_t out_ld,
                   void* stream);

/* Length regulation (models.py:361-368 one-hot matmul == gather) fused with the decoder's x2
 * nearest upsample (models.py:500): frame r of item b copies token j where
 * cum[j] <= r / rep < cum[j+1], cum = exclusive prefix sum of max(dur[b, j], 0) over j < min(lens_t[b], Tt)
 * (durations and token rows beyond that are not read).  x [B,Tt,C]; dur int32 [B,Tt]; out [B,To,C] (rows >=
 * rep*sum zero); out_lens[b] = min(rep*sum, To). */
int as_length_regulate(const void* x, int32_t x_dtype, int64_t x_ld, int32_t B, int32_t Tt,
                       int32_t C, const int32_t* dur, const int32_t* lens_t, int32_t rep,
                       int32_t To, void* out, int32_t out_dtype, int64_t out_ld,
                       int32_t* out_lens, void* stream);

/* Integer durations on the device (models.py:361: pred_dur = torch.round(duration).clamp(min=1), round-half-to-even):
 * dur[b,t] = max(1, rint(pred[b,t])) for t < lens_t[b], 0 beyond; sum[b] = sum_t dur[b,t] (half-rate frames of
 * utterance b; may be NULL).  Keeps the predictor -> length-regulator hand-off on the device, so durations are an
 * INPUT of the captured CUDA graph and the host reads back B integers instead of doing 2*Tt+1 syncs (models.py:362-366).
 * pred fp32 [B,Tt] with row stride pred_ld; dur int32 [B,Tt] contiguous; sum int32 [B]. */
int as_round_durations(const float* pred, int64_t pred_ld, int32_t B, int32_t Tt, const int32_t* lens_t,
                       int32_t* dur, int32_t* sum, void* stream);

/* as_round_durations with a speaking-rate scale (prosody duration_scale): dur[b,t] = max(1, rint(pred[b,t] * s)),
 * s = scale[b * scale_ld + t] fp32, or scale[b] (one value per utterance) when scale_ld == 0.  A scale of 1 gives
 * the bits of as_round_durations. */
int as_round_durations_scaled(const float* pred, int64_t pred_ld, int32_t B, int32_t Tt, const int32_t* lens_t,
                              const float* scale, int64_t scale_ld, int32_t* dur, int32_t* sum, void* stream);

/* Per-utterance prosody edits of the arts predictor's tracks (models.py:369), in place, frames t < lens[b] only:
 *   F0  fp32 [B,Tm,1] (z-normalised, hz = f0 * pitch_std + pitch_mean): on voiced frames (hz >= 50 Hz)
 *       hz' = exp(mu + range * (ln hz - mu) + shift * ln2 / 12), f0' = f0 + (hz' - hz) / pitch_std, mu = mean of
 *       ln hz over the utterance's voiced frames (no voiced frame: F0 unchanged);
 *   N   fp32 [B,Tm,1] (log-norm energy): n' = n + dB * ln10 / 10 / energy_std;
 *   EMA fp32 [B,Tm,10]: e' = m_c + scale_c * (e - m_c) + offset_c, m_c = channel mean over the valid frames.
 * ctrl fp32 [B, AS_PROSODY_CTRL] = {shift, range, dB, 0, scale[10], offset[10]}; *_ld are row strides (elements
 * per frame) of dense [B,Tm,*] buffers.  A track whose controls are identity is not written.  One CTA per
 * utterance with a fixed reduction order: an utterance's result does not depend on B, Tm or its batch-mates. */
#define AS_PROSODY_CTRL 24
int as_prosody_apply(float* f0, int64_t f0_ld, float* n, int64_t n_ld, float* ema, int64_t ema_ld, int32_t B,
                     int32_t Tm, const int32_t* lens, const float* ctrl, double pitch_mean, double pitch_std,
                     double energy_std, void* stream);

/* Output audio formats (artspeech_b200/audio.py): resampling of fp32 waveforms by up/down and encoding, one launch.
 *   y[b,m] = sum_{j=0..K-1} table[p][j] * x[b, i0 - j],  n = m*down + half_len, i0 = n / up, p = n % up,
 * with x zero outside [0, n_in_b), n_in_b = min(in_lens[b], S_in) (S_in when in_lens is NULL): one fp32 fma chain over
 * j = 0..K-1 in that order, so a value depends only on its row's samples and m.  table fp32 [up][table_ld], 16-byte
 * aligned, table_ld >= K and a multiple of 4.  up == down == 1 is the identity y = x (table, K, half_len ignored).
 * x [B, >= S_in] with row stride x_ld; out [B, S_out] with row stride out_ld (elements).  Output r of row b is sample
 * m = m0 + r: y encoded for m < n_out_b = ceil(n_in_b * up / down), the encoding's silence code beyond.  Encodings:
 *   AS_AUDIO_F32 float y;  AS_AUDIO_PCM16 int16 clamp(rint(32767 y), -32768, 32767) (the AS_PCM16 conv epilogue);
 *   AS_AUDIO_MULAW / AS_AUDIO_ALAW uint8 ITU-T G.711 code of that int16 (audioop.lin2ulaw / lin2alaw, width 2).
 * Silence is 0, 0, 0xFF, 0xD5.  out_lens int32 [B] (may be NULL, must not alias in_lens) receives n_out_b.  Lengths
 * are read and written on the device: no host synchronisation.  Filters whose shared memory
 * (as_resample_smem_bytes) exceeds AS_AUDIO_SMEM_MAX are refused with AS_ERR_SHAPE. */
typedef enum as_audio_encoding { AS_AUDIO_F32 = 0, AS_AUDIO_PCM16 = 1, AS_AUDIO_MULAW = 2, AS_AUDIO_ALAW = 3 } as_audio_encoding;
#define AS_AUDIO_TILE 1024
#define AS_AUDIO_SMEM_MAX (96 * 1024)
size_t as_resample_smem_bytes(int32_t up, int32_t down, int32_t K, int32_t table_ld);
int as_resample_encode(const float* x, int64_t x_ld, int32_t B, int32_t S_in, const int32_t* in_lens,
                       const float* table, int32_t table_ld, int32_t up, int32_t down, int32_t K, int32_t half_len,
                       int32_t m0, int32_t S_out, void* out, int64_t out_ld, int32_t encoding, int32_t* out_lens,
                       void* stream);
/* As as_resample_encode, with a per-utterance gain: y[b,m] above is multiplied by gain[b] (fp32 [B], device) in one
 * fp32 multiply before it is encoded (on the identity path y = x[b,m] * gain[b]); silence codes are unchanged.
 * gain == NULL is exactly as_resample_encode. */
int as_resample_encode_gain(const float* x, int64_t x_ld, int32_t B, int32_t S_in, const int32_t* in_lens,
                            const float* table, int32_t table_ld, int32_t up, int32_t down, int32_t K,
                            int32_t half_len, int32_t m0, int32_t S_out, void* out, int64_t out_ld, int32_t encoding,
                            int32_t* out_lens, const float* gain, void* stream);

/* Loudness meter (artspeech_b200/audio.py, ITU-R BS.1770 integrated loudness and 4x true peak) and normalisation
 * gain, per utterance of n_b = min(lens[b], S) samples (S when lens is NULL) of x [B, >= S] (row stride x_ld) at
 * fs Hz (a multiple of 10 in [8000, 192000]).  Samples at or beyond n_b are never read.
 *   K-weighting: two cascaded biquads (transposed direct form II, zero initial state, fp64), kw = {b0, b1, b2, a1,
 *   a2} of the shelf stage then of the high-pass stage (host array of 10 doubles, audio.k_weighting(fs)).
 *   Segments of g = fs/10 samples; E_s = sum of y^2 over segment s (fp64).  Blocks j = 0 .. n_b/g - 4:
 *   z_j = (((E_j + E_{j+1}) + E_{j+2}) + E_{j+3}) / (4 g); when n_b < 4 g a single block z = (sum_s E_s) / n_b.
 *   L_j = -0.691 + 10 log10 z_j; J_a = {L_j > -70}; G = -0.691 + 10 log10(mean_{J_a} z) - 10;
 *   J_g = {j in J_a : L_j > G}; loudness = -0.691 + 10 log10(mean_{J_g} z), -inf when J_a is empty or n_b = 0.
 *   True peak: TP = max(|x_i|, |y4_m|), y4[4q + r] = sum_{j=0..20} tp_table[r][j] * x[q + 10 - j] (one fp32 fma
 *   chain, x zero outside [0, n_b)), q = 0 .. n_b - 1; tp_table is the [4][AS_LOUDNESS_TP_LD] fp32 polyphase table
 *   of the 4x resampler (AudioFormat's design with up 4, down 1: 81 taps), a host array.  true_peak = 20 log10 TP
 *   (-inf for 0).
 *   gain_db = 0 when loudness is -inf, else min(target - loudness, ceiling - true_peak); gain = fp32(10^(gain_db/20)).
 * Outputs (device, [B]): loudness_out, true_peak_out, gain_db_out fp64 (gain_db_out may be NULL), gain_out fp32 (may
 * be NULL).  Three launches; every sum is taken in an order fixed by the utterance's own sample indices, so the results
 * do not depend on B, S, x_ld or the other utterances.  Lengths are read on the device: no host synchronisation.
 * workspace: device, at least as_loudness_workspace_bytes(B, S, fs) bytes, 256-byte aligned.  S is limited to
 * AS_LOUDNESS_MAX_TILES * 8 segments (54 minutes at 24 kHz). */
#define AS_LOUDNESS_TP_LD 24
#define AS_LOUDNESS_MAX_TILES 4096
#define AS_LOUDNESS_LAUNCHES 3
size_t as_loudness_workspace_bytes(int32_t B, int64_t S, int32_t fs);
int as_loudness_measure(const float* x, int64_t x_ld, int32_t B, int64_t S, const int32_t* lens, int32_t fs,
                        const double* kw, const float* tp_table, double target, double ceiling, void* workspace,
                        size_t workspace_bytes, double* loudness_out, double* true_peak_out, double* gain_db_out,
                        float* gain_out, void* stream);

/* Synthesis watermark (artspeech_b200/audio.py states the format).  Pattern bins k = AS_WM_K_LO ..
 * AS_WM_K_LO + AS_WM_BINS - 1 of an AS_WM_PERIOD-point period at 8 kHz (300 - 3400 Hz); AS_WM_SYMBOLS lags per symbol.
 *
 * as_watermark_embed: y[b,t] = x[b,t] + (alpha e(t)) c[t mod AS_WM_PERIOD_24K] (one fp32 fma) for t < n_b =
 * min(lens[b], S) (S when lens is NULL), y[b,t] = 0 for n_b <= t < S.  e(t): RMS of the 240-sample frames (zeros at
 * and beyond n_b), linear between frame centres 240 f + 119.5, held beyond the first and last.  pattern fp32
 * [AS_WM_PERIOD_24K], 16-byte aligned (audio.Watermark.device_pattern).  x [B, >= S] row stride x_ld; out [B, S]
 * row stride out_ld, not aliasing x.  Samples at or beyond n_b are never read; lengths are read on the device.  Each
 * frame's sum has one order, so the result does not depend on B, S, the strides or the batch-mates.  One launch. */
#define AS_WM_PERIOD 4096
#define AS_WM_PERIOD_24K 12288
#define AS_WM_K_LO 154
#define AS_WM_BINS 1587
#define AS_WM_BINS_LD 1588
#define AS_WM_SYMBOLS 256
#define AS_WM_DETECT_LAUNCHES 2
int as_watermark_embed(const float* x, int64_t x_ld, int32_t B, int32_t S, const int32_t* lens, const float* pattern,
                       float alpha, float* out, int64_t out_ld, void* stream);

/* Encoded samples to fp32, elementwise: AS_AUDIO_PCM16 int16 v -> v / 32768; AS_AUDIO_MULAW / AS_AUDIO_ALAW uint8 ->
 * audioop.ulaw2lin / alaw2lin (width 2) / 32768.  in [B, >= S] row stride in_ld (elements); out fp32 [B, S] row
 * stride out_ld.  One launch: as_audio_to_mono with C = 1 and no lengths. */
int as_audio_decode(const void* in, int64_t in_ld, int32_t B, int32_t S, int32_t encoding, float* out, int64_t out_ld,
                    void* stream);

/* Encoded samples with C interleaved channels (1 <= C <= AS_AUDIO_MAX_CHANNELS) to mono fp32 (voice enrollment,
 * artspeech_b200/frontend.py):  out[b,t] = (d(x[b, t C]) + ... + d(x[b, t C + C - 1])) / C, an fp32 sum in channel
 * order then one fp32 divide (numpy's float32 mean over the channels), for t < n_b = min(lens[b], S) (S when lens is
 * NULL); out[b,t] = 0 for n_b <= t < S.  d decodes as as_audio_decode (AS_AUDIO_F32: the value itself).  in [B,
 * >= S C] elements of the encoding's type with row stride in_ld (elements); out fp32 [B, S] row stride out_ld, not
 * aliasing in.  Samples at or beyond n_b are never read; lengths are read on the device.  One launch. */
#define AS_AUDIO_MAX_CHANNELS 8
int as_audio_to_mono(const void* in, int64_t in_ld, int32_t B, int32_t S, int32_t C, int32_t encoding,
                     const int32_t* lens, float* out, int64_t out_ld, void* stream);

/* Leading / trailing silence of 24 kHz fp32 utterances (librosa 0.10 effects.trim with frame 2048, hop 512),
 * y [B, >= S] row stride y_ld, n_b = min(lens[b], S) (S when lens is NULL):
 *   q_j = sum of y^2 over block j = [512 j, 512 j + 512) in fp64, zeros at and beyond n_b;
 *   p_f = (((q_{f-2} + q_{f-1}) + q_f) + q_{f+1}) / 2048 for frames f < F = 1 + n_b / 512 (blocks outside
 *   [0, ceil(n_b / 512)) count as 0): the squared RMS of librosa's centred, zero-padded frames;
 *   P = max_f p_f; frame f is non-silent iff 10 log10(max(1e-10, p_f)) - 10 log10(max(1e-10, P)) > -top_db;
 *   bounds[b] = (512 first, min(n_b, 512 (last + 1))) over the non-silent frames; (0, 0) when n_b = 0.
 * bounds int32 [B][2] (device).  Two launches (block sums, then one CTA per utterance), no atomics, no host
 * synchronisation; every sum's shape follows from n_b alone, so the bounds do not depend on B, S, y_ld or the
 * batch-mates.  Samples at or beyond n_b are never read.  workspace: device, at least
 * as_trim_workspace_bytes(B, S) bytes, 8-byte aligned.  top_db finite and positive. */
#define AS_TRIM_LAUNCHES 2
size_t as_trim_workspace_bytes(int32_t B, int32_t S);
int as_trim_bounds(const float* y, int64_t y_ld, int32_t B, int32_t S, const int32_t* lens, double top_db,
                   void* workspace, size_t workspace_bytes, int32_t* bounds, void* stream);

/* Stationary-noise suppression of 24 kHz fp32 rows (voice enrollment, artspeech_b200/frontend.py step 2b), y [B, >= S]
 * row stride y_ld, n_b = min(lens[b], S) (S when lens is NULL), F_b = 1 + n_b / 128 frames:
 *   X[f, k]: 257-bin real FFT of the frame w[i] y[128 f - 256 + i], i < 512 (zeros outside [0, n_b)), fp32;
 *   P = re^2 + im^2 as two rounded fp32 products and one rounded add;
 *   lambda[k] = max(1e-20, P_(r)[k] / c) in fp64, P_(r)[k] the (F_b / 10)-th smallest (0-based) of P[0 .. F_b), k];
 *   in fp64 (__dmul_rn, __dadd_rn, __ddiv_rn, in this order): gamma = P / lambda, m = max(gamma - 1, 0),
 *   xi_0 = m_0, xi_f = alpha A_{f-1} + one_minus_alpha m_f, W = xi / (1 + xi), A = (W W) gamma, and
 *   G = max(W, g_min) rounded to fp32;
 *   out[t] = sum_f w[j] irfft(G_f X_f)[j] / sum_f w[j]^2, j = t - 128 f + 256, over f < F_b covering t, ascending;
 *   out[t] = 0 for n_b <= t < S.
 * window fp32 [512] (periodic Hann), twiddle / itwiddle fp32 [256][2] = (cos, -sin) / (cos, sin)(2 pi m / 512), device.
 * reduction_db in [0, 60]; g_min = 10^(-reduction_db / 20), c = -log1p(-0.1), alpha = 0.98 and one_minus_alpha =
 * 1 - alpha, computed on the host in fp64.  out [B, S] row stride out_ld, not aliasing y.
 * workspace: device, 256-byte aligned, at least as_denoise_workspace_bytes(B, S) bytes = X (complex fp32
 * [B][1 + S / 128][AS_DENOISE_BINS], 16 bytes per input sample) at offset 0, then G (fp32, same shape), then lambda
 * (fp64 [B][AS_DENOISE_BINS]), each starting on a 256-byte boundary.  AS_DENOISE_LAUNCHES launches (STFT; noise
 * profile and gain; inverse FFT and overlap-add), no floating-point atomics, no host synchronisation; every value of a
 * row follows from its own samples, so the output does not depend on B, S, the strides or the batch-mates.  Samples
 * at or beyond n_b are never read. */
#define AS_DENOISE_BINS 257
#define AS_DENOISE_LAUNCHES 3
size_t as_denoise_workspace_bytes(int32_t B, int32_t S);
int as_denoise(const float* y, int64_t y_ld, int32_t B, int32_t S, const int32_t* lens, double reduction_db,
               const float* window, const float* twiddle, const float* itwiddle, double c, double g_min, double alpha,
               double one_minus_alpha, void* workspace, size_t workspace_bytes, float* out, int64_t out_ld,
               void* stream);

/* Watermark detector on 8 kHz fp32 utterances x [B, >= S] (row stride x_ld), n_b = min(lens[b], S) (S when NULL):
 *   z[t] = x[t] / e(t) where e(t) >= 1e-4, else 0 (e as in the embedder with 80-sample frames); Z_p = DFT of
 *   z[4096 p .. 4096 p + 4095] (zeros beyond n_b) at the pattern bins, p < ceil(n_b / 4096); A = sum_p Z_p,
 *   S = sum_p |Z_p|^2 (fp32, p in order), G = A / S (0 where S = 0);
 *   r_i[tau] = sum_k Re(G(k) E_i(k) e^{j 2 pi k tau / 4096}), E_i = spectra[i] = e^{-j phi_i(k)};
 *   lag = argmax |r_0| (lowest on ties), score = |r_0[lag]| / sqrt(mean r_0^2) (0 when r_0 is 0), detected =
 *   score >= threshold, message = s_1 | s_2 << 8 with s_i = argmax_{s < 256} |r_i[(lag + 16 s) mod 4096]|.
 * spectra fp32 [3][AS_WM_BINS_LD][2] (complex, device); twiddles fp32 [2048][2] = (cos, -sin)(2 pi m / 4096) (device).
 * Outputs (device, [B]): score fp32, lag / message int32, detected uint8.  workspace: device, at least
 * as_watermark_workspace_bytes(B, S) bytes.  AS_WM_DETECT_LAUNCHES launches, no atomics, no host synchronisation;
 * every sum's shape follows from n_b alone, so the results do not depend on B, S, x_ld or the batch-mates. */
size_t as_watermark_workspace_bytes(int32_t B, int32_t S);
int as_watermark_detect(const float* x, int64_t x_ld, int32_t B, int32_t S, const int32_t* lens, const float* spectra,
                        const float* twiddles, float threshold, void* workspace, size_t workspace_bytes, float* score,
                        int32_t* lag, int32_t* message, uint8_t* detected, void* stream);

/* Direct convolution for tiny input-channel counts (Cin <= 16) on CUDA cores: first layers of the
 * 2-D stacks (1 -> 64, 3x3), F0/N/EMA 1x1 convs of the decoder (models.py:480-482, 502-504).
 * x [B,T,F,Cin]; w fp32 [ntaps][Cout][Cin]; taps host arrays; stride 1; zero padding; outputs as
 * as_conv_igemm (raw / activated). */
int as_conv_small(const void* x, int32_t x_dtype, int64_t x_ld, int32_t B, int32_t T, int32_t F,
                  int32_t Cin, const float* w, const float* bias, int32_t ntaps,
                  const int32_t* tap_dt, const int32_t* tap_df, int32_t Cout, const int32_t* lens,
                  void* y_raw, int32_t y_raw_dtype, int64_t y_raw_ld, void* y_act,
                  int32_t y_act_dtype, int64_t y_act_ld, int32_t act, float slope, void* stream);

/* Depthwise convolution over (T,F) with stride (models.py:27-31,116; conformer
 * convolution.py:136-149 with glu != 0: the input has 2C channels and value = x[c]*sigmoid(x[C+c])).
 * w fp32 [kt*kf][C] (BatchNorm already folded), bias [C] or NULL; out = act(conv). */
int as_dwconv(const void* x, int32_t x_dtype, int64_t x_ld, int32_t B, int32_t T, int32_t F,
              int32_t C, int32_t glu, const float* w, const float* bias, int32_t kt, int32_t kf,
              int32_t st, int32_t sf, int32_t pt, int32_t pf, int32_t To, int32_t Fo,
              const int32_t* lens_in, const int32_t* lens_out, int32_t act, float slope,
              void* out, int32_t out_dtype, int64_t out_ld, void* stream);

/* Average pooling pt x pf (stride = window) with the reference's replicate padding of the last T
 * position when T is odd (models.py:43-57,127-130); To = ceil(T/pt), Fo = F/pf. */
int as_avgpool(const void* x, int32_t x_dtype, int64_t x_ld, int32_t B, int32_t T, int32_t F,
               int32_t C, int32_t pt, int32_t pf, void* out, int32_t out_dtype, int64_t out_ld,
               void* stream);

/* y = maxpool_F(lrelu(x*scale[c] + shift[c]), pf)  (Utils/JDC/model.py:163-167,34-38);
 * Fo = F / pf (floor). */
int as_affine_act_maxpool(const void* x, int32_t x_dtype, int64_t x_ld, int32_t B, int32_t T,
                          int32_t F, int32_t C, const float* scale, const float* shift,
                          float slope, int32_t pf, void* out, int32_t out_dtype, int64_t out_ld,
                          void* stream);

/* out[b,c] = mean over (t in {0, ts, 2ts, ..} < T, f < F) of lrelu(x[b,t,f,c])
 * (LeakyReLU + AdaptiveAvgPool, models.py:390-393; ts = 2 evaluates a stride-2 conv) */
int as_global_avgpool(const void* x, int32_t x_dtype, int64_t x_ld, int32_t B, int32_t T,
                      int32_t F, int32_t C, int32_t t_stride, float slope, void* out,
                      int32_t out_dtype, int64_t out_ld, void* stream);

/* Bidirectional single-layer LSTM recurrence with packed-sequence semantics (PyTorch gate order
 * i,f,g,o; models.py:555-564,606-618; Utils/JDC/model.py:128).  xproj fp32 [B,T,2*4H] =
 * W_ih x + b_ih + b_hh for (forward | reverse); whh_t fp32 [2][H][4H] = weight_hh transposed
 * (k-major, so the 4H gate threads read consecutive floats); out [B,T,2H] with (forward |
 * reverse) halves, zeros beyond lens[b]; the reverse direction starts at lens[b]-1. */
int as_bilstm(const float* xproj, int64_t xproj_ld, const float* whh_t, int32_t B, int32_t T,
              int32_t H, const int32_t* lens, void* out, int32_t out_dtype, int64_t out_ld,
              void* stream);

/* One LSTM step from zero state per row (the reference's mis-oriented EMA LSTM at batch 1,
 * Utils/EMA/EMA_Predictor.py:44,80): c = sig(i)*tanh(g), h = sig(o)*tanh(c) for both directions.
 * xproj fp32 [rows, 2*4H] -> out [rows, 2H]. */
int as_lstm_onestep(const float* xproj, int64_t xproj_ld, int64_t rows, int32_t H, void* out,
                    int32_t out_dtype, int64_t out_ld, void* stream);

/* log-norm energy (models.py:655-660): out[b,t] = log(||exp(mel[b,:,t]*4 - 4)||_2), mel fp32
 * channels-first [B,n_mels,T] (the reference's own input layout). */
int as_log_norm(const float* mel, int32_t B, int32_t n_mels, int32_t T, float* out, void* stream);

/* Layout/dtype change between the reference's channels-first tensors and channels-last
 * activations: dst[b,t,c] = src[b,c,t] (to_channels_last != 0, rows >= lens zeroed) or the
 * inverse.  Optional per-channel affine y = (x - sub[c]) * mul[c] on the way. */
int as_transpose_cast(const void* src, int32_t src_dtype, void* dst, int32_t dst_dtype, int32_t B,
                      int32_t C, int32_t T, int64_t cl_ld, int32_t to_channels_last,
                      const float* sub, const float* mul, const int32_t* lens, void* stream);

/* ------------------------------------------------------------------------------------------
 * Log-mel front-end of the reference recordings — replaces test.py:40-47 / meldataset.py:42-49:
 * torchaudio MelSpectrogram(n_mels, n_fft 2048, win_length, hop) (centre = True, reflect padding, periodic
 * Hann window zero-padded to n_fft, power 2, HTK filterbank) then (log(log_eps + mel) - mean) / std.
 *   wave   fp32 [B, N] rows of wave_ld samples; lens int32 [B] samples per recording or NULL (each must
 *          exceed n_fft / 2); window fp32 [n_fft]; twiddle fp32 [n_fft/2][2] = (cos, -sin)(2 pi k / n_fft);
 *   fb     fp32 [n_fft/2 + 1, n_mels]; fb_range int32 [n_mels][2] = first bin and bin count of each filter;
 *   out    fp32 [B, n_mels, n_frames] (channels-first like the reference's mel), n_frames = 1 + N / hop;
 *          frames beyond 1 + lens[b] / hop are written as zeros.
 * ------------------------------------------------------------------------------------------ */
int as_log_mel(const float* wave, int64_t wave_ld, const int32_t* lens, int32_t B, int32_t N,
               const float* window, const float* twiddle, const float* fb, const int32_t* fb_range,
               int32_t n_fft, int32_t hop, int32_t n_mels, float log_eps, float mean, float std,
               float* out, int32_t n_frames, void* stream);
/* as_log_mel of a span of each row: recording b is the lens[b] samples wave[b * wave_ld + starts[b] ...] (both int32
 * [B], device, required), reflect-padded at the span's own ends; starts[b] + lens[b] <= N.  The arithmetic is
 * as_log_mel's: a span gives the bits as_log_mel gives for the same samples copied to the start of a row. */
int as_log_mel_span(const float* wave, int64_t wave_ld, const int32_t* starts, const int32_t* lens, int32_t B,
                    int32_t N, const float* window, const float* twiddle, const float* fb, const int32_t* fb_range,
                    int32_t n_fft, int32_t hop, int32_t n_mels, float log_eps, float mean, float std, float* out,
                    int32_t n_frames, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ARTSPEECH_B200_H_ */
