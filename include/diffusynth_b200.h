/* diffusynth_b200 -- C ABI of the B200 (sm_100a) implementation of DiffuSynth's
 * text-to-timbre sampling path.
 *
 * The reference (WxuanYuan/diffusynth) is pure Python/PyTorch and has no FFI; the Python
 * classes in diffusynth_b200/ keep the reference's surfaces (DiffSynthSampler,
 * ConditionedUnet.forward, VectorQuantizerEMA.forward, Decoder/Encoder.forward,
 * decode_stft/istft ...) and route them to these entry points through ctypes
 * (INTEGRATION.md shows the binding).  Each entry cites the reference code it replaces
 * (paths relative to the reference root).
 *
 * Conventions: plain pointers and sizes only; every pointer named d_* is DEVICE memory owned
 * by the caller; `stream` is a cudaStream_t passed as void*; all calls are asynchronous on
 * that stream and capturable into a CUDA graph; return value 0 = ok, <0 = error
 * (-1 invalid argument/shape, -2 CUDA error, -3 NCCL error, -4 unsupported);
 * ds_last_error() returns the message of the calling thread's last failure.
 * Activation tensors are 16-bit ("act16", see ds_operand_dtype) channels-last ("NHWC") unless a name says f32/nchw.
 */
#ifndef DIFFUSYNTH_B200_H
#define DIFFUSYNTH_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* ds_last_error(void);
int ds_version(void);
/* 16-bit storage / tensor-core operand format the library was built with: 1 = IEEE fp16 (default),
   0 = bf16 (-DDS_OPERANDS_BF16).  "act16" below means this type. */
int ds_operand_dtype(void);
/* Device sanity: returns 0 when device `dev` is compute capability 10.x. */
int ds_check_device(int dev);

/* ----------------------------------------------------------------------------------------
 * Implicit-GEMM convolution on tcgen05 tensor cores (TMEM accumulators, TMA-fed).
 * Replaces every dense nn.Conv2d / nn.ConvTranspose2d on the path:
 *   ConvNextBlock.net[1], net[4], res_conv      model/diffusion_components.py:122,125,128
 *   Downsample / Upsample (4x4 stride 2)        model/diffusion_components.py:32-39
 *   LinearCrossAttentionAdd.to_qkv / to_out     model/diffusion_components.py:263-264
 *   final_conv[1]                               model/diffusion.py:174
 *   VQGAN Encoder/Decoder convs                 model/VQGAN.py:149-174,191,216,254-259
 * and, folded into its epilogue, the GroupNorm(1,C) that precedes the conv
 * (diffusion_components.py:121,124,148), bias, GELU (:123), the residual add (:139),
 * and the (sum, sum-of-squares) partials the next GroupNorm needs.
 *
 * GEMM view: M = pixels of an (Hb x Wb = 128)-pixel spatial tile of one sample, N = output
 * channels (tile BN), K = taps x input channels.  Up to two channel-concatenated sources
 * (pad_and_concat, diffusion_components.py:236-249) are read in place.
 * -------------------------------------------------------------------------------------- */
#define DS_MAX_TAPS 16
#define DS_MAX_GROUPS 4

typedef struct ds_conv_tap {
  int8_t dy, dx;   /* pixel offset of this tap inside its view */
  int8_t view;     /* which (parity) view of the source the tap reads: 0..3 */
  int8_t pad_;
} ds_conv_tap;

typedef struct ds_conv_gemm_args {
  /* sources: act16 NHWC [N, Hs, Ws, C]; source 1 optional (C1 = 0), concatenated after source 0 along C.
     A "view" v of a source is a strided pixel window, given in PIXEL units so that it applies to both
     sources: pixel(n, y, x) = view_off[v] + n*view_sn + y*view_sh + x*view_sw, extent Hv x Wv; the
     element offset in a source with C channels is pixel*C + c.  Stride-1 convs use the identity view,
     the 4x4 stride-2 conv the four (row parity, column parity) views of its input. */
  const void* d_src0;
  const void* d_src1;
  int32_t C0, C1;
  int32_t N;                /* samples */
  int32_t src_batch_mod;    /* if >0, sample n reads sample n % src_batch_mod of SOURCE 0 (and of d_stats_in); source 1 is indexed by n.
                               Classifier-free guidance: tensors computed once for both halves of the doubled batch. */
  int32_t Hv, Wv;           /* extent of every view (pixels) */
  int64_t view_sn, view_sh, view_sw;   /* pixel strides of a view per unit of (n, y, x) */
  int64_t view_off[4];      /* pixel offset of each view's origin */
  int32_t num_views;
  int32_t view_wv[4], view_hv[4];      /* per-view extents where they differ (odd input sizes of the stride-2 conv: the even-parity
                                          view holds one more column/row than the odd one); 0 = Wv / Hv */
  /* GEMM pixel grid (per sample) and tile shape */
  int32_t H, W;             /* output-tile grid extent */
  int32_t Hb, Wb;           /* Hb*Wb == 128 */
  /* weights: act16 [Z, Cout_pad, K] K-major, K = ntaps*(C0+C1) ordered tap-major then channel
     (source 0 channels first).  Z = groups, or N when per_sample_weights. */
  const void* d_weight;
  int32_t Cout_pad;         /* multiple of BN */
  int32_t Cout;             /* real output channels (<= Cout_pad) */
  int32_t BN;               /* N tile: multiple of 16, <= 256 */
  int32_t BK;               /* 32 or 64; must divide C0 and C1 */
  int32_t ntaps, groups;
  int32_t per_sample_weights;
  ds_conv_tap taps[DS_MAX_GROUPS][DS_MAX_TAPS];
  /* epilogue:  v = rstd*acc - rstd*mean*e1[cls][o] + e2[cls][o] + sbias[n][o];  act;  + residual */
  const void* d_stats_in;   /* statistics buffer of the (GroupNorm(1,C)-normalised) source, or NULL: float2
                               [N][2 + stats_in_slots], entry [n][0] = (mean, rstd) published by the producer */
  int32_t stats_in_slots;
  float stats_out_inv_count; /* 1 / (elements per sample of THIS call's output), used when d_stats_out is set */
  float eps;                /* GroupNorm eps used when publishing (mean, rstd) of the output */
  const float* d_e1;        /* [ncls][Cout_pad] or NULL */
  const float* d_e2;        /* [ncls][Cout_pad]: bias (+ folded GroupNorm beta term) */
  int32_t ncls;             /* 1, or 9 = (top/mid/bottom) x (left/mid/right) border classes of a 3x3 */
  const float* d_sbias;     /* per-sample bias [N][sbias_stride] or NULL */
  int32_t sbias_stride;
  int32_t act;              /* 0 none, 1 GELU(erf) */
  const void* d_residual;   /* act16, pixel strides below, or NULL */
  int64_t res_sn, res_sh, res_sw;      /* in elements */
  void* d_out;              /* act16 out, or NULL */
  int64_t out_sn, out_sh, out_sw;      /* in elements */
  int64_t out_goff[DS_MAX_GROUPS];     /* element offset per group (sub-pixel phase of ConvTranspose) */
  float* d_out_f32_nchw;    /* optional fp32 [N, Cout, H, W] output (final conv) */
  void* d_stats_out;        /* statistics buffer of the output, float2 [N][2 + ds_conv_gemm_stats_slots()], zero-initialised
                               once by the caller (entry [n][1] is an arrival counter that resets itself), or NULL:
                               [n][2+i] = (sum, sumsq) partial of tile-warp i, [n][0] = (mean, rstd) written by the last arriver */
} ds_conv_gemm_args;

int ds_conv_gemm(const ds_conv_gemm_args* args, void* stream);
/* number of (sum, sumsq) partial slots per sample the call writes to d_stats_out (buffer holds 2 more entries) */
int ds_conv_gemm_stats_slots(const ds_conv_gemm_args* args);
/* Same contract on plain CUDA cores; exists only to cross-check the tcgen05 kernel in tests. */
int ds_conv_gemm_reference(const ds_conv_gemm_args* args, void* stream);

/* The launch ds_conv_gemm would make for these arguments (host only, launches nothing; ds_conv_gemm launches from the same
   computation).  A work item is one 128-pixel M-tile x BN-channel N-tile (cg = 1) or a pair of M-tiles on a two-CTA cluster
   (cg = 2); the grid's CTAs (CTA pairs) walk the items with a stride of grid (grid / 2). */
typedef struct ds_conv_gemm_plan_info {
  int32_t BK, BN;           /* K block and N tile (as given in the arguments) */
  int32_t cg;               /* CTAs per MMA: 1, or 2 (cta_group::2 pairs) */
  int32_t pair_flat;        /* cg = 2 pairs run over the flattened (sample, M-tile) index (odd M-tiles per sample) */
  int32_t epi;              /* epilogue variant: 0 generic (fp32 / ragged output), 1 fold, 2 fold + GELU, 3 + residual, 4 bias only */
  int32_t two_per_sm;       /* two resident CTAs per SM (plain 1x1 convolutions) */
  int32_t nacc;             /* tensor-memory accumulators per CTA: 2 (double-buffered) or 1 */
  int32_t sps, stages;      /* K-blocks per pipeline stage, pipeline stages */
  int32_t num_tiles;        /* work items */
  int32_t grid;             /* CTAs launched */
} ds_conv_gemm_plan_info;
int ds_conv_gemm_plan(const ds_conv_gemm_args* args, ds_conv_gemm_plan_info* info);

/* ----------------------------------------------------------------------------------------
 * Sampler step kernels (model/DiffSynthSampler.py).
 * -------------------------------------------------------------------------------------- */
/* Fused CFG combine + DDIM/DDPM update, one coalesced fp32 pass (K11).  Replaces :320-343.
   d_coef (device) = {sqrt(1-a_t), sqrt(a_t), sqrt(a_prev), sqrt(1-a_prev-sigma^2), sigma, cfg_scale}.
   d_eps_u NULL <=> CFG == 1.0 (:311-312).  d_z NULL only when sigma == 0.  n = element count (%4). */
int ds_ddim_step(const float* d_eps_u, const float* d_eps_c, const float* d_x, const float* d_z,
                 const float* d_coef, float* d_out, long long n, void* stream);
/* q_sample (:271-294): out = coef[0]*x0 + coef[1]*noise; per_sample > 0: d_coef holds one {a, b} pair per sample of
   per_sample elements (per-sample timesteps, :17-22), 0: one pair for the whole tensor. */
int ds_q_sample(const float* d_x0, const float* d_noise, const float* d_coef, float* d_out, long long n, long long per_sample,
                void* stream);
/* inpaint blend (:499-510): img = m*(coef[0]*guide + coef[1]*noise) + (1-m)*img; mask [B,mask_channels,H,W] with
   mask_channels 1 (broadcast over C) or C (the reference's inpaint caller repeats it, inpaint_with_text.py:229-231). */
int ds_mask_blend(const float* d_guide, const float* d_noise, const float* d_mask, int mask_channels, const float* d_coef,
                  float* d_img, int B, int C, long long hw, void* stream);

/* ----------------------------------------------------------------------------------------
 * U-Net pieces that are not GEMMs (model/diffusion_components.py, model/diffusion.py).
 * -------------------------------------------------------------------------------------- */
/* ConvNextBlock.ds_conv (:118,131) + time-embedding bias (:133-136) + partials of net[0] GroupNorm (:121).
   src_batch_mod > 0: sample n reads sample n % src_batch_mod of source 0 (source 1 is indexed by n).
   out = act16(bias + sum over the 49 taps of x * w), accumulated in fp32.  Two kernels, whose weights differ:
     H >= 16: warp-level tensor cores on 16-row tiles; the weights are rounded to the 16-bit operand type first.
     H <  16: packed fp32 FMA on 8-row tiles; the weights stay fp32.
   The (sum, sumsq) partials are of the fp32 values before the 16-bit rounding. */
int ds_dwconv7(const void* d_src0, const void* d_src1, int C0, int C1, int src_batch_mod, const float* d_weight,
               const float* d_tbias, long long tbias_stride, void* d_out, void* d_stats, float eps, int N, int H, int W, void* stream);
int ds_dwconv7_stats_slots(int C, int H, int W);
/* init_conv 7x7 (model/diffusion.py:82,208) as a tensor-core GEMM: 7x7xCin patches of the fp32 NCHW input -> act16 [N, H, W, 224] (k = ky*32 + kx*4 + ci), then ds_conv_gemm 1x1. */
int ds_stem_im2col(const float* d_x, void* d_col, int N, int Cin, int H, int W, void* stream);
/* SinusoidalPositionEmbeddings (:42-56) and the small Linear layers (time_mlp, per-block mlp,
   label_embedding, label_key/label_query, the text tower's pooler / projections): out = act_out(bias + W . act_in(in));
   act 0 none, 1 GELU(erf), 2 SiLU (act_in only), 3 tanh, 4 ReLU (act_out only). */
int ds_sinusoidal_embedding(const long long* d_t, float* d_out, int N, int dim, void* stream);
/* ConditionalEmbedding for condition_type "instrument_family" (diffusion_components.py:161,167): out[n] = table[ids[n]], fp32. */
int ds_embedding_gather(const float* d_table, const long long* d_ids, float* d_out, int N, int D, int rows, void* stream);
int ds_linear(const float* d_in, long long in_stride, const float* d_w, const float* d_bias, float* d_out,
              long long out_stride, int N, int K, int O, int act_in, int act_out, void* stream);
/* Linear attention core (LinearCrossAttentionAdd.forward :271-293; VQGAN LinearAttention :261-272). */
int ds_attn_chunks(long long npix);
long long ds_attn_part_floats(int N, int heads, long long npix);
int ds_attn_ctx_partial(const void* d_qkv, void* d_q_out, float* d_part, int N, int heads, long long npix,
                        int q_mode, float scale, void* stream);
/* Fused PreNorm (folded GroupNorm(1,C)) + to_qkv + q soft-max + partial context of the U-Net attention (:148-151,263,271-289):
   the to_qkv GEMM on tcgen05 with k and v kept on chip (P = exp(k - m) and S = P^T V in the epilogue); writes only
   q' = softmax_d(q) * scale (act16 [N][npix][128]) and the chunk partials ds_attn_finalize consumes.  heads must be 4 (x 32).
   d_x act16 NHWC [x_batch_mod or N][npix][C]; d_weight act16 [384][C] (q | k | v rows, gamma folded); d_e1 (nullable) / d_e2 fp32 [384];
   d_stats_in statistics buffer of x (nullable); d_sbias fp32 [N][sbias_stride] = label_query | label_key | 0 (nullable). */
int ds_attn_qkv_ctx(const void* d_x, int C, int x_batch_mod, const void* d_stats_in, int stats_in_slots, const void* d_weight,
                    const float* d_e1, const float* d_e2, const float* d_sbias, long long sbias_stride, void* d_q_out, float* d_part,
                    int N, int heads, long long npix, float scale, void* stream);
int ds_attn_finalize(const float* d_part, const float* d_wout, void* d_M, int N, int heads, long long npix,
                     int C, int Cout_pad, void* stream);
/* LinearCrossAttention ("linear_cat", diffusion_components.py:171-207): the condition contributes one extra key / value token,
   k = cat([k, label_key(emb)]), v = cat([v, label_value(emb)]) (:187-195); d_label_k / d_label_v fp32 [N][label_stride]. */
int ds_attn_finalize_cat(const float* d_part, const float* d_label_k, const float* d_label_v, long long label_stride,
                         const float* d_wout, void* d_M, int N, int heads, long long npix, int C, int Cout_pad, void* stream);
/* to_out[1] GroupNorm(1,C) + Residual (:264, :22-29): out = GN(y)*gamma+beta + x.  x_batch_mod > 0: sample n adds x[n % x_batch_mod]. */
int ds_gn_apply_residual(const void* d_y, const void* d_x, void* d_out, const void* d_stats, int slots,
                         const float* d_gamma, const float* d_beta, int N, int C, long long hw, int x_batch_mod, void* stream);

/* ----------------------------------------------------------------------------------------
 * VQGAN (model/VQGAN.py) and the spectrogram <-> waveform transforms (tools.py + librosa call sites).
 * -------------------------------------------------------------------------------------- */
/* VectorQuantizerEMA.forward eval (:98-146): bit-exact argmin over the expanded fp32 distance; out = x+(q-x). */
int ds_vq_quantize(const float* d_x, const float* d_codebook, int K, float* d_out, long long* d_idx,
                   int B, long long hw, void* stream);
/* GroupNorm(G, eps) + activation (Normalize/nonlinearity :12-27) as statistics + apply passes; act 0/1 relu/2 swish. */
int ds_group_stats(const void* d_x, void* d_part, int N, int C, int Cp, int G, long long hw, int chunks, void* stream);
int ds_gn_act(const void* d_x, void* d_out, const void* d_part, int chunks, const float* d_gamma, const float* d_beta,
              int N, int C, int Cp, int G, long long hw, float eps, int act, void* stream);
int ds_add_bf16(const void* d_a, const void* d_b, void* d_out, long long n, void* stream);
/* x[n][pixel][c] += bias[n*bias_stride + c] in place, act16 NHWC [N, hw, C] (bias_stride 0: one row): the time embedding that
   ResnetBlock adds between its two conv + GroupNorm + SiLU blocks (model/diffusion_components.py:79-104, use_convnext=False). */
int ds_add_channel_bias(void* d_x, const float* d_bias, long long bias_stride, int N, int C, long long hw, void* stream);
/* Decoder heads (:394-398): softplus / tanh / tanh of (a + b), fp32 NCHW [N,3,H,W]; b (nin_shortcut branch) nullable. */
int ds_decoder_head(const float* d_a, const float* d_b, float* d_out, int N, long long hw, void* stream);
int ds_nchw_f32_to_nhwc_bf16(const float* d_in, void* d_out, int N, int C, int Cp, long long hw, void* stream);
int ds_nhwc_bf16_to_nchw_f32(const void* d_in, float* d_out, int N, int C, int Cp, long long hw, void* stream);
/* decode_stft + depad_STFT + librosa.istft(hop 256, win 1024) (tools.py:334-345,185-191; utils.py:241). */
long long ds_istft_length(int T);
int ds_stft_decode_istft(const float* d_spec, float* d_frames, float* d_wave, int B, int T, void* stream);
/* librosa.stft(n_fft 1024, hop 256) + pad_STFT + encode_stft (sound2sound_with_text.py:85-94; tools.py:170-182,320-331). */
int ds_stft_encode(const float* d_wave, long long L, float* d_spec, int B, int Tpad, void* stream);
/* tools.decode_stft / tools.encode_stft (tools.py:334-345, 320-331) as stand-alone elementwise kernels behind the numpy drop-ins of
   diffusynth_b200.codec: d_enc [3][plane] real <-> d_D [plane] complex (re, im interleaved); is_double: float64 instead of float32. */
int ds_decode_stft(const void* d_enc, void* d_D, long long plane, int is_double, void* stream);
int ds_encode_stft(const void* d_D, void* d_enc, long long plane, int is_double, void* stream);
/* Griffin-Lim phase update (the loop body of librosa.griffinlim as called by tools.py:63-76,194-223: hop 256, win 1024,
   momentum 0.99): d_rebuilt = ds_stft_encode(ds_stft_decode_istft(d_spec)) as [B,3,512,T]; d_tprev fp32 [B,512,T,2] holds the
   previous rebuilt STFT (ignored and initialised when first != 0); channels 1, 2 (cos, sin) of d_spec are overwritten. */
int ds_griffinlim_update(const float* d_rebuilt, float* d_tprev, float* d_spec, float momentum, int first, int B, int T,
                         void* stream);

/* ----------------------------------------------------------------------------------------
 * Note arrangements (webUI/natural_language_guided_4/track_maker.py:42 after the per-note closure of track_maker.DiffSynth):
 * every note is pitch-shifted, scaled, placed at its onset and summed into one track.  16 kHz throughout.  Host arrays
 * (lengths, n_steps, onsets, offsets, gains) are read and checked before any device work, then uploaded into the workspace with
 * one cudaMemcpyAsync, so these two calls cannot be captured in a graph.
 * -------------------------------------------------------------------------------------- */
/* librosa.effects.pitch_shift(y, sr=16000, n_steps=n_steps[k], bins_per_octave=12) for B items packed back to back in d_in
   (item k: lengths[k] samples, fp32), written to d_out in the same layout: stft(n_fft 2048, hop 512, periodic Hann, centre zero
   padding) -> librosa.phase_vocoder(rate = 2^(-n/12), hop 512) -> istft(length = round(L/rate)) -> resample from 16000/rate to
   16000 Hz -> fix_length(L).  The resampler is a Kaiser-windowed sinc (resampy kaiser_best parameters), not librosa's default
   soxr; n_steps == 0 skips it like librosa.resample.  |n_steps[k]| <= 24, finite.  d_ws: ds_pitch_shift_workspace bytes.  After the
   call the workspace holds the stages at the byte offsets stage_offsets[0..3] (nullable): the STFTs (complex64 [sum T_in][1025],
   T_in = 1 + L/512), the stretched spectra ([sum T_out][1025], T_out = ceil(T_in/rate)), the windowed iSTFT frames (fp32
   [sum T_out][2048]) and the time-stretched signals (fp32, round(L/rate) samples each), all packed in item order. */
int ds_pitch_shift_workspace(const long long* lengths, const double* n_steps, int B, long long* bytes, long long* stage_offsets);
int ds_pitch_shift(const float* d_in, float* d_out, const long long* lengths, const double* n_steps, int B, void* d_ws, long long ws_bytes,
                   void* stream);
/* Track mix (track_maker.py's placement loop): d_track[j] = sum over notes n in input order, fp32, of
   gains[n] * d_src[src_offsets[n] + j - onsets[n]] where 0 <= j - onsets[n] < lengths[n]; no normalisation, no envelope.  A gather
   over track samples, bit-identical run to run.  Every onsets[n] + lengths[n] <= track_len, src_offsets[n] >= 0.  This is
   ds_mix_arrangement with every fade_out 0 and target_peak 0, and its workspace holds those K int64 fades too: as with every
   call here, size d_ws from ds_mix_track_workspace, never from a formula. */
int ds_mix_track_workspace(const long long* lengths, const long long* onsets, int K, long long track_len, long long* bytes);
int ds_mix_track(const float* d_src, const long long* src_offsets, const long long* lengths, const long long* onsets, const float* gains,
                 int K, float* d_track, long long track_len, void* d_ws, long long ws_bytes, void* stream);
/* Arrangement mix (several tracks summed into one piece): ds_mix_track with a linear fade at the end of every note and optional
   peak normalisation.  d_track[j] = sum over notes n in input order, fp32, of gains[n] * env_n(i) * d_src[src_offsets[n] + i],
   i = j - onsets[n], 0 <= i < L = lengths[n]; with F = min(fade_out[n], L), env_n(i) = 1 for i < L - F and (L - i) / F after (1/F on
   the last sample).  A note with fade_out[n] == 0 is summed exactly as ds_mix_track sums it: a fade-free call is bit-identical to
   ds_mix_track.  target_peak > 0 then scales the track in place by target_peak / max|d_track| (computed on the device: no host
   synchronisation; an all-zero track stays zero; bit-identical run to run); 0 leaves it unscaled.  fade_out[n] >= 0, finite
   target_peak >= 0, src_offsets[n] >= 0, every onsets[n] + lengths[n] <= track_len.  d_ws: ds_mix_arrangement_workspace bytes,
   which include one peak partial per 1024 track samples when target_peak > 0. */
int ds_mix_arrangement_workspace(const long long* lengths, const long long* onsets, const long long* fade_out, int K, float target_peak,
                                 long long track_len, long long* bytes);
int ds_mix_arrangement(const float* d_src, const long long* src_offsets, const long long* lengths, const long long* onsets,
                       const float* gains, const long long* fade_out, int K, float target_peak, float* d_track, long long track_len,
                       void* d_ws, long long ws_bytes, void* stream);
/* Stereo arrangement mix: ds_mix_arrangement into two channels, with a constant-power pan per note.  d_out is planar fp32
   [2][track_len], left then right: d_out[c * track_len + j] = sum over notes n in input order, fp32, of
   g_c[n] * env_n(i) * d_src[src_offsets[n] + i], with i and env_n as in ds_mix_arrangement (one envelope for both channels).  The
   pan law is host arithmetic in float64, rounded once to fp32 per note and channel: g_L = fl32(gains[n] * c(1 + pans[n])),
   g_R = fl32(gains[n] * c(1 - pans[n])), c(u) = cos(pi u / 4) with c(2) = 0 exactly.  So pan -1 is hard left (g_L = gains[n]
   exactly, g_R = 0), pan 0 gives g_L == g_R (-3 dB each) and pans p and -p swap the two gains exactly.  target_peak > 0 then
   scales both channels in place by ONE factor, target_peak / max over both channels of |d_out| (the balance between channels is
   kept; no host synchronisation; an all-zero piece stays zero).  Every check of ds_mix_arrangement applies; pans is non-null and
   every pans[n] is finite with |pans[n]| <= 1.  d_ws: ds_mix_stereo_workspace bytes.  Bit-identical run to run. */
int ds_mix_stereo_workspace(const long long* lengths, const long long* onsets, const long long* fade_out, const float* pans, int K,
                            float target_peak, long long track_len, long long* bytes);
int ds_mix_stereo(const float* d_src, const long long* src_offsets, const long long* lengths, const long long* onsets, const float* gains,
                  const float* pans, const long long* fade_out, int K, float target_peak, float* d_out, long long track_len, void* d_ws,
                  long long ws_bytes, void* stream);
/* Batched linear convolution (scipy.signal.fftconvolve along the last axis; a project extension, used for convolution reverb):
   B signals packed back to back in d_x (item k: x_lengths[k] = N_k samples, fp32) and H impulse responses packed in d_h (IR i:
   h_lengths[i] samples).  Item k is convolved with IR h_index[k] (items may share an IR, whose spectra are computed once), and
   writes out_lengths[k] samples of its full convolution (N_k + M - 1 samples, M = h_lengths[h_index[k]]) starting at full index
   out_start[k], packed back to back in item order in d_out: mode "full" is out_start 0, out_lengths N + M - 1; "same" and
   "valid" are crops of it.  Arithmetic: uniformly partitioned FFTs, P = 1024, 2048-point real transforms in fp32.  Output
   segment s is Y_s = sum over q in ASCENDING order of X_{s-q} * H_q (1025 complex bins each), inverse-transformed to the 2047
   samples at s * 1024; output j = seg_s[j - 1024 s] + seg_{s-1}[j - 1024 (s-1)], added in that order.  No atomics: item k's
   result does not depend on the rest of the batch (a batch equals each item run alone, bit for bit) and repeats bit for bit.
   accumulate 0 overwrites d_out; 1 writes fl(d_out[j] + conv[j]).  target_peak > 0 then scales ALL outputs of the call in place
   by ONE factor, target_peak / max |d_out| over every item (both channels of a stereo piece are items of one call; an all-zero
   output stays zero; no host synchronisation); 0 leaves them unscaled.  Checks, before any device work: non-null pointers;
   B, H >= 1; every length >= 1; 0 <= h_index[k] < H; out_start[k] >= 0 and out_start[k] + out_lengths[k] <= N_k + M - 1;
   finite target_peak >= 0; accumulate 0 or 1; ws_bytes large enough.  d_ws: ds_fftconvolve_workspace bytes (the metadata, the
   spectra of every block and partition, 8200 bytes per 1024 samples, and the segments, 8192 bytes per 1024 output samples
   computed).  4 launches, 3 without a peak, and one host-to-device copy, whatever B, N and M. */
int ds_fftconvolve_workspace(const long long* x_lengths, int B, const long long* h_lengths, int H, const long long* h_index,
                             const long long* out_start, const long long* out_lengths, float target_peak, long long* bytes);
int ds_fftconvolve(const float* d_x, const float* d_h, float* d_out, const long long* x_lengths, int B, const long long* h_lengths, int H,
                   const long long* h_index, const long long* out_start, const long long* out_lengths, int accumulate, float target_peak,
                   void* d_ws, long long ws_bytes, void* stream);

/* ----------------------------------------------------------------------------------------
 * Sample-rate conversion of uploaded audio (tools.adjust_audio_length, tools.py:126-151, as sound2sound_with_text.py:75-82 calls
 * it): librosa.resample(x, orig_sr=sr_in[k], target_sr=sr_out[k], res_type="kaiser_best") for B items packed back to back in d_in
 * (item k: lengths[k] samples, fp32), each written to d_out (packed, item k: out_lengths[k] samples, or librosa's length
 * ceil(lengths[k] * (sr_out[k] / sr_in[k])) evaluated in float64 when out_lengths is NULL): zero past librosa's length, cropped
 * below it (fix_length fused).  out_k[j] = sum_i xn_k[i] h(i - j * sr_in/sr_out) with pitch.cu's filter (resampy kaiser_best
 * parameters, not librosa's default soxr); equal rates copy.  normalize_peak != 0 first divides item k by max(max|x_k|, 1e-12)
 * (IEEE division), as the upload handler does.  Integer rates in 1..DS_RESAMPLE_MAX_RATE and lengths in 1..DS_RESAMPLE_MAX_LENGTH,
 * so that j * (sr_in / gcd) stays in int64.  Pairs whose polyphase table has more than 2^20 coefficients (e.g. 44101 -> 16000) or
 * whose staged window is too large evaluate the same coefficients per tap, with bit-identical results; DS_RESAMPLE_DIRECT=1 in
 * the environment makes every pair do so (A/B timing).  Each output sums its taps in ascending input order: an item's result
 * does not depend on the rest of the batch.  Host arrays are checked before any device work and uploaded with one
 * cudaMemcpyAsync; 2 launches, 3 with normalize_peak, whatever B.  d_ws: ds_resample_workspace bytes. */
#define DS_RESAMPLE_MAX_RATE 4194304LL
#define DS_RESAMPLE_MAX_LENGTH 1099511627776LL
int ds_resample_workspace(const long long* lengths, const long long* sr_in, const long long* sr_out, const long long* out_lengths, int B,
                          long long* bytes);
int ds_resample(const float* d_in, float* d_out, const long long* lengths, const long long* sr_in, const long long* sr_out,
                const long long* out_lengths, int normalize_peak, int B, void* d_ws, long long ws_bytes, void* stream);

/* ----------------------------------------------------------------------------------------
 * Mask zoom for inpainting with text (webUI/natural_language_guided_4/inpaint_with_text.py: the spectrogram mask is shrunk to the
 * latent grid): scipy.ndimage.zoom(a, (h/H, w/W)) with scipy's defaults (order 3, mode 'constant', prefilter, grid_mode False)
 * for B 2-D fp32 arrays packed back to back in d_in (item k: in_shapes[2k] x in_shapes[2k+1], row-major), each written to d_out
 * (packed, item k: out_shapes[2k] x out_shapes[2k+1]).  Separable: the cubic B-spline prefilter (mirror boundary) and the
 * interpolation at x = o * (n-1)/(out-1) run along the rows' axis, then along the columns' axis, in float64 as scipy does; the
 * result is rounded once to fp32.  Every dimension in 1..DS_MASK_ZOOM_MAX_DIM, so that every element and byte offset of up to
 * 2^31 items fits in int64.  Each output sums in a fixed order: an item's result does not depend on the rest of the batch.  Host
 * arrays are checked before any device work and uploaded with one cudaMemcpyAsync; 2 launches whatever B.
 * d_ws: ds_mask_zoom_workspace bytes.
 * -------------------------------------------------------------------------------------- */
#define DS_MASK_ZOOM_MAX_DIM 16384LL
int ds_mask_zoom_workspace(const long long* in_shapes, const long long* out_shapes, int B, long long* bytes);
int ds_mask_zoom(const float* d_in, float* d_out, const long long* in_shapes, const long long* out_shapes, int B, void* d_ws,
                 long long ws_bytes, void* stream);

/* ----------------------------------------------------------------------------------------
 * Timbre morph rows (model/DiffSynthSampler.py:224-269, generate_linear_noise with both endpoints, as interpolate uses it, batched):
 * P sequences x N frames (N >= 2), row p*N + k = frame k of sequence p, a = k / (N - 1).  d_e0 / d_e1: endpoint noises [P, n] fp32
 * (n % 4 == 0; n = 4*128*64 for the repeat strategy's train-width noise), d_c0 / d_c1: endpoint conditions [P, L] fp32.  Writes
 * d_noise [P*N, n] and d_cond [P*N, L].
 *   DS_MORPH_LINEAR (:170-174): fl(fl(a e1) + fl((1 - a) e0)) with a, 1 - a evaluated in double and rounded to fp32 (as torch
 *     rounds a Python scalar), no FMA contraction: bit-identical to generate_linear_noise.
 *   DS_MORPH_SLERP (no reference entry): theta = acos(clamp(<e0,e1> / (|e0| |e1|), -1, 1)) per sequence from a float64 reduction in
 *     a fixed order; row = fl(w0 e0 + w1 e1), w0 = sin((1 - a) theta) / sin theta, w1 = sin(a theta) / sin theta, in float64.  A
 *     sequence with sin theta < 1e-6 (identical or antipodal endpoints) or a zero endpoint takes the linear rows.  Frames 0 and
 *     N - 1 equal the endpoints exactly.
 * Conditions always take the linear expression, except that an element equal in both endpoints is copied as it is (so equal
 * conditions give every frame exactly that condition).  A sequence's rows do not depend on P (bit for bit) and repeat run to run.  Every
 * argument is checked before any device work, including P * N * max(n, L) in int64; no host synchronisation.  Launches: 1 (linear),
 * 2 (slerp).  d_ws: ds_morph_rows_workspace bytes (0 for the linear path, where d_ws may be NULL).
 * -------------------------------------------------------------------------------------- */
#define DS_MORPH_LINEAR 0
#define DS_MORPH_SLERP 1
int ds_morph_rows_workspace(int P, int N, long long n, long long L, int path, long long* bytes);
int ds_morph_rows(const float* d_e0, const float* d_e1, const float* d_c0, const float* d_c1, int P, int N, long long n, long long L,
                  int path, float* d_noise, float* d_cond, void* d_ws, long long ws_bytes, void* stream);

/* ----------------------------------------------------------------------------------------
 * Image products of the decode glue (webUI/natural_language_guided_4/utils.py), batched:
 *   spectrogram_to_Gradio_image (:8-50, with tools.np_power_to_db tools.py:41-50) and phase_to_Gradio_image (:53-91)
 *   of |D| / angle(D) for D = depad_STFT(decode_stft(spec)) (:229-238): uint8 [B, 513, T, 3], flipped vertically;
 *   latent_representation_to_Gradio_image (:94-128): per-channel min-max to 0..255, 8x enlarged, flipped: uint8 [B, 8H, 8W, 4].
 * dB scale and angle are evaluated in float64 like the reference (numpy on complex128).
 * -------------------------------------------------------------------------------------- */
int ds_spec_images(const float* d_spec, void* d_mag_img, void* d_phase_img, void* d_absmax /* scratch: 8 bytes per sample */,
                   int B, int T, void* stream);
int ds_latent_image(const float* d_lat, void* d_img, void* d_minmax /* scratch: 32 bytes per sample */, int B, int H, int W,
                    void* stream);

/* ----------------------------------------------------------------------------------------
 * Text-conditioning front end (text2sound.py:89-109 -> multi_modal_model.get_text_features, model/multimodal_model.py:114-116):
 * transformers' ClapTextModel (RoBERTa-base) + ClapProjectionLayer + L2 normalisation, then ProjectionHead (:14-47).  The dense
 * layers are ds_conv_gemm calls over the token axis; these are the remaining pieces (diffusynth_b200/text.py is the host).
 * -------------------------------------------------------------------------------------- */
/* ClapTextEmbeddings: LayerNorm(word[ids] + position[cumsum(ids != pad) * (ids != pad) + pad] + token_type[0]) -> act16 [B*L][D]. */
int ds_text_embed_ln(const long long* d_ids, const float* d_word, const float* d_pos, const float* d_type0, const float* d_gamma, const float* d_beta,
                     void* d_out, int B, int L, int D, int pad_idx, float eps, void* stream);
/* LayerNorm over the rows of act16 [T][D], in place (post-LN blocks: the residual is added by the producing GEMM's epilogue). */
int ds_layernorm_rows(void* d_x, const float* d_gamma, const float* d_beta, int T, int D, float eps, void* stream);
/* softmax(q k^T * scale + mask) v per (sample, head), head size 64: d_qkv act16 [B][L][3*heads*64] (q | k | v), d_mask int64 [B][L],
   d_out act16 [B][L][heads*64]. */
int ds_text_attention(const void* d_qkv, const long long* d_mask, void* d_out, int B, int L, int heads, float scale, void* stream);
int ds_cls_gather(const void* d_x, float* d_out, int B, int L, int D, void* stream);                 /* fp32 out[b] = x[b][0][:] */
int ds_l2_normalize_rows(float* d_x, int B, int D, void* stream);                                     /* F.normalize(x, dim=-1) in place */
/* ProjectionLayer tail (multimodal_model.py:28-31): x = LayerNorm(x + y) * gamma + beta, fp32 rows, in place on x. */
int ds_add_layernorm_rows_f32(float* d_x, const float* d_y, const float* d_gamma, const float* d_beta, int B, int D, float eps, void* stream);

/* ========================================================================================
 * Module-level entry points (SURVEY section 8b): the network plans, the weight packing and the sampling graph live behind
 * opaque handles inside the library, so a host in any language loads a reference checkpoint by its state_dict names and runs
 * whole modules; the Python classes of diffusynth_b200/ are thin hosts over exactly these calls.  A handle belongs to one
 * device (the current device of the creating thread) and to one host thread at a time; distinct handles are independent.
 * ====================================================================================== */
#define DS_MAX_LEVELS 8

/* ---- ConditionedUnet (model/diffusion.py:21-258; ctor arguments :22-33) ---- */
typedef struct ds_unet_config {
  int32_t in_dim, out_dim;                 /* out_dim <= 0: in_dim (diffusion.py:35) */
  int32_t n_levels;                        /* len(down_dims) == len(up_dims) */
  int32_t down_dims[DS_MAX_LEVELS], up_dims[DS_MAX_LEVELS];
  int32_t mid_depth;                       /* <= 0: 3 */
  int32_t with_time_emb;                   /* 0: no time_mlp, blocks without their mlp (diffusion.py:107-109) */
  int32_t time_dim;                        /* <= 0: 4 * down_dims[0] (diffusion.py:99) */
  int32_t use_convnext;                    /* 1: ConvNextBlock (deployed); 0: ResnetBlock (diffusion_components.py:59-104) */
  int32_t convnext_mult;                   /* <= 0: 2 */
  int32_t attn_type;                       /* 0 = "linear_add" (deployed, app.py:40), 1 = "linear_cat" */
  int32_t condition_type;                  /* 0 = "natural_language_prompt" (d_cond fp32 [N][label_emb_dim]), 1 = "instrument_family" (d_cond int64 [N]) */
  int32_t label_emb_dim;
  int32_t n_label_class;                   /* condition_type 1: the embedding table has n_label_class + 1 rows (diffusion.py:63-64) */
  int32_t resnet_block_groups;             /* use_convnext 0: GroupNorm groups of the ResnetBlocks (<= 0: 8) */
  int32_t batch_invariant;                 /* 0: jobs too small to fill the SMs run narrow N tiles (lower latency; a sample's low-order bits then depend on the
                                              batch it runs in, through the grouping of the GroupNorm partial sums); 1: always the widest tiling, every sample
                                              bit-identical whatever the batch / shard it is part of */
} ds_unet_config;
typedef struct ds_unet ds_unet;
int ds_unet_create(const ds_unet_config* cfg, ds_unet** out);       /* -4 for an unknown attn_type / condition_type */
void ds_unet_destroy(ds_unet* h);
/* One parameter by its reference state_dict name (e.g. "downs.0.0.net.1.weight"); fp32, `data` may be host or device memory. */
int ds_unet_load(ds_unet* h, const char* name, const float* data, const long long* shape, int ndim);
/* Pack the loaded parameters for the device (fails naming the first missing / mis-shaped parameter).  Invalidates earlier plans. */
int ds_unet_finalize(ds_unet* h);
/* model(x, time, condition) (diffusion.py:187-258): d_x fp32 [N,in_dim,H,W], d_t int64 [N], d_cond fp32 [N,label_emb_dim] (or int64
   [N] class labels; NULL = condition=None) -> d_out fp32 [N,out_dim,H,W].  The call sequence of a given (N, H, W) is built on first
   use and replayed afterwards. */
int ds_unet_forward(ds_unet* h, const float* d_x, const long long* d_t, const void* d_cond, float* d_out, int N, int H, int W,
                    void* stream);
/* The plan of one evaluation shape, for hosts that drive the sampling loop themselves (generic sampler loops, per-step probes):
   x_batch_mod > 0 with uniform_time = the guidance-doubled batch of DiffSynthSampler.ddim_sample (:307-319): N = 2 * x_batch_mod
   samples read x_batch_mod latents and ONE timestep (d_t[0]).  d_cond / d_eps are the plan's own device buffers. */
typedef struct ds_unet_plan_io {
  int32_t plan;                            /* plan id for ds_unet_plan_run* */
  float* d_cond;                           /* [N][label_emb_dim] (int64 [N] for class labels): write the conditions here, then ds_unet_plan_run_cond */
  float* d_eps;                            /* [N][out_dim][H][W]: result of ds_unet_plan_run */
  int32_t launches, cond_launches;         /* kernels per ds_unet_plan_run / ds_unet_plan_run_cond */
} ds_unet_plan_io;
int ds_unet_plan_get(ds_unet* h, int N, int H, int W, int x_batch_mod, int uniform_time, ds_unet_plan_io* io);
int ds_unet_plan_run_cond(ds_unet* h, int plan, void* stream);      /* label_embedding + label_query / label_key: step-invariant */
int ds_unet_plan_run(ds_unet* h, int plan, const float* d_x, const long long* d_t, void* stream);

/* ---- VQGAN (model/VQGAN.py:403-458; ctor arguments :404-418) ---- */
typedef struct ds_vqgan_config {
  int32_t in_channels, out_channels, embedding_dim;      /* embedding_dim must be 4 */
  int32_t n_hidden, hidden_channels[DS_MAX_LEVELS];
  int32_t block_depth;
  int32_t n_attn_pos, attn_pos[DS_MAX_LEVELS];
  int32_t attn_with_skip;
  int32_t act_relu;                        /* 1: act_type == "relu", 0: swish (decoder ResnetBlocks; the encoder's are always swish, :441) */
  int32_t num_embeddings, num_groups;
  int32_t batch_invariant;                 /* as ds_unet_config.batch_invariant */
} ds_vqgan_config;
typedef struct ds_vqgan ds_vqgan;
int ds_vqgan_create(const ds_vqgan_config* cfg, ds_vqgan** out);
void ds_vqgan_destroy(ds_vqgan* h);
int ds_vqgan_load(ds_vqgan* h, const char* name, const float* data, const long long* shape, int ndim);   /* "_decoder._layers.0.weight", ... */
int ds_vqgan_finalize(ds_vqgan* h);
/* VectorQuantizerEMA.forward eval (:98-146) with the handle's codebook; Decoder.forward (:390-400): d_latent fp32 [B,4,H,W] ->
   d_spec fp32 [B,out_channels,4H,4W]; Encoder.forward (:323-326): d_spec fp32 [B,in_channels,H,W] -> d_latent fp32 [B,4,H/4,W/4]. */
int ds_vqgan_quantize(ds_vqgan* h, const float* d_x, float* d_out, long long* d_idx, int B, long long hw, void* stream);
int ds_vqgan_decode(ds_vqgan* h, const float* d_latent, float* d_spec, int B, int H, int W, void* stream);
int ds_vqgan_encode(ds_vqgan* h, const float* d_spec, float* d_latent, int B, int H, int W, void* stream);

/* ---- the sampling loop as ONE CUDA graph (model/DiffSynthSampler.py:425-517 p_sample_loop; tail = text2sound.py:128-134,
   utils.py:224-241): n_iter x [ U-Net on the (guidance-doubled) batch, fused CFG + DDIM/DDPM update, optional inpaint blend ],
   then quantiser -> decoder -> STFT+ decode + iSTFT.  All buffers are caller-owned device memory at fixed addresses; the
   step-dependent scalars live in the tables, so one graph serves every schedule / seed / prompt of its shape. ---- */
typedef struct ds_sample_buffers {
  float* d_imgs;                 /* [n_iter+1][B,C,H,W]: [0] = start latent (input), [k+1] = latent after step k */
  const float* d_coef;           /* [n_iter][8]: ds_ddim_step coefficients of step k */
  const long long* d_ttab;       /* [n_iter]: timestep fed to the U-Net at step k (timestep_map of the respaced schedule) */
  const float* d_noise;          /* [n_iter][B,C,H,W] per-step noise (ddpm), or NULL (ddim, sigma = 0) */
  const float* d_cond;           /* [N][label_emb_dim], N = 2B with guidance ([uncond x B | cond]) else B; read at every run */
  const float* d_guide;          /* inpainting (:499-510), all four or none: guide latent [B,C,H,W] */
  const float* d_init_noise;     /*   the noise q_sample mixes into the guide [B,C,H,W] */
  const float* d_masks;          /*   [n_iter][B,C,H,W] */
  const float* d_blend_coef;     /*   [n_iter][2] */
  float* d_quantized;            /* tail outputs (with a ds_vqgan): [B,C,H,W] */
  long long* d_indices;          /*   [B*H*W] codebook indices */
  float* d_spec;                 /*   [B,3,4H,4W] or NULL */
  float* d_wave;                 /*   [B, ds_istft_length(4W)] or NULL */
} ds_sample_buffers;
typedef struct ds_sample_graph ds_sample_graph;
/* cfg_on: classifier-free guidance (CFG != 1.0, :307-319); vqgan NULL: no tail; use_graph 0 replays the launches eagerly
   (profilers that cannot follow a captured graph).  Runs one warm-up step on `stream` before capturing. */
int ds_sample_graph_build(ds_unet* unet, ds_vqgan* vqgan, const ds_sample_buffers* bufs, int B, int H, int W, int n_iter, int cfg_on,
                          int use_graph, void* stream, ds_sample_graph** out);
int ds_sample_graph_run(ds_sample_graph* g, void* stream);
int ds_sample_graph_launches(const ds_sample_graph* g);     /* kernels per ds_sample_graph_run */
void ds_sample_graph_destroy(ds_sample_graph* g);

/* ---- the one collective of the sharded job (SURVEY 8e): an all-gather of the rank-local waveforms over NCCL.  The library binds
   libnccl.so.2 at run time (the copy already loaded in the process, e.g. PyTorch's, else the system one). ---- */
typedef struct ds_comm ds_comm;
int ds_comm_unique_id(void* id128);                                        /* rank 0: 128 bytes to hand to every rank */
int ds_comm_init(int rank, int world, const void* id128, ds_comm** out);  /* -3 on any NCCL failure */
/* dtype: 0 = fp32, 1 = act16, 2 = int64; count = elements contributed per rank; d_recv holds world * count. */
int ds_allgather(ds_comm* c, const void* d_send, void* d_recv, long long count, int dtype, void* stream);
void ds_comm_destroy(ds_comm* c);

#ifdef __cplusplus
}
#endif
#endif /* DIFFUSYNTH_B200_H */
