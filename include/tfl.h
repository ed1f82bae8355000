/* tfl.h -- C ABI of the B200-native TF-Locoformer separation forward path.
 *
 * The reference (chynggi/mss-tf-locoformer) is pure Python on PyTorch; the "FFI" a
 * maintainer binds is therefore ctypes (see INTEGRATION.md).  Every entry point below
 * replaces a reference nn.Module.forward (file:line cited per function), takes plain
 * device pointers + sizes + a cudaStream_t, is asynchronous on that stream, never
 * allocates or frees device memory and keeps no pointer past the call (the packed-weight
 * buffer and workspace are caller-owned).  Return value: 0 = OK, < 0 = error
 * (tfl_last_error() gives the message for the calling thread).
 *
 * Activation layout: channels-last [B, Tf, F, C] fp32 ("x"); spectrograms are
 * [B, (S,) Tf, F] interleaved (re, im) fp32 == torch.complex64.
 */
#ifndef TFL_H_
#define TFL_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* tfl_stream_t; /* == cudaStream_t */

#define TFL_PRECISION_FP32 0 /* CUDA-core fp32 everywhere: the <=1e-4 / >=70 dB parity mode            */
#define TFL_PRECISION_BF16 1 /* tcgen05 bf16 MMAs with fp32 TMEM accumulation, fp32 residual stream      */
/* TFL_PRECISION_TF32: what the reference computes on a GPU without autocast (cuDNN convolutions in TF32 by default,
 * matmuls and SDPA in fp32):
 *   STFT, iSTFT, RMSGroupNorm, gLN statistics, RoPE, residual stream   exact fp32, as in TFL_PRECISION_FP32
 *   encoder conv + gLN, decoder                                        the tf32 mma.sync kernels of TFL_PRECISION_BF16
 *   ConvSwiGLU FFN (conv1d + SwiGLU, transposed conv + bias + residual) tcgen05 kind::tf32: operands rounded to tf32
 *                                                                      (cvt.rna), fp32 accumulation in TMEM
 *   q|k|v projection + RoPE, attention, head merge + residual          exact fp32, as in TFL_PRECISION_FP32
 * Workspace layout and size are those of TFL_PRECISION_FP32. */
#define TFL_PRECISION_TF32 2
#define TFL_AXIS_FREQ 0      /* sequences run along F, one per (b, t)  -- freq_path                      */
#define TFL_AXIS_TIME 1      /* sequences run along Tf, one per (b, f) -- frame_path                     */

/* Constructor arguments of TFLocoformerMSS (models/mss_tflocoformer.py:104-129) /
 * TFLocoformerSeparator (standalone/tflocoformer_separator.py:59-81). */
typedef struct tfl_config {
  int32_t n_fft;        /* 0 for spectrogram-in/spectrogram-out separators */
  int32_t hop;
  int32_t n_src;        /* n_sources / num_spk */
  int32_t n_layers;
  int32_t emb_dim;      /* C */
  int32_t num_groups;   /* RMSGroupNorm groups */
  int32_t tf_order;     /* 0 = "ft", 1 = "tf" */
  int32_t n_heads;
  int32_t attention_dim;
  int32_t rope;         /* 1 = pos_enc "rope", 0 = "nope" */
  int32_t macaron;      /* 1 when ffn_type is a 2-list */
  int32_t ffn_hidden0;  /* hidden dim of ffn[0] (post-attention; LAST entry of the config list) */
  int32_t ffn_hidden1;  /* hidden dim of ffn[1] (pre-attention; FIRST entry), 0 if !macaron    */
  int32_t conv_kernel;  /* conv1d_kernel; conv1d_shift must be 1 */
  int32_t enc_in_ch;    /* input channels of the encoder conv: 2 (re, im); 0 = no conv encoder/decoder (band-split) */
  float eps;
} tfl_config;

typedef struct tfl_plan tfl_plan;

int tfl_version(void);
const char* tfl_last_error(void);
/* Kernels launched by this library since it was loaded (host-side counter). */
uint64_t tfl_launch_count(void);

int tfl_plan_create(const tfl_config* cfg, tfl_plan** out);
void tfl_plan_destroy(tfl_plan* plan);

/* Number of fp32 weight pointers tfl_pack_weights expects, and the packed size.
 * Pointer order == reference state_dict order (SURVEY.md section 8b):
 *   conv.0.weight, conv.0.bias, conv.1.weight, conv.1.bias,                      (if enc_in_ch)
 *   per layer i, per path p in (freq_path, frame_path):
 *     [ffn_norm.0.gamma, ffn_norm.1.gamma if macaron], then per ffn j in (0[,1]):
 *     conv1d.weight, conv1d.bias, deconv1d.weight, deconv1d.bias;
 *     attn_norm.gamma, [attn.rope.freqs if rope], attn.qkv.weight, attn.aggregate_heads.0.weight
 *   deconv.weight, deconv.bias                                                  (if enc_in_ch) */
int tfl_num_weight_tensors(const tfl_plan* plan);
size_t tfl_packed_bytes(const tfl_plan* plan);
int tfl_pack_weights(const tfl_plan* plan, const float* const* weights, int n_weights,
                     void* packed, size_t packed_bytes, tfl_stream_t stream);

size_t tfl_workspace_bytes(const tfl_plan* plan, int batch, int n_frames, int n_freq, int precision);

/* models/mss_tflocoformer.py:36-54 + :207-214.  audio [B, T] -> spec [B, Tf, F, 2]. */
int tfl_stft(const tfl_plan* plan, const void* packed, const float* audio, int batch, int n_samples,
             float* spec, tfl_stream_t stream);
/* :141-146, :218-219.  spec [B, Tf, F, Cin] -> x [B, Tf, F, C] (conv 3x3 + gLN). */
int tfl_enc_conv_gln(const tfl_plan* plan, const void* packed, const float* spec, int batch, int n_frames,
                     int n_freq, float* x, void* workspace, size_t ws_bytes, tfl_stream_t stream);
/* The same stage in the arithmetic of `precision`: TFL_PRECISION_FP32 = tfl_enc_conv_gln; TFL_PRECISION_BF16 = the tf32
 * mma.sync encoder that tfl_forward / tfl_separator_forward run in bf16 mode (spectrogram and weights rounded to tf32,
 * fp32 sums, gLN statistics in double); TFL_PRECISION_TF32 runs the same kernels as TFL_PRECISION_BF16. */
int tfl_enc_conv_gln_mode(const tfl_plan* plan, const void* packed, const float* spec, int batch, int n_frames,
                          int n_freq, float* x, void* workspace, size_t ws_bytes, int precision, tfl_stream_t stream);
/* :682-706.  x [rows, C] -> y [rows, C] with the gamma of (layer, axis, which) where
 * which = 0: ffn_norm.0, 1: ffn_norm.1, 2: attn_norm. */
int tfl_rms_group_norm(const tfl_plan* plan, const void* packed, int layer, int axis, int which,
                       const float* x, float* y, int64_t rows, tfl_stream_t stream);
/* :443-447 / :459-462 -> :626-655.  In place: x += ConvSwiGLU(RMSGroupNorm(x)) along `axis`. */
int tfl_conv_swiglu_ffn(const tfl_plan* plan, const void* packed, int layer, int axis, int ffn_index,
                        float* x, int batch, int n_frames, int n_freq, void* workspace, size_t ws_bytes,
                        int precision, tfl_stream_t stream);
/* Same sub-block, out of place: y = x + ConvSwiGLU(RMSGroupNorm(x)); x and y must not overlap.  This is the form the
 * bf16 kernel computes natively (tfl_blocks ping-pongs two residual buffers); the in-place call above adds a copy. */
int tfl_conv_swiglu_ffn_out(const tfl_plan* plan, const void* packed, int layer, int axis, int ffn_index,
                            const float* x, float* y, int batch, int n_frames, int n_freq, void* workspace,
                            size_t ws_bytes, int precision, tfl_stream_t stream);
/* :452-456 -> :504-559.  In place: x += MHSA_RoPE(RMSGroupNorm(x)) along `axis`. */
int tfl_rope_attn(const tfl_plan* plan, const void* packed, int layer, int axis, float* x, int batch,
                  int n_frames, int n_freq, void* workspace, size_t ws_bytes, int precision,
                  tfl_stream_t stream);
/* :182, :229-237.  x [B, Tf, F, C] -> est [B, S, Tf, F, 2] (complex64 [B, S, Tf, F]). */
int tfl_dec_conv(const tfl_plan* plan, const void* packed, const float* x, int batch, int n_frames,
                 int n_freq, float* est, tfl_stream_t stream);
/* The same stage in the arithmetic of `precision`: TFL_PRECISION_FP32 = tfl_dec_conv; TFL_PRECISION_BF16 = the tf32
 * mma.sync decoder that tfl_forward / tfl_separator_forward run in bf16 mode (operands rounded to tf32, fp32 sums);
 * TFL_PRECISION_TF32 runs the same kernels as TFL_PRECISION_BF16. */
int tfl_dec_conv_mode(const tfl_plan* plan, const void* packed, const float* x, int batch, int n_frames,
                      int n_freq, float* est, int precision, tfl_stream_t stream);
/* :56-75, :239-250.  est [B, S, Tf, F, 2] -> audio [S, B, n_samples] (all sources, one launch). */
int tfl_istft_ola(const tfl_plan* plan, const void* packed, const float* est, int batch, int n_frames,
                  int n_samples, float* audio, tfl_stream_t stream);
/* :222-226.  All n_layers TFLocoformerBlocks in place on x. */
int tfl_blocks(const tfl_plan* plan, const void* packed, float* x, int batch, int n_frames, int n_freq,
               void* workspace, size_t ws_bytes, int precision, tfl_stream_t stream);
/* TFLocoformerMSS.forward, :184-258.  mixture [B, T] -> audio [S, B, T]; est_spec (optional,
 * may be NULL) receives the separated spectrograms [B, S, Tf, F, 2]. */
int tfl_forward(const tfl_plan* plan, const void* packed, const float* mixture, int batch, int n_samples,
                float* audio, float* est_spec, void* workspace, size_t ws_bytes, int precision,
                tfl_stream_t stream);
/* TFLocoformerSeparator.forward, standalone/tflocoformer_separator.py:131-171.
 * spec [B, T, F, 2] -> est [B, S, T, F, 2]. */
int tfl_separator_forward(const tfl_plan* plan, const void* packed, const float* spec, int batch,
                          int n_frames, int n_freq, float* est, void* workspace, size_t ws_bytes,
                          int precision, tfl_stream_t stream);
/* Full-track stitch (new; SURVEY.md F3): track[S, n_track] += window(seg) * seg_audio[S, B, seg_len]
 * for segments seg_index0 .. seg_index0 + B - 1 of n_seg_total at 50 % overlap.  `track` holds the samples
 * [track_origin, track_origin + n_track) of the full track (a rank's own range plus its halo; 0 = whole track). */
int tfl_segment_ola(const float* seg_audio, int n_src, int batch, int seg_len, int seg_index0,
                    int n_seg_total, float* track, int64_t n_track, int64_t track_origin, tfl_stream_t stream);
/* The same stitch at any hop (0 < hop < seg_len, segment i starts at i * hop) and over several channels:
 * track[rows, channels, n_track] += sum_i w_i * seg_audio[rows, batch * channels, seg_len] / E, where row
 * b * channels + c of seg_audio is channel c of segment seg_index0 + b, and E(t) = sum of the windows of all
 * n_seg_total segments covering sample t (1 at hop = seg_len / 2).  One thread per output sample, no atomics:
 * bitwise reproducible for a given batch.  `track` holds samples [track_origin, track_origin + n_track). */
int tfl_segment_ola_hop(const float* seg_audio, int rows, int channels, int batch, int seg_len, int hop,
                        int seg_index0, int n_seg_total, float* track, int64_t n_track, int64_t track_origin,
                        tfl_stream_t stream);

/* evaluation/metrics.py:14-168 on the device.  est, tgt [rows, n] fp32 -> out5 [rows][5] double =
 * {sum e, sum t, sum e^2, sum t^2, sum e*t}: SI-SDR, SDR and the file's "SAR" / "SIR" are closed forms of these sums
 * (mss_tf_locoformer_b200/metrics.py).  scratch: >= rows * 64 * 5 doubles. */
int tfl_pair_stats(const float* est, const float* tgt, int rows, int64_t n, double* out5, double* scratch,
                   size_t scratch_bytes, tfl_stream_t stream);

/* ---- training step (SURVEY.md section 8(f) N1): /root/reference/training/train.py:68-172 ------------------------------
 * fp32 on CUDA cores.  Gradients leave in ONE flat fp32 buffer: one slice per state_dict tensor, in tfl_pack_weights order
 * and in the reference's own tensor layout, so param.grad of the reference model is the parity target, the data-parallel
 * all-reduce is one NCCL call on the buffer, and clipping + AdamW are two kernels over it. */
typedef struct tfl_loss_config {   /* MSSLoss(loss_type='combined'), models/mss_loss.py:18-109 */
  float si_sdr_weight, l1_weight, spectral_weight, eps;
  int32_t spec_n_fft, spec_hop;    /* SpectralLoss STFT (2048 / 1024 in the reference, :184-193) */
} tfl_loss_config;
/* Returns the flat buffer's length in floats; offsets[i] = start of tensor i's gradient (-1: not trainable, i.e.
 * attn.rope.freqs), sizes[i] = its element count (both may be NULL). */
int64_t tfl_train_grad_layout(const tfl_plan* plan, int64_t* offsets, int64_t* sizes, int n_weights);
size_t tfl_train_workspace_bytes(const tfl_plan* plan, int batch, int n_samples, int spec_n_fft, int spec_hop);
size_t tfl_train_stage_workspace_bytes(const tfl_plan* plan, int batch, int n_frames, int n_freq);
/* forward (sub-block inputs saved) -> MSSLoss -> backward.  `weights`: the raw fp32 device tensors tfl_pack_weights took
 * (the data-gradient GEMMs read qkv.weight / aggregate_heads.weight in place); mixture [B, T]; targets [S, B, T] (mono,
 * train.py:103-110); grads: flat buffer (overwritten); loss_out[0] = total_loss, then {si_sdr, l1, spectral} per source
 * (device, 1 + 3 S floats); est_audio (optional) [S, B, T].  Dropout is not applied (p = 0). */
int tfl_train_forward_backward(const tfl_plan* plan, const void* packed, const float* const* weights, int n_weights,
                               const float* mixture, const float* targets, int batch, int n_samples,
                               const tfl_loss_config* loss, float* grads, float* loss_out, float* est_audio,
                               void* workspace, size_t ws_bytes, tfl_stream_t stream);
/* Backward of one sub-block (x_out = x_in + branch(x_in)): dx holds dL/dx_out on entry, dL/dx_in on exit; the
 * sub-block's parameter gradients are accumulated into their slices of `grads`.  models/mss_tflocoformer.py:443-462. */
int tfl_conv_swiglu_ffn_bwd(const tfl_plan* plan, const void* packed, const float* const* weights, int n_weights, int layer,
                            int axis, int ffn_index, const float* x_in, float* dx, int batch, int n_frames, int n_freq,
                            float* grads, void* workspace, size_t ws_bytes, tfl_stream_t stream);
int tfl_rope_attn_bwd(const tfl_plan* plan, const void* packed, const float* const* weights, int n_weights, int layer,
                      int axis, const float* x_in, float* dx, int batch, int n_frames, int n_freq, float* grads,
                      void* workspace, size_t ws_bytes, tfl_stream_t stream);
/* ---- autograd of the separators: a forward that keeps its activations, and its backward from an upstream gradient ----
 * Arithmetic = TFL_OPT_TRAIN_MODE, exactly as in tfl_train_forward_backward.  The workspace of one saved forward (sub-block
 * inputs x_0 .. x_n_sub plus the dx, scratch and weight-gradient buffers of the backward) must stay untouched between a
 * forward and its backward; a caller that keeps several forwards alive gives each its own workspace. */
size_t tfl_sep_train_workspace_bytes(const tfl_plan* plan, int batch, int n_frames, int n_freq);
/* TFLocoformerSeparator (plan with enc_in_ch == 2): spec [B, Tf, F, 2] -> est [B, S, Tf, F, 2]. */
int tfl_sep_train_forward(const tfl_plan* plan, const void* packed, const float* spec, int batch, int n_frames,
                          int n_freq, float* est, void* workspace, size_t ws_bytes, tfl_stream_t stream);
/* d_est [B, S, Tf, F, 2] (+ the forward's spec, packed image and workspace) -> grads (tfl_train_grad_layout,
 * overwritten).  `weights`: the raw fp32 device tensors tfl_pack_weights took.  No gradient for spec. */
int tfl_sep_train_backward(const tfl_plan* plan, const void* packed, const float* const* weights, int n_weights,
                           const float* d_est, const float* spec, int batch, int n_frames, int n_freq, float* grads,
                           void* workspace, size_t ws_bytes, tfl_stream_t stream);
/* tfl_sep_train_backward plus the input gradient d_spec [B, Tf, F, 2] (overwritten). */
int tfl_sep_train_backward_input(const tfl_plan* plan, const void* packed, const float* const* weights, int n_weights,
                                 const float* d_est, const float* spec, int batch, int n_frames, int n_freq, float* grads,
                                 void* workspace, size_t ws_bytes, tfl_stream_t stream, float* d_spec);
/* TFLocoformerMSS (plan with the STFT and enc_in_ch == 2, at most 4 sources, n_samples > n_fft/2).  The workspace holds
 * the saved forward, the spectrogram and the buffers of the mixture gradient; no loss buffers. */
size_t tfl_mss_train_workspace_bytes(const tfl_plan* plan, int batch, int n_samples);
/* mixture [B, T] -> audio [S, B, T] and / or est [B, S, Tf, F, 2] (either may be NULL). */
int tfl_mss_train_forward(const tfl_plan* plan, const void* packed, const float* mixture, int batch, int n_samples,
                          float* audio, float* est, void* workspace, size_t ws_bytes, tfl_stream_t stream);
/* Exactly one of d_audio [S, B, T] / d_est [B, S, Tf, F, 2] -> grads (tfl_train_grad_layout, overwritten) and, when
 * d_mixture is not NULL, d_mixture [B, T] (overwritten).  Same packed image and workspace as the forward. */
int tfl_mss_train_backward(const tfl_plan* plan, const void* packed, const float* const* weights, int n_weights,
                           const float* d_audio, const float* d_est, int batch, int n_samples, float* grads,
                           float* d_mixture, void* workspace, size_t ws_bytes, tfl_stream_t stream);
/* Blocks-only plan (enc_in_ch == 0): x_in [B, Tf, F, C] -> x_out (all Locoformer blocks); backward: dx_out -> dx_in and
 * grads (overwritten).  x_in / x_out and dx_out / dx_in may not overlap. */
int tfl_blocks_train_forward(const tfl_plan* plan, const void* packed, const float* x_in, int batch, int n_frames,
                             int n_freq, float* x_out, void* workspace, size_t ws_bytes, tfl_stream_t stream);
int tfl_blocks_train_backward(const tfl_plan* plan, const void* packed, const float* const* weights, int n_weights,
                              const float* dx_out, int batch, int n_frames, int n_freq, float* dx_in, float* grads,
                              void* workspace, size_t ws_bytes, tfl_stream_t stream);
/* torch.nn.utils.clip_grad_norm_ (train.py:141): norm_out[0] = total L2 norm, norm_out[1] = min(1, max_norm / (norm + 1e-6))
 * (device, 2 floats; no host sync).  scratch: >= 592 doubles. */
int tfl_grad_clip_norm(const float* grads, int64_t n, float max_norm, float* norm_out, double* scratch,
                       size_t scratch_bytes, tfl_stream_t stream);
/* acc = (overwrite ? 0 : acc) + scale * grads -- gradient accumulation over micro-batches (train.py:117-146, the
 * `loss / gradient_accumulation_steps` of the reference folded into `scale`). */
int tfl_grad_accumulate(float* acc, const float* grads, int64_t n, float scale, int overwrite, tfl_stream_t stream);
/* torch.optim.AdamW step `step` (1-based) over flat buffers (train.py:351-357); `clip` = norm_out above or NULL. */
int tfl_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, const float* clip,
                   float lr, float beta1, float beta2, float eps, float weight_decay, int step, tfl_stream_t stream);

/* Every mbarrier wait in the tcgen05 kernels is bounded (~2 s).  A wait that expires is a pipeline protocol error: the
 * kernel records {1, block, thread, shared-memory address of the barrier, parity} in a host-mapped record and traps, so
 * the launch fails loudly (cudaErrorLaunchFailed at the next synchronising call) and every later tfl_* entry point
 * returns an error naming the record.  This call copies the record to out5 (no device access) and optionally clears it. */
int tfl_debug_timeout(uint32_t* out5, int reset);

/* BandSplitModule.band_split, standalone/bslocoformer_separator.py:241-254.  spec [B, M, T, F, 2] -> x [B, T, nb, C].
 * `weights` is one fp32 buffer, `table` (device int64, 16 entries per band) its index:
 *   [0] first bin  [1] width  [2] gn.weight  [3] gn.bias  [4] conv.weight^T [K][C]  [5] conv.bias            (split)
 *   [6] gn.weight  [7] gn.bias  [8] W1^T [C][4C]  [9] b1  [10] W3^T [4C][4C]  [11] b3  [12] W4^T [4C][O]  [13] b4  (decode) */
int tfl_bs_band_split(const float* spec, int batch, int n_chan, int n_frames, int n_freq, int emb_dim, int n_bands,
                      int max_width, const int64_t* table, const float* weights, float* x, tfl_stream_t stream);
/* BandSplitModule.bandwise_decoding + complex mask, :256-270 and :175-182.
 * x [B, T, nb, C], spec [B, M, T, F, 2] -> est [B, S, M, T, F, 2] (= spec * mask when masking != 0). */
int tfl_bs_band_decode(const float* x, const float* spec, int batch, int n_chan, int n_frames, int n_freq, int emb_dim,
                       int n_bands, int n_src, const int64_t* table, const float* weights, float* est, int masking,
                       tfl_stream_t stream);

/* Backward of the two band stages (autograd of BSLocoformerSeparator), fp32 CUDA cores.  `d_weights` is laid out like
 * `weights` (same table offsets, the conv weights transposed as there); each call overwrites the entries of its stage.
 * Weight gradients are dense products over the B * T rows of a band, one CTA per output tile (deterministic).
 * workspace: >= tfl_bs_band_bwd_workspace_bytes. */
size_t tfl_bs_band_bwd_workspace_bytes(int batch, int n_chan, int n_frames, int n_freq, int emb_dim, int n_bands,
                                       int n_src, int max_width);
/* x [B, T, nb, C] (the decoder's input), spec, d_est [B, S, M, T, F, 2] -> dx [B, T, nb, C] and the gradients of table
 * entries 6..13 (GroupNorm w / b, W1^T / b1, W3^T / b3, W4^T / b4).  The forward is recomputed per (band, frame tile). */
int tfl_bs_band_decode_bwd(const float* x, const float* spec, const float* d_est, int batch, int n_chan, int n_frames,
                           int n_freq, int emb_dim, int n_bands, int n_src, int max_width, const int64_t* table,
                           const float* weights, int masking, float* dx, float* d_weights, void* workspace,
                           size_t ws_bytes, tfl_stream_t stream);
/* spec, dx [B, T, nb, C] (gradient of the band-split output) -> gradients of table entries 2..5 (GroupNorm(1, K_b) w / b,
 * conv^T / bias).  No input gradient. */
int tfl_bs_band_split_bwd(const float* spec, const float* dx, int batch, int n_chan, int n_frames, int n_freq, int emb_dim,
                          int n_bands, int max_width, const int64_t* table, const float* weights, float* d_weights,
                          void* workspace, size_t ws_bytes, tfl_stream_t stream);

/* Diagnostic: process-wide switches used for A/B measurements (not part of the reference-facing surface).
 *   TFL_OPT_ATTN_KERNEL  1 = attn_tc_kernel (P through shared memory), 2 = attn_tc2_kernel (P in TMEM; default)
 *   TFL_OPT_FFN_KERNEL   1 = ffn_tc_kernel (two tiles per CTA), 2 = ffn_tc2_kernel (cta_group::2, one tile per CTA of a
 *                        2-CTA cluster; default where the shape allows it)
 *   TFL_OPT_TAIL_KERNEL  1 = attn_tail_rows_kernel (CUDA cores), 2 = attn_tail_mma_kernel (mma.sync; default)
 *   TFL_OPT_PDL          1 = programmatic dependent launch of the bf16 kernels of a step, 0 = plain launches (default:
 *                        measured neutral, 97.8 vs 97.8 ms per step -- the persistent kernels leave no SM free to start on)
 *   TFL_OPT_TRAIN_MODE   arithmetic of the training entry points: 0 = exact fp32 on CUDA cores (gradient-parity mode);
 *                        1 = every GEMM as mma.sync tf32 operands with fp32 accumulation; 2 (default) = 1 + the FORWARD
 *                        pass of the sub-blocks on the bf16 tcgen05 kernels of the inference path (the reference trains
 *                        with `tf32: true` under bf16 autocast); the backward pass recomputes on the tf32 path
 *   TFL_OPT_DEC_KERNEL   bf16-mode decoder: 1 = dec_conv_mma_kernel (9-tap gather), 2 = dec_conv_scatter_kernel (every
 *                        input row read once, rolling output-frame accumulators in shared memory; default for
 *                        emb_dim in {32, 64, 96, 128})
 *   TFL_OPT_TRACE_BASE   first chunk / tile index the pipeline trace records (64 entries per event; default 0)
 *   TFL_OPT_DETERMINISTIC  1 = bitwise-reproducible training entry points: every reduction over rows of the backward pass
 *                        (weight-gradient GEMM splits, bias / gamma / decoder / encoder gradients, encoder statistics, loss
 *                        row sums) stores per-split or per-block partials that one kernel adds in index order, with grids
 *                        sized from the shapes alone (never the SM count), instead of fp32 / double atomics.  0 (default) =
 *                        atomics.  Read when a training call is made: the *_train_workspace_bytes queries add the partials
 *                        buffer only when it is 1, so the option must have the same value for the size query, a saved
 *                        forward and its backward.  The inference entry points are deterministic and ignore it.  The
 *                        Python layer sets it from torch.are_deterministic_algorithms_enabled(). */
enum { TFL_OPT_ATTN_KERNEL = 0, TFL_OPT_FFN_KERNEL = 1, TFL_OPT_TRACE_BASE = 2, TFL_OPT_TAIL_KERNEL = 3, TFL_OPT_PDL = 4,
       TFL_OPT_TRAIN_MODE = 5, TFL_OPT_DEC_KERNEL = 6, TFL_OPT_DETERMINISTIC = 7, TFL_OPT_COUNT = 8 };
int tfl_debug_set_option(int key, int value);

/* Diagnostic: install (or clear with NULL) a device buffer of >= 16 * 64 uint64 in which block 0 of the tcgen05 FFN
 * kernel records clock64() stamps of its pipeline events ([event * 64 + chunk index]). */
int tfl_debug_set_trace(void* device_buffer);

/* Diagnostic: exercises the tcgen05 plumbing of the bf16 path on one 128-row tile.
 * mode 0: D[128, N] = sum_{tap < taps} A[m + tap, :] . B[tap][n, :]   A [128 + taps - 1, Kd], B [taps, N, Kd]
 * mode 1: D[128, N] = A[m, :] . B[:, n]                               A [128, Kd], B [Kd, N] (N-contiguous)
 * mode 2: as mode 1 with A staged in TMEM (tcgen05.st) instead of shared memory; N <= 128, Kd <= 256
 * Operands are rounded to bf16, accumulation is fp32.  scratch: >= taps * N * Kd * 2 bytes.
 * mode 3: mode 0's row-shifted tap product in tcgen05 kind::tf32 through the tap-GEMM kernel of TFL_PRECISION_TF32's FFN
 *         (operands rounded to tf32 with cvt.rna, fp32 accumulation; Kd % 8 == 0).  scratch: >= taps * N * Kd * 4 bytes. */
int tfl_tc_selftest(const float* A, const float* B, float* D, void* scratch, int N, int Kd, int taps, int mode,
                    tfl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* TFL_H_ */
