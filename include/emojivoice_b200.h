/*
 * emojivoice_b200 -- C ABI of the B200-native synthesis hot path.
 *
 * One shared library (libemojivoice_b200.so, sm_100a only) holds every CUDA kernel and the layer
 * orchestration of the path   MatchaTTS.synthesise(...) -> vocoder(mel) [-> denoiser]   of
 * rosielab/emojivoice.  The reference has no FFI for this path (it is plain PyTorch); the entry points below
 * are therefore cut at the python calls a maintainer would rebind, and each one names the reference
 * interface it replaces (paths relative to /root/reference/).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name ends in _host;
 *   - tensors use the reference's own layouts (channel-first, contiguous, fp32 / int64);
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); no entry point synchronises, allocates
 *     outputs, or spawns threads; scratch comes from the caller via the *_workspace_bytes() queries;
 *   - every function returns 0 on success or a negative ev_status; ev_last_error() gives the message;
 *     nothing throws across the boundary; a context is not re-entrant.
 *   - there is no CPU fallback: on a machine without an sm_100 device ev_create() fails.
 */
#ifndef EMOJIVOICE_B200_H
#define EMOJIVOICE_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define EV_API __attribute__((visibility("default")))
#else
#define EV_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ev_ctx ev_ctx;

typedef enum {
  EV_OK = 0,
  EV_ERR_INVALID = -1,   /* bad argument / unsupported configuration */
  EV_ERR_CUDA = -2,      /* a CUDA runtime or driver call failed */
  EV_ERR_MISSING = -3,   /* a required weight tensor was not supplied */
  EV_ERR_STATE = -4,     /* weights not loaded / workspace too small */
  EV_ERR_NO_DEVICE = -5  /* no sm_100 device */
} ev_status;

/* Arithmetic of the dense contractions in the decoder and vocoder (the text encoder and the duration /
 * alignment stage are always fp32 + integer so that durations stay bit-exact). */
typedef enum {
  EV_PREC_FP32 = 0, /* fp32 CUDA-core implicit GEMM, fixed summation order (parity mode, rel-L2 <= 1e-4) */
  EV_PREC_BF16 = 1  /* bf16 operands on tcgen05 tensor cores, fp32 TMEM accumulation, fp32 residual streams */
} ev_precision;

/* A named fp32 device tensor in the reference's state_dict layout (SURVEY.md 8a "weights contract"). */
typedef struct {
  const char* name;
  const float* data;
  int32_t ndim;
  int64_t shape[4];
} ev_tensor;

/* Hyper-parameters of MatchaTTS.__init__ (Matcha-TTS/matcha/models/matcha_tts.py:27-76,
 * configs/model/{matcha,encoder/default,decoder/default}.yaml). */
typedef struct {
  int32_t n_vocab, n_spks, spk_emb_dim, n_feats;
  int32_t enc_channels, enc_filter_channels, enc_filter_channels_dp, enc_heads, enc_layers, enc_kernel, enc_prenet;
  int32_t dec_channels, dec_heads, dec_head_dim, dec_mid_blocks;
  float mel_mean, mel_std;
} ev_matcha_cfg;

/* HiFi-GAN generator hyper-parameters (Matcha-TTS/matcha/hifigan/config.py:1-28). */
typedef struct {
  int32_t num_mels, upsample_initial_channel, n_ups, n_kernels;
  int32_t upsample_rates[8], upsample_kernel_sizes[8];
  int32_t resblock_kernel_sizes[4], resblock_dilation_sizes[4][3];
} ev_hifigan_cfg;

/* ---- lifetime -------------------------------------------------------------------------------------- */
EV_API int ev_create(ev_ctx** out, int device);
EV_API int ev_destroy(ev_ctx* ctx);
EV_API const char* ev_last_error(const ev_ctx* ctx); /* also valid with ctx == NULL (last creation error) */
EV_API int ev_version(void);

/* ---- weights ---------------------------------------------------------------------------------------
 * Replace MatchaTTS.load_state_dict / load_from_checkpoint (feel_me.py:156-159) and
 * Generator.load_state_dict + remove_weight_norm (feel_me.py:161-167, hifigan/models.py:199-206).
 * The library packs its own copies (kernel layouts, bf16 twins); the caller's tensors may be freed after
 * the call returns (the call synchronises `stream`). */
EV_API int ev_load_matcha(ev_ctx* ctx, const ev_tensor* weights, int n_weights, const ev_matcha_cfg* cfg, void* stream);
EV_API int ev_load_hifigan(ev_ctx* ctx, const ev_tensor* weights, int n_weights, const ev_hifigan_cfg* cfg, void* stream);

/* ---- text encoder + duration predictor + length stage ------------------------------------------------
 * Replaces matcha_tts.py:116-124: spk_emb lookup, TextEncoder.forward (text_encoder.py:378-410),
 * w = exp(logw)*mask, w_ceil = ceil(w)*length_scale, y_lengths = trunc(max(sum(w_ceil),1)).
 *   x (B,Tx) int64, x_lengths (B) int64, spks (B) int64 (ignored when n_spks == 1)
 *   out: spk_emb (B,spk_emb_dim), mu_x (B,n_feats,Tx), logw (B,1,Tx), w_ceil (B,1,Tx), y_lengths (B) int64
 *        summary (2) int64, nullable: [0] = max(y_lengths) -- the one scalar the host reads back to size the
 *        decoder (y_lengths.max(), utils/model.py:18); [1] = id-range flags (bit 0: a token id of a valid
 *        position outside [0, n_vocab); bit 1: a speaker id outside [0, n_spks)) -- nn.Embedding raises
 *        IndexError for those (matcha_tts.py:118, text_encoder.py:397); the library clamps and reports. */
EV_API size_t ev_encode_workspace_bytes(const ev_ctx* ctx, int B, int Tx);
EV_API int ev_encode(ev_ctx* ctx, const int64_t* x, const int64_t* x_lengths, const int64_t* spks, int B, int Tx,
              float length_scale, float* spk_emb, float* mu_x, float* logw, float* w_ceil, int64_t* y_lengths,
              int64_t* summary, void* workspace, size_t workspace_bytes, void* stream);
/* Per-item length scale: the same call with a speaking rate per utterance, length_scales (B) device fp32 (ev_encode is this
 * call with length_scale in every entry).  Item b's w_ceil and y_lengths are bit-identical to those of ev_encode on the same
 * batch with length_scale = length_scales[b]: the encoder does not read the length scale and the length stage is per row.
 * The values stay on the device (no host synchronisation, capturable): a finite, positive scale per item is the caller's
 * duty, as in the reference, which multiplies by whatever it is given.  Uses ev_encode_workspace_bytes. */
EV_API int ev_encode_items(ev_ctx* ctx, const int64_t* x, const int64_t* x_lengths, const int64_t* spks, int B, int Tx,
              const float* length_scales, float* spk_emb, float* mu_x, float* logw, float* w_ceil, int64_t* y_lengths,
              int64_t* summary, void* workspace, size_t workspace_bytes, void* stream);

/* ---- alignment / length regulator (integer, bit-exact) -----------------------------------------------
 * Replaces matcha_tts.py:129-135: sequence_mask, generate_path (utils/model.py:29-41) and
 * mu_y = attn^T mu_x (a gather).  T_pad = fix_len_compatibility(max y_lengths) is computed by the caller
 * (it fixes the output shapes; utils/model.py:14-20).
 *   out: attn (B,Tx,T_pad) 0/1 fp32, mu_y (B,n_feats,T_pad), y_mask (B,1,T_pad) */
EV_API size_t ev_align_workspace_bytes(const ev_ctx* ctx, int B, int Tx, int T_pad);
EV_API int ev_align(ev_ctx* ctx, const float* w_ceil, const int64_t* x_lengths, const int64_t* y_lengths,
             const float* mu_x, int B, int Tx, int T_pad, float* attn, float* mu_y, float* y_mask, void* workspace,
             size_t workspace_bytes, void* stream);

/* ---- flow-matching decoder -----------------------------------------------------------------------------
 * Replaces CFM.forward + solve_euler + Decoder.forward + denormalize (flow_matching.py:32-85,
 * decoder.py:363-443, utils/model.py:71-90): x0 = z*temperature, n_timesteps Euler steps of the U-Net
 * estimator on the padded extent T_pad (a multiple of 4), mel = x*mel_std + mel_mean.
 *   mu_y, z, out decoder_out, mel : (B,n_feats,T_pad);  spk_emb (B,spk_emb_dim) or NULL;  y_lengths (B) int64 */
EV_API size_t ev_decode_workspace_bytes(const ev_ctx* ctx, int B, int T_pad, int n_timesteps);
EV_API int ev_decode(ev_ctx* ctx, const float* mu_y, const int64_t* y_lengths, const float* z, const float* spk_emb,
              int B, int T_pad, int n_timesteps, float temperature, int precision, float* decoder_out,
              float* mel, void* workspace, size_t workspace_bytes, void* stream);
/* Per-item step count and temperature: item b takes n_steps_host[b] >= 1 Euler steps (host int32, B) from
 * x0 = z * temperatures[b] (device fp32, B).  Item b's decoder_out and mel are bit-identical to those of ev_decode on the same
 * batch (same mu_y, y_lengths, z, T_pad) called with (n_steps_host[b], temperatures[b]) for every item: items of a padded batch
 * interact only through T_pad (GroupNorm, attention and masks are per item).  Item b integrates on its own schedule
 * t_span = linspace(0, 1, n_b + 1); the call runs max n_b steps, and at steps k >= n_b item b's state is held by a select
 * (not by a zero step: x + 0*v would change -0.0 and turn an infinite v into NaN) while the item still passes through the
 * estimator.  Equal counts run the kernels and launches of ev_decode.  The step counts are read on the host; the
 * temperatures stay on the device (capturable).  Rejects a null pointer or n_b < 1 with EV_ERR_INVALID. */
EV_API size_t ev_decode_items_workspace_bytes(const ev_ctx* ctx, int B, int T_pad, int n_max);
EV_API int ev_decode_items(ev_ctx* ctx, const float* mu_y, const int64_t* y_lengths, const float* z, const float* spk_emb,
              int B, int T_pad, const int32_t* n_steps_host, const float* temperatures, int precision, float* decoder_out,
              float* mel, void* workspace, size_t workspace_bytes, void* stream);

/* ---- seeded prior noise ---------------------------------------------------------------------------------------
 * The z of flow_matching.py:51 (randn_like(mu), before the temperature) as a function of a seed per utterance:
 * seeds (B) device int64, read as uint64; z (B,n_feats,T) fp32.  Seed s keys Philox4x32-10 (Random123) with
 * k = (s mod 2^32, s >> 32); feature f and frame group q = t >> 2 give (w0,w1,w2,w3) = Philox(counter = (q, f, 0, 0), k), and
 *   u = (w0 + 0.5) 2^-32,  v = w1 2^-32,  z[f,4q] = sqrt(-2 ln u) cos(2 pi v),  z[f,4q+1] = sqrt(-2 ln u) sin(2 pi v),
 * with (w2, w3) giving frames 4q+2 and 4q+3 the same way; float64 arithmetic rounded once to fp32, |z| <= 6.77, never inf or NaN.
 * Row b depends on (seeds[b], f, t) only: not on B, T, the row's position or the other seeds, so frames [0, T) of a longer
 * call are those of a shorter one, bit for bit.  Any T >= 1; no weights needed; one launch; no host synchronisation
 * (capturable, a replay reads new seeds).  Null pointers or an empty shape: EV_ERR_INVALID. */
EV_API int ev_prior_noise(ev_ctx* ctx, const int64_t* seeds, int B, int n_feats, int T, float* z, void* stream);

/* ---- HiFi-GAN generator ----------------------------------------------------------------------------------
 * Replaces Generator.forward (hifigan/models.py:181-197) followed by the `.clamp(-1, 1)` of to_waveform
 * (feel_me.py:181-187; a no-op after tanh, kept for the contract).  mel (B,num_mels,T) -> wav (B,1,T*prod(rates)). */
EV_API size_t ev_vocode_workspace_bytes(const ev_ctx* ctx, int B, int T);
EV_API int ev_vocode(ev_ctx* ctx, const float* mel, int B, int T, int precision, float* wav, void* workspace,
              size_t workspace_bytes, void* stream);
/* Ragged batch: the same generator for a padded batch whose item b holds mel_lengths[b] valid frames (device int64, the
 * `mel_lengths` synthesise returns; NULL = ev_vocode).  Replaces the pair "vocoder(mel) on the padded batch, then crop
 * each waveform to [: length * hop]" of the reference's batched caller (Matcha-TTS/matcha/cli.py:291-317): wav[b] is
 * bit-identical to ev_vocode's on [0, mel_lengths[b]*hop) and ZERO beyond (the reference leaves vocoded prior noise there,
 * which every caller crops away).  The generator is convolutional with a finite receptive field, so time tiles that start
 * more than that field (computed per layer from the configuration) past an utterance's end are not computed at all. */
EV_API int ev_vocode_ragged(ev_ctx* ctx, const float* mel, const int64_t* mel_lengths, int B, int T, int precision,
              float* wav, void* workspace, size_t workspace_bytes, void* stream);

/* ---- bias denoiser -----------------------------------------------------------------------------------------
 * Replaces Denoiser.forward (hifigan/denoiser.py:58-64): centred hann STFT(1024, hop 256) -> magnitude minus
 * strength*bias_spec clamped at 0 -> inverse STFT with the original phase.  ev_denoiser_init computes
 * bias_spec = |STFT(vocoder(zeros(1,80,88)))|[:, :, 0] (denoiser.py:17-56) with the loaded generator.
 *   audio (B,L) -> out (B,L'), L' = hop*(L/hop) as torch.istft returns; bias_spec_out (n_fft/2+1) optional. */
EV_API size_t ev_denoise_workspace_bytes(const ev_ctx* ctx, int B, int L);
EV_API int ev_denoiser_init(ev_ctx* ctx, float* bias_spec_out, void* workspace, size_t workspace_bytes, void* stream);
EV_API int ev_denoise(ev_ctx* ctx, const float* audio, int B, int L, float strength, float* out, void* workspace,
               size_t workspace_bytes, void* stream);
/* Ragged batch: the same denoiser for a padded batch whose item b holds lengths[b] valid mel frames (device int64, samples
 * [0, lengths[b]*256); NULL = ev_denoise).  out[b] is bit-identical to ev_denoise's on [0, lengths[b]*256) and ZERO beyond.
 * Only the STFT frames those samples reach are transformed: frames f <= lengths[b] + 1, computed in pairs (f0, f0 + 1), f0
 * even, so at most floor((lengths[b] + 1) / 2) + 1 pairs per item.  Lengths are clamped to [0, L/256] on the device (a value
 * there cannot be checked without a host synchronisation).  Uses ev_denoise_workspace_bytes; B <= 2048. */
EV_API int ev_denoise_ragged(ev_ctx* ctx, const float* audio, const int64_t* lengths, int B, int L, float strength, float* out,
              void* workspace, size_t workspace_bytes, void* stream);

/* ---- vocoder + denoiser on a padded batch -------------------------------------------------------------------
 * Replaces the reference's reply path  audio = vocoder(mel).clamp(-1, 1); audio = denoiser(audio, strength)  (feel_me.py:181-187)
 * in the batched form of Matcha-TTS/matcha/cli.py:300,307-311, which then crops each waveform to [: length * 256].
 *   mel (B,num_mels,T), mel_lengths (B) device int64 (synthesise's mel_lengths) -> wav (B,1,T*256).
 * wav[b] is bit-identical to "ev_vocode, then ev_denoise" on [0, mel_lengths[b]*256) and ZERO beyond.  The generator runs as
 * ev_vocode_ragged on min(mel_lengths[b] + 4, T) frames (the denoised samples read no audio at or past (len + 4) * 256) and
 * the denoiser as ev_denoise_ragged on mel_lengths[b].  Needs ev_denoiser_init (EV_ERR_STATE before it); lengths are clamped
 * to [0, T] on the device; T >= 3, B <= 2048, a generator hop of 256.  No host synchronisation: capturable in a CUDA graph. */
EV_API size_t ev_to_waveform_ragged_workspace_bytes(const ev_ctx* ctx, int B, int T);
EV_API int ev_to_waveform_ragged(ev_ctx* ctx, const float* mel, const int64_t* mel_lengths, int B, int T, int precision,
              float strength, float* wav, void* workspace, size_t workspace_bytes, void* stream);

/* ---- vocoder + denoiser with a strength per item, or none -----------------------------------------------------
 * The same calls with a denoiser setting per utterance: strengths (B) device fp32, denoise (B) device uint8 (0 = item b is
 * not denoised; NULL = every item is).  Item b is, bit for bit,
 *   denoised:     what ev_to_waveform_ragged / ev_denoise_ragged give it on the same batch with strength = strengths[b];
 *   not denoised: ev_to_waveform_items: what ev_vocode_ragged gives it on the same batch and mel_lengths (the clamped generator
 *                 output); ev_denoise_items: its audio truncated to L' = 256*(L/256) samples.
 * Either way, on [0, lengths[b]*256) and ZERO beyond when lengths are given.  Strength 0 is not "not denoised": the STFT /
 * ISTFT round trip changes low bits.  A not-denoised item adds no STFT frames, and ev_to_waveform_items vocodes it on
 * mel_lengths[b] frames rather than mel_lengths[b] + 4.  Equal strengths with every item denoised are the scalar calls'
 * results; callers that hold equal values pass the number.  Strengths and flags stay on the device (no host
 * synchronisation, capturable; a finite strength is the caller's duty).  Other rules as the scalar calls. */
EV_API size_t ev_denoise_items_workspace_bytes(const ev_ctx* ctx, int B, int L);
EV_API int ev_denoise_items(ev_ctx* ctx, const float* audio, const int64_t* lengths, int B, int L, const float* strengths,
              const uint8_t* denoise, float* out, void* workspace, size_t workspace_bytes, void* stream);
EV_API size_t ev_to_waveform_items_workspace_bytes(const ev_ctx* ctx, int B, int T);
EV_API int ev_to_waveform_items(ev_ctx* ctx, const float* mel, const int64_t* mel_lengths, int B, int T, int precision,
              const float* strengths, const uint8_t* denoise, float* wav, void* workspace, size_t workspace_bytes, void* stream);

/* ---- monotonic alignment search (SURVEY 8 f4; training-side, the reference's only native component) ------------
 * replaces  maximum_path_c(paths, values, t_xs, t_ys, max_neg_val)   Matcha-TTS/matcha/utils/monotonic_align/core.pyx:42-47
 * (called through monotonic_align.maximum_path, __init__.py:7-22, from MatchaTTS.forward, models/matcha_tts.py:198).
 *   value (B,Tx,Ty) fp32 log-likelihoods (already multiplied by the mask, as __init__.py:13 does), t_xs / t_ys (B) int32
 *   valid extents -> path (B,Tx,Ty) int32 0/1, bit-identical to the Cython code.  `value` is NOT modified (the
 *   reference accumulates in a private copy).  As in the reference, t_ys[b] >= t_xs[b] is required. */
EV_API size_t ev_maximum_path_workspace_bytes(const ev_ctx* ctx, int B, int Tx, int Ty);
EV_API int ev_maximum_path(ev_ctx* ctx, const float* value, const int32_t* t_xs, const int32_t* t_ys, int B, int Tx, int Ty,
                    float max_neg_val, int32_t* path, void* workspace, size_t workspace_bytes, void* stream);

/* ---- training-side forward pass (SURVEY 8 f4): loss values, no backward ------------------------------------------
 * ev_estimator replaces ONE call of the flow-matching estimator  Decoder.forward(x, mask, mu, t, spks)
 * (Matcha-TTS/matcha/models/components/decoder.py:363-443) with a time per item, as CFM.compute_loss calls it
 * (components/flow_matching.py:114):  y, mu, out v : (B,n_feats,T_pad) channel-first, t (B) fp32, v = estimator(...) (masked).
 *
 * ev_train_forward replaces MatchaTTS.forward after the text encoder (models/matcha_tts.py:177-245) together with
 * CFM.compute_loss (flow_matching.py:87-118) and duration_loss (utils/model.py:44-46):
 *   mu_x (B,n_feats,Tx), logw (B,1,Tx) from ev_encode; y (B,n_feats,Ty) target mel; t_rand (B) and z (B,n_feats,Tc) are the
 *   reference's random draws (torch.rand / torch.randn_like, flow_matching.py:106-108), passed in so that runs can be compared;
 *   durations (B,Tx) or NULL = use_precomputed_durations (matcha_tts.py:185-186), else the alignment is searched (mas.cu);
 *   out_size > 0 cuts a segment of that many frames at out_offset[b] (int64, the reference draws it with random.choice,
 *   matcha_tts.py:211-233); Tc = out_size or Ty must be a multiple of 4.
 *   out: losses[3] = dur_loss, prior_loss, diff_loss (device fp32), attn (B,Tx,Tc) 0/1 fp32. */
EV_API size_t ev_estimator_workspace_bytes(const ev_ctx* ctx, int B, int T_pad);
EV_API int ev_estimator(ev_ctx* ctx, const float* y, const int64_t* y_lengths, const float* mu, const float* t, const float* spk_emb,
                 int B, int T_pad, int precision, float* v_out, void* workspace, size_t workspace_bytes, void* stream);
EV_API size_t ev_train_forward_workspace_bytes(const ev_ctx* ctx, int B, int Tx, int Ty, int out_size);
EV_API int ev_train_forward(ev_ctx* ctx, const float* mu_x, const float* logw, const int64_t* x_lengths, const float* y,
                     const int64_t* y_lengths, const float* spk_emb, const float* t_rand, const float* z, const float* durations,
                     int out_size, const int64_t* out_offset, int B, int Tx, int Ty, float sigma_min, int prior_loss, int precision,
                     float* losses, float* attn, void* workspace, size_t workspace_bytes, void* stream);

/* ---- bookkeeping the bench reads: kernels launched by this context since the last reset ------------------- */
EV_API int64_t ev_launch_count(const ev_ctx* ctx, int reset);

/* ---- per-kernel timing for roofline reports (CUDA events on the launching stream around every launch) ----------
 * ev_profile_begin switches recording on; ev_profile_end synchronises the device, aggregates per kernel class and
 * switches it off.  `flops` / `bytes` are the ALGORITHMIC work of the launches (valid, un-padded work only). */
typedef struct {
  char name[48];
  int64_t launches;
  double total_ms;
  double flops;
  double bytes;
} ev_kernel_stat;
EV_API int ev_profile_begin(ev_ctx* ctx);
EV_API int ev_profile_end(ev_ctx* ctx, ev_kernel_stat* out, int max_entries, int* n_out);

/* ---- unit-test hooks (one kernel each; used by tests/ through the same ABI) -------------------------------
 * conv1d: x (B,Cin,T) fp32, w (Cout,Cin,K) [or (Cin,Cout,K) when transposed!=0], bias (Cout) or NULL ->
 * y (B,Cout,Tout); same arithmetic path as the models use (precision selects CUDA-core fp32 / tcgen05 bf16). */
EV_API int ev_test_conv1d(ev_ctx* ctx, const float* x, const float* w, const float* bias, int B, int Cin, int T, int Cout,
                   int K, int stride, int padding, int dilation, int transposed, int precision, float* y,
                   void* stream);
/* Decoder self-attention alone (diffusers Attention as transformer.py:266-271 calls it: scale 1/8, float mask ADDED to the
 * logits, all T keys in the softmax).  qkv (B, 3*H*64, T) channel-first [q | k | v]; y_lengths (B) int64 or NULL; a key
 * t is "valid" (+1) while (t << len_shift) < y_lengths[b].  out (B, H*64, T).  precision: fp32 CUDA cores / bf16 tcgen05. */
EV_API int ev_test_attention(ev_ctx* ctx, const float* qkv, const int64_t* y_lengths, int B, int T, int H, int len_shift,
                      int precision, float* out, void* stream);
/* Text-encoder self-attention alone (MultiHeadAttention.attention, text_encoder.py:223-246: RoPE on the first half of each
 * 128-wide head, scores / sqrt(128), -1e4 where the query OR the key is padded).  qkv (B, T, 3*H*128) CHANNEL-LAST [q | k | v],
 * x_lengths (B) int64 or NULL, out (B, T, H*128).  impl 0: fp32 CUDA cores; 1: tcgen05 with 3xFP16 split operands (T <= 384).
 * repeat / avg_us_host as ev_test_ff_block. */
EV_API int ev_test_encoder_attention(ev_ctx* ctx, const float* qkv, const int64_t* x_lengths, int B, int T, int H, int impl,
                              float* out, int repeat, float* avg_us_host, void* stream);
/* The same at head width hd (RoPE on the first hd / 2 features, scores / sqrt(hd)): qkv (B, T, 3*H*hd), out (B, T, H*hd).
 * impl 0 takes hd = 64, 96 or 128, impl 1 hd = 96 or 128; any other pair is refused with EV_ERR_INVALID.
 * ev_test_encoder_attention is this call with hd = 128. */
EV_API int ev_test_encoder_attention_hd(ev_ctx* ctx, const float* qkv, const int64_t* x_lengths, int B, int T, int H, int hd,
                                 int impl, float* out, int repeat, float* avg_us_host, void* stream);
/* The float32 Euler times/steps of flow_matching.py:52,68-83 as the library computes them (pure host code). */
/* Fused LayerNorm + feed-forward of one decoder transformer block (transformer.py:296-316): x (B,T,256) CHANNEL-LAST,
 * w1 (inner,256), w2 (256,inner), snake_a = exp(alpha), snake_invb = 1/(exp(beta)+1e-9); out (B,T,256) channel-last,
 * out = (x + W2 snake(W1 LN(x) + b1) + b2) * mask, computed with bf16 tensor-core operands.  repeat > 0 and avg_us_host
 * != NULL: the launch is repeated and its average duration (us, CUDA events) written to the host float. */
EV_API int ev_test_ff_block(ev_ctx* ctx, const float* x, const float* ln_g, const float* ln_b, const float* w1, const float* b1,
              const float* snake_a, const float* snake_invb, const float* w2, const float* b2, const int64_t* y_lengths,
              int B, int T, int inner, int len_shift, float* out, int repeat, float* avg_us_host, void* stream);
/* ff_tc's attention tail mode alone (transformer.py:283-316): x = xr + att Wo^T + bo in front of the feed-forward above, one launch.
 * xr_cf (B,256,T) CHANNEL-FIRST fp32 residual stream, att (B,T,128) channel-last fp32 (rounded to bf16 inside), wo (256,128), bo (256);
 * the other arguments as ev_test_ff_block. */
EV_API int ev_test_tf_tail(ev_ctx* ctx, const float* xr_cf, const float* att, const float* wo, const float* bo, const float* ln_g,
              const float* ln_b, const float* w1, const float* b1, const float* snake_a, const float* snake_invb, const float* w2,
              const float* b2, const int64_t* y_lengths, int B, int T, int inner, int len_shift, float* out, int repeat,
              float* avg_us_host, void* stream);
/* Fused ResnetBlock1D + pre-LayerNorm of one decoder level (decoder.py:32-61, transformer.py:262; resnet_tc.cu) alone.
 * weights: ev_tensor list named conv1.weight (256,C_in,3), conv1.bias, gn1.weight, gn1.bias and, when full != 0, temb (256),
 * conv2.weight (256,256,3), conv2.bias, gn2.weight, gn2.bias, res.weight (256,C_in,1), res.bias, ln.weight, ln.bias.
 * x (B,C_in,T) channel-first fp32 (masked + rounded to bf16 inside); outputs (B,T,256) channel-last fp32:
 * out_a = (Mish(GN1(conv1 x)) m + temb) m, out_xr = Mish(GN2(conv2 a)) m + res(x), out_n = LayerNorm(out_xr);
 * full == 0: out_a = Mish(GN1(conv1 x)) m only (the decoder's final_block); full == 2: as 1, but the kernel writes the stream
 * channel-first (the layout ff_tc's tail mode reads; handed back channel-last).  repeat / avg_us_host as ev_test_ff_block. */
EV_API int ev_test_resnet_block(ev_ctx* ctx, const ev_tensor* weights, int n_weights, const float* x, const int64_t* y_lengths,
              int B, int T, int C_in, int len_shift, int full, float* out_a, float* out_xr, float* out_n, int repeat,
              float* avg_us_host, void* stream);
/* One HiFi-GAN ResBlock1 (hifigan/models.py:90-97, dilations 1, 3, 5) and its share of the multi-receptive-field mean
 * (:186-192), through the code the vocoder runs for each block.  weights: ev_tensor list named convs1.{0,1,2}.weight (C,C,k),
 * convs1.{0,1,2}.bias, convs2.{0,1,2}.weight, convs2.{0,1,2}.bias.  x (B,C,L) channel-first fp32; sum_in (B,L,C) fp32, read when
 * mode >= 1.  mode 0: sum = y; 1: sum = sum_in + y; 2: v = (sum_in + y) * inv_n, sum = v if write_f32 (else sum = sum_in),
 * act = lrelu(v, slope_out) if want_act.  lengths (B) int64 frames or NULL: a ragged batch as ev_vocode_ragged plans it (item b
 * needs rows [0, (lengths[b] + margin) * rows_per_frame)).  impl 0: six conv launches, 1: the fused kernel (resblock_tc.cu; bf16 only).
 * precision: EV_PREC_FP32 (impl 0 only) / EV_PREC_BF16.  schedule: NULL or int32[4] {EV_RB_CLUSTER, EV_RB_OCC2, EV_RB_WAVE,
 * EV_RB_RESIDENT} for this call, -1 = the environment's; a forced value the kernel cannot honour is EV_ERR_INVALID.
 * Outputs (B,L,C) channel-last fp32: sum, and act (bf16 widened; may be NULL).  A row the call does not write holds NaN (all bits
 * set); a write outside the B*L rows fails the call.  report: NULL or int32[9] of what the fused kernel launched: CTAs per cluster,
 * CTAs per SM, wavefront schedule, resident weights, weight ring slots, epilogue warps, grid, output rows per window, windows
 * (zeros for impl 0). */
EV_API int ev_test_resblock(ev_ctx* ctx, const ev_tensor* weights, int n_weights, int C, int k, const float* x, const float* sum_in,
              int B, int L, int mode, float inv_n, float slope_out, int write_f32, int want_act, const int64_t* lengths,
              int rows_per_frame, int margin, int impl, int precision, const int32_t* schedule, float* sum, float* act,
              int32_t* report, void* stream);
/* One tensor-core convolution (conv_tc.cu) with its fused epilogue, through the dispatch the models use (bf16 operands, or the
 * text encoder's split fp32 paths).  Every tensor is the caller's: outputs are written in place and nothing else is touched, so
 * the caller can surround them with guard rows and padding columns and check those afterwards.
 *   w (C_out,C_in,K) or, transposed, (C_in,C_out,K) fp32 and bias (C_out) fp32 or NULL: packed like every layer.
 *   precision 1: bf16 operands, x bf16; 2: 3xTF32, 3: 3xFP16 (C_in % 64 == 0), x fp32 dense (x_bs == T*x_ld); outputs fp32 only.
 *   x (B,T,C_in) channel-last at x + b*x_bs + t*x_ld + c.  res, res2, out_f32 fp32 and out_act bf16 (B,T_out,C_out) channel-last
 *   with their own ld / bs, each NULL when unused.  Per output element, on rows t < T_out (mask m = (t << len_shift) < lengths[b]):
 *     v = (acc + bias), 0 where !m if mask_pre;  v = v*alpha + res + res2;  v = v * (1/div)
 *     out_f32 = v, or a if f32_is_act;  out_act = bf16(a);  a = act(v), 0 where !m if mask_act
 *   act 0 identity, 1 ReLU, 2 LeakyReLU(slope), 4 SnakeBeta with snake_a = exp(alpha_c), snake_invb = 1/(exp(beta_c) + 1e-9).
 *   gn_sum (B,gn_groups,2) fp64 or NULL: the sum and sum of squares of out_f32 per 32-channel group are added in.
 *   lengths (B) int64 or NULL = no mask.  ragged_lengths (B) int64 frames or NULL: a compact tile list as ev_vocode_ragged plans it
 *   (rows [0, (ragged_lengths[b] + ragged_margin) * rows_per_frame) are needed; precision 1 only).
 *   schedule_host: NULL or int32[8] {lean, mb, ctas_per_sm, epi_warps, resident, bk32, halo, share}, -1 = the environment's
 *   EV_TC_* choice; a forced choice the launch cannot honour is EV_ERR_INVALID.  report_host: NULL or int32[19] of what ran: BN,
 *   m-blocks, CTAs per SM, epilogue warps, MMA issuers, resident weights, activation / weight ring slots, K-chunk width, halo reuse,
 *   TMA boxes per activation tile, lean epilogue, vector epilogue, split mode (0 bf16, 1 3xTF32, 2 3xFP16), accumulation groups
 *   per tile, operand sharing, compact tile list, grid, tiles.  Synchronises `stream`. */
typedef struct {
  int32_t B, C_in, T, C_out, K, stride, pad, dilation, transposed, precision;
  const float* w;
  const float* bias;
  const void* x;
  int64_t x_ld, x_bs;
  const float* res;
  int64_t res_ld, res_bs;
  const float* res2;
  int64_t res2_ld, res2_bs;
  float* out_f32;
  int64_t f32_ld, f32_bs;
  void* out_act;
  int64_t act_ld, act_bs;
  double* gn_sum;
  const int64_t* lengths;
  const float* snake_a;
  const float* snake_invb;
  int32_t gn_groups, len_shift, mask_pre, mask_act, act, f32_is_act;
  float slope, alpha, div;
  int32_t ragged_margin, rows_per_frame;
  const int64_t* ragged_lengths;
  const int32_t* schedule_host;
  int32_t* report_host;
} ev_conv_epilogue_test;
EV_API int ev_test_conv_epilogue(ev_ctx* ctx, const ev_conv_epilogue_test* args, void* stream);
/* EV_RN_TRACE=1: clock64 stamps [32] of CTA 0 of the most recent fused ResNet-block launch (host buffer). */
EV_API int ev_test_resnet_trace(ev_ctx* ctx, uint64_t* out_host, int n);
/* Host-only: how many mel frames past an utterance's end ev_vocode_ragged still computes in front of conv_pre (pre), of
 * upsampler i (up[i]) and inside stage i (stage[i]), i < n_ups -- upper bounds of the generator's look-ahead. */
EV_API int ev_test_vocoder_margins(const ev_hifigan_cfg* cfg, int32_t* stage, int32_t* up, int32_t* pre);
EV_API int ev_test_euler_schedule(int n_timesteps, float* t_host, float* dt_host);
/* The tables ev_decode_items uses for mixed step counts, (max n) x B row-major each (pure host code): row k of item b is step k
 * of ev_test_euler_schedule(n_b); past its last step an item repeats its last time with a zero step. */
EV_API int ev_test_euler_tables(const int32_t* n_steps_host, int B, float* t_host, float* dt_host);
/* y_lengths of torch.sum order: sums (B,Tx) fp32 rows exactly as ATen's CPU float32 reduction does. */
EV_API int ev_test_row_sum(ev_ctx* ctx, const float* x, int B, int Tx, float* out, void* stream);
/* Diagnostic (EV_TC_TRACE=1): clock64 stamps [CTA][16] of the most recent tensor-core conv launch's pipeline milestones
 * (0 entry, 1 prologue done, 2 after griddepcontrol.wait, 3 first TMA issued, 4 first operands landed, 5 first tile's MMAs
 * committed, 6 last commit, 7 first accumulator seen by the epilogue, 8 first tile stored, 9 last tile stored, 10 exit,
 * 11 %globaltimer at entry); synchronises the device.  scripts/conv_trace.py prints the medians. */
/* EV_FF_DEBUG & 16: clock64 stamps [192] of the first tile of CTA 0 of the most recent ff_tc launch (host buffer). */
EV_API int ev_test_ff_trace(ev_ctx* ctx, uint64_t* out_host, int n);
EV_API int ev_test_conv_trace(ev_ctx* ctx, uint64_t* out_host, int n);

#ifdef __cplusplus
}
#endif
#endif /* EMOJIVOICE_B200_H */
