// Host-callable launchers of the non-GEMM kernels (elementwise.cu, attention.cu, align.cu, vocoder_tail.cu).
// Everything is channel-last (b, t, c) unless a name says `cf` (channel-first, the reference's API layout).
#pragma once
#include "common.cuh"

namespace ev {

// ---- layout / glue -------------------------------------------------------------------------------------------
// out[b,t,c] = in[b,c,t] * scale (* mask)       OutT in {float, bf16}
template <typename OutT>
cudaError_t cf_to_cl(const float* in, int B, int C, int T, OutT* out, long long out_ld, long long out_bs, float scale,
                     RowMask mask, cudaStream_t s);
// out[b,c,t] = in[b,t,c] * mul + add
cudaError_t cl_to_cf(const float* in, long long in_ld, long long in_bs, int B, int C, int T, float* out, float mul,
                     float add, cudaStream_t s);
cudaError_t i64_to_i32(const long long* in, int* out, int n, cudaStream_t s);
// dst[i] = vals[i], i < n <= 32: tiny host->device constant upload that is CUDA-graph capturable
cudaError_t upload_floats(float* dst, const float* vals_host, int n, cudaStream_t s);
// dst[i] = words[i], i < n: host->device upload of a table of 32-bit words through kernel parameters (graph capturable, no
// pageable copy), kUploadWords words per launch
constexpr int kUploadWords = 960;
cudaError_t upload_words(void* dst, const void* words_host, int n, cudaStream_t s);

// ---- text encoder --------------------------------------------------------------------------------------------
// text_encoder.py:397: out[b,t,:] = emb[ids[b,t]] * scale, zero on padded rows
// ids outside [0, n_vocab) (valid rows only) are clamped for the lookup and reported as bit 0 of *flags (nullable):
// nn.Embedding raises IndexError there, and so does the python layer once it reads the flags
cudaError_t embed_tokens(const long long* ids, const float* emb, int B, int Tx, int C, int n_vocab, float scale,
                         RowMask mask, float* out, long long out_ld, long long* flags, cudaStream_t s);
// matcha_tts.py:118: out[b,:] = table[clamp(ids[b])]
cudaError_t embed_speakers(const long long* ids, const float* table, int B, int dim, int n_spks, float* out, long long* flags /* bit 1 */,
                           cudaStream_t s);
// text_encoder.py:402-403: buf[b,t,c0:c0+dim] = spk[b,:] (masked rows -> 0)
cudaError_t fill_speaker_channels(const float* spk, int B, int T, int dim, RowMask mask, float* buf, long long ld,
                                  int c0, cudaStream_t s);

// Channel LayerNorm of a row (text_encoder.py:15-33 with eps=1e-4; nn.LayerNorm with eps=1e-5, transformer.py:195,231):
//   y = LN(relu?(x + add?)) ; y = relu?(y) ; y *= mask  -> out_f32 and/or out_act
struct LnArgs {
  const float* x = nullptr; long long x_ld = 0;
  const float* add = nullptr; long long add_ld = 0;
  const float* gamma = nullptr; const float* beta = nullptr;
  float eps = 1e-5f;
  int pre_relu = 0, post_relu = 0;
  RowMask mask = {nullptr, 0};
  float* out_f32 = nullptr; long long f32_ld = 0;
  void* out_act = nullptr; long long act_ld = 0;
  void* split = nullptr;     // optional [rows][2C] fp16: the [hi | lo] halves of y * kF16ActScale, i.e. the pre-split operand of a
                             // following 3xFP16 conv (what split_f16_kernel would make of out_f32; saves that launch)
  int B = 0, T = 0, C = 0;   // rows are (b, t); row stride applies to b*T + t
};
template <typename ActT> cudaError_t layer_norm_rows(const LnArgs& a, cudaStream_t s);

// ---- attention (fp32 CUDA-core flash attention over channel-last q,k,v) -----------------------------------------
struct AttnArgs {
  const float* q = nullptr; const float* k = nullptr; const float* v = nullptr;  // (b, t, h*D + d), row stride ld
  long long ld = 0, bs = 0;
  int B = 0, T = 0, H = 0, D = 0;
  float scale = 1.0f;
  const int* lens = nullptr; int len_shift = 0;
  int mode = 0;            // 0: encoder (-1e4 fill where query or key is padded, text_encoder.py:241)
                           // 1: decoder (additive +1 on valid keys, diffusers float attn_mask, SURVEY H1)
  const float* rope_cos = nullptr; const float* rope_sin = nullptr; int rope_dim = 0;  // tables [t][rope_dim/2]
  void* out = nullptr; long long out_ld = 0, out_bs = 0;   // (b, t, h*D + d)
  void* split = nullptr;   // attention_enc_tc only: optional [B*T][2*H*D] fp16 [hi | lo] halves of out * kF16ActScale (see LnArgs::split)
};
template <typename ActT> cudaError_t attention_rows(const AttnArgs& a, cudaStream_t s);
// Text-encoder attention (mode 0, head width 96 or 128 with RoPE on half the head, T <= 384) on tcgen05 with 3xFP16 split operands, fp32 output
// (attention_enc_tc.cu); any other shape stays on attention_rows<float>.
bool attention_enc_tc_supported(const AttnArgs& a);
cudaError_t attention_enc_tc(const AttnArgs& a, cudaStream_t s);
// Decoder attention (mode 1 semantics) on tcgen05 tensor cores: bf16 q|k|v packed per row, head_dim 64 (attention_tc.cu)
struct AttnTcArgs {
  const bf16* qkv = nullptr; long long ld = 0, bs = 0;   // (b, t, [q | k | v]), each section `inner` wide, head h at h*64
  int B = 0, T = 0, H = 0, D = 64, inner = 0;
  float scale = 1.0f;
  const int* lens = nullptr; int len_shift = 0;
  bf16* out = nullptr; long long out_ld = 0, out_bs = 0;
  int skip_padded_queries = 0;   // 1: blocks of 128 queries that lie wholly in the padding are not computed (rows left unwritten)
};
cudaError_t attention_tc(const AttnTcArgs& a, cudaStream_t s, std::string* err);
cudaError_t rope_tables(float* cos_t, float* sin_t, int T, int rope_dim, float base, cudaStream_t s);

// ---- duration / alignment (integer, bit-exact) -------------------------------------------------------------------
// y_max (nullable): atomicMax of the lengths (zeroed by the caller) -- the one scalar the host reads back (utils/model.py:18)
// length_scales (device, B) or nullptr: item b's w_ceil = ceil(w) * length_scales[b], else * length_scale
cudaError_t durations(const float* logw, const int* x_lens, int B, int Tx, float length_scale, const float* length_scales,
                      float* w_ceil, long long* y_lengths, long long* y_max, cudaStream_t s);
cudaError_t row_sum_aten(const float* x, int B, int Tx, float* out, cudaStream_t s);
cudaError_t generate_path(const float* w_ceil, const int* x_lens, const int* y_lens, int B, int Tx, int T_pad,
                          float* attn, int* frame_token, cudaStream_t s);
cudaError_t gather_mu(const float* mu_x_cf, const int* frame_token, const int* y_lens, int B, int C, int Tx, int T_pad,
                      float* mu_y_cf, float* y_mask, cudaStream_t s);

// ---- decoder -----------------------------------------------------------------------------------------------------
// sinusoidal timestep embedding (decoder.py:14-29): out[s, :] for the n Euler times
cudaError_t time_sinusoid(const float* t_steps, int n, int dim, float* out, cudaStream_t s);
// xin[b,t,:] = [x0 | mu | spk] * mask ; x_state = x0 = z*temperature      (decoder.py:384-388, flow_matching.py:51)
// temperatures (device, B) or nullptr: item b's x0 = z * temperatures[b], else z * temperature
template <typename ActT>
cudaError_t decoder_pack_input(const float* z_cf, const float* mu_cf, const float* spk, int B, int F, int S, int T,
                               float temperature, const float* temperatures, RowMask mask, float* x_state, ActT* xin,
                               long long xin_ld, cudaStream_t s);
// GroupNorm statistics over (channels-in-group x ALL padded frames) per batch item (decoder.py:37, SURVEY H1)
cudaError_t group_norm_stats(const float* x, int B, int T, int C, int groups, double* partial, int* n_chunks_out,
                             cudaStream_t s);
struct GnApplyArgs {
  const float* x = nullptr;           // conv output (b,t,c), dense
  const double* partial = nullptr; int n_chunks = 0;
  const float* gamma = nullptr; const float* beta = nullptr; float eps = 1e-5f;
  int B = 0, T = 0, C = 0, groups = 8;
  RowMask mask = {nullptr, 0};
  const float* temb = nullptr;        // [C] added after Mish*mask (resnet block1), then masked again
  long long temb_bs = 0;              // item stride of temb (0: one time step for the whole batch; training draws one t per item)
  const float* res = nullptr; long long res_ld = 0;      // + res (resnet output = h + res_conv(x))
  float* out_f32 = nullptr; long long f32_ld = 0;        // y (after res)
  void* out_act = nullptr; long long act_ld = 0;         // y as next conv operand
  // optional fused LayerNorm of the fp32 result (pre-LN of the following transformer block)
  const float* ln_gamma = nullptr; const float* ln_beta = nullptr; void* out_ln = nullptr; long long ln_ld = 0;
};
template <typename ActT> cudaError_t group_norm_apply(const GnApplyArgs& a, cudaStream_t s);

// ---- vocoder tail ---------------------------------------------------------------------------------------------------
// hifigan/models.py:193-195 + to_waveform clamp: wav[b,t] = clamp(tanh(bias + sum_{j,c} w[j,c]*lrelu(x[b,t+j-3,c],0.01)))
// lens (device [B], frames) != nullptr: samples t >= lens[b]*hop are written as 0 without reading x (ragged batch)
cudaError_t conv_post_tanh(const float* x, int B, int L, int C, const float* w /*[7][C]*/, const float* bias, float* wav,
                           const int* lens, int hop, cudaStream_t s);

}  // namespace ev
