// Matcha-TTS inference graph on the GPU: weight loading, text encoder + duration stage, alignment, and the
// flow-matching U-Net decoder integrated with Euler steps.  Layer order follows the reference exactly
// (text_encoder.py:378-410, matcha_tts.py:116-143, flow_matching.py:55-85, decoder.py:363-443); see DESIGN.md for
// the buffer plan.  All intermediate tensors are channel-last and live in the caller's workspace.
#include <algorithm>
#include <cmath>
#include <cstdlib>

#include "ctx.cuh"

using namespace ev;

namespace {

cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// ------------------------------------------------------------------------------------------------ loading
int load_resnet(ev_ctx* ctx, WeightStore& ws, const std::string& p, int c_in, int c, int td, ResnetW* r) {
  r->c_in = c_in;
  EV_TRY(make_conv(ctx, ws, {p + ".block1.block.0.weight"}, {p + ".block1.block.0.bias"}, c, c_in, 3, 1, 1, 1, CONV_NORMAL, TC_BF16, &r->conv1));
  EV_TRY(make_conv(ctx, ws, {p + ".block2.block.0.weight"}, {p + ".block2.block.0.bias"}, c, c, 3, 1, 1, 1, CONV_NORMAL, TC_BF16, &r->conv2));
  EV_TRY(make_conv(ctx, ws, {p + ".res_conv.weight"}, {p + ".res_conv.bias"}, c, c_in, 1, 1, 0, 1, CONV_NORMAL, TC_BF16, &r->res));
  EV_TRY(ws.copy_vec(p + ".block1.block.1.weight", c, &r->gn1_g));
  EV_TRY(ws.copy_vec(p + ".block1.block.1.bias", c, &r->gn1_b));
  EV_TRY(ws.copy_vec(p + ".block2.block.1.weight", c, &r->gn2_g));
  EV_TRY(ws.copy_vec(p + ".block2.block.1.bias", c, &r->gn2_b));
  (void)td;
  return 0;
}

__global__ void snake_prep_kernel(const float* alpha, const float* beta, int n, float* ea, float* invb) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    ea[i] = expf(alpha[i]);                           // transformer.py:72-73 (log-scale parameters)
    invb[i] = 1.0f / (expf(beta[i]) + 0.000000001f);  // transformer.py:78
  }
}

int load_transformer(ev_ctx* ctx, WeightStore& ws, const std::string& p, int c, int inner, TransformerW* t) {
  EV_TRY(ws.copy_vec(p + ".norm1.weight", c, &t->ln1_g));
  EV_TRY(ws.copy_vec(p + ".norm1.bias", c, &t->ln1_b));
  EV_TRY(ws.copy_vec(p + ".norm3.weight", c, &t->ln3_g));
  EV_TRY(ws.copy_vec(p + ".norm3.bias", c, &t->ln3_b));
  EV_TRY(make_conv(ctx, ws, {p + ".attn1.to_q.weight", p + ".attn1.to_k.weight", p + ".attn1.to_v.weight"}, {}, inner, c, 1, 1, 0, 1, CONV_NORMAL, TC_BF16, &t->qkv));
  EV_TRY(make_conv(ctx, ws, {p + ".attn1.to_out.0.weight"}, {p + ".attn1.to_out.0.bias"}, c, inner, 1, 1, 0, 1, CONV_NORMAL, TC_BF16, &t->out));
  EV_TRY(make_conv(ctx, ws, {p + ".ff.net.0.proj.weight"}, {p + ".ff.net.0.proj.bias"}, 4 * c, c, 1, 1, 0, 1, CONV_NORMAL, TC_BF16, &t->ff1));
  EV_TRY(make_conv(ctx, ws, {p + ".ff.net.2.weight"}, {p + ".ff.net.2.bias"}, c, 4 * c, 1, 1, 0, 1, CONV_NORMAL, TC_BF16, &t->ff2));
  const ev_tensor* al = ws.get(p + ".ff.net.0.alpha", {4LL * c});
  const ev_tensor* be = ws.get(p + ".ff.net.0.beta", {4LL * c});
  if (!al || !be) return EV_ERR_MISSING;
  void* q;
  EV_TRY(device_alloc(ctx, (size_t)4 * c * sizeof(float), &q, false, ws.stream));
  t->snake_a = reinterpret_cast<float*>(q);
  EV_TRY(device_alloc(ctx, (size_t)4 * c * sizeof(float), &q, false, ws.stream));
  t->snake_invb = reinterpret_cast<float*>(q);
  snake_prep_kernel<<<ceil_div(4 * c, 256), 256, 0, ws.stream>>>(al->data, be->data, 4 * c, t->snake_a, t->snake_invb);
  EV_CUDA(ctx, cudaGetLastError());
  return 0;
}

constexpr int kRopeMaxT = 4096;

}  // namespace

extern "C" int ev_load_matcha(ev_ctx* ctx, const ev_tensor* weights, int n_weights, const ev_matcha_cfg* cfg, void* stream) {
  if (!ctx || !weights || !cfg) return EV_ERR_INVALID;
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  if (ctx->matcha.loaded) return fail(ctx, EV_ERR_STATE, "matcha weights already loaded in this context");
  const ev_matcha_cfg& c = *cfg;
  const int H = c.enc_channels + (c.n_spks > 1 ? c.spk_emb_dim : 0);
  const int D = c.dec_channels;
  const int inner = c.dec_heads * c.dec_head_dim;
  const int dec_in = 2 * c.n_feats + (c.n_spks > 1 ? c.spk_emb_dim : 0);
  // head widths with an encoder attention kernel (attention.cu; 96 and 128 also attention_enc_tc.cu)
  if (c.enc_heads <= 0 || H % c.enc_heads || (H / c.enc_heads != 64 && H / c.enc_heads != 96 && H / c.enc_heads != 128))
    return fail(ctx, EV_ERR_INVALID, "text-encoder head width must be 64, 96 or 128");
  if (c.dec_head_dim != 64 || D % 32 || D > 256 || (D / 8) > 32 || c.dec_mid_blocks != 2)
    return fail(ctx, EV_ERR_INVALID, "decoder must be the (c,c) U-Net with head_dim 64, <=256 channels, 2 mid blocks");
  if ((c.enc_channels & 3) || (H & 3) || (dec_in & 7) || (c.n_feats & 7) || c.enc_kernel > kMaxTaps)
    return fail(ctx, EV_ERR_INVALID, "channel counts must be multiples of 8");
  MatchaW& m = ctx->matcha;
  m.cfg = c;
  WeightStore ws(ctx, weights, n_weights, s);
  if (c.n_spks > 1) EV_TRY(ws.copy_vec("spk_emb.weight", (long long)c.n_spks * c.spk_emb_dim, &m.spk_table));
  EV_TRY(ws.copy_vec("encoder.emb.weight", (long long)c.n_vocab * c.enc_channels, &m.tok_emb));
  const int C = c.enc_channels;
  if (c.enc_prenet) {
    for (int i = 0; i < 3; ++i) {
      const std::string p = "encoder.prenet.conv_layers." + std::to_string(i), n = "encoder.prenet.norm_layers." + std::to_string(i);
      EV_TRY(make_conv(ctx, ws, {p + ".weight"}, {p + ".bias"}, C, C, 5, 1, 2, 1, CONV_NORMAL, TC_TF32X3, &m.pre_conv[i]));
      EV_TRY(ws.copy_vec(n + ".gamma", C, &m.pre_g[i]));
      EV_TRY(ws.copy_vec(n + ".beta", C, &m.pre_b[i]));
    }
    EV_TRY(make_conv(ctx, ws, {"encoder.prenet.proj.weight"}, {"encoder.prenet.proj.bias"}, C, C, 1, 1, 0, 1, CONV_NORMAL, TC_TF32X3, &m.pre_proj));
  }
  m.enc.resize(c.enc_layers);
  const int ek = c.enc_kernel;
  for (int i = 0; i < c.enc_layers; ++i) {
    EncLayerW& L = m.enc[i];
    const std::string a = "encoder.encoder.attn_layers." + std::to_string(i), f = "encoder.encoder.ffn_layers." + std::to_string(i);
    EV_TRY(make_conv(ctx, ws, {a + ".conv_q.weight", a + ".conv_k.weight", a + ".conv_v.weight"},
                     {a + ".conv_q.bias", a + ".conv_k.bias", a + ".conv_v.bias"}, H, H, 1, 1, 0, 1, CONV_NORMAL, TC_TF32X3, &L.qkv));
    EV_TRY(make_conv(ctx, ws, {a + ".conv_o.weight"}, {a + ".conv_o.bias"}, H, H, 1, 1, 0, 1, CONV_NORMAL, TC_TF32X3, &L.o));
    EV_TRY(make_conv(ctx, ws, {f + ".conv_1.weight"}, {f + ".conv_1.bias"}, c.enc_filter_channels, H, ek, 1, ek / 2, 1, CONV_NORMAL, TC_TF32X3, &L.ffn1));
    EV_TRY(make_conv(ctx, ws, {f + ".conv_2.weight"}, {f + ".conv_2.bias"}, H, c.enc_filter_channels, ek, 1, ek / 2, 1, CONV_NORMAL, TC_TF32X3, &L.ffn2));
    EV_TRY(ws.copy_vec("encoder.encoder.norm_layers_1." + std::to_string(i) + ".gamma", H, &L.ln1_g));
    EV_TRY(ws.copy_vec("encoder.encoder.norm_layers_1." + std::to_string(i) + ".beta", H, &L.ln1_b));
    EV_TRY(ws.copy_vec("encoder.encoder.norm_layers_2." + std::to_string(i) + ".gamma", H, &L.ln2_g));
    EV_TRY(ws.copy_vec("encoder.encoder.norm_layers_2." + std::to_string(i) + ".beta", H, &L.ln2_b));
  }
  EV_TRY(make_conv(ctx, ws, {"encoder.proj_m.weight"}, {"encoder.proj_m.bias"}, c.n_feats, H, 1, 1, 0, 1, CONV_NORMAL, TC_TF32X3, &m.proj_m));
  const int Fd = c.enc_filter_channels_dp;
  EV_TRY(make_conv(ctx, ws, {"encoder.proj_w.conv_1.weight"}, {"encoder.proj_w.conv_1.bias"}, Fd, H, 3, 1, 1, 1, CONV_NORMAL, TC_TF32X3, &m.dp_conv1));
  EV_TRY(make_conv(ctx, ws, {"encoder.proj_w.conv_2.weight"}, {"encoder.proj_w.conv_2.bias"}, Fd, Fd, 3, 1, 1, 1, CONV_NORMAL, TC_TF32X3, &m.dp_conv2));
  EV_TRY(make_conv(ctx, ws, {"encoder.proj_w.proj.weight"}, {"encoder.proj_w.proj.bias"}, 1, Fd, 1, 1, 0, 1, CONV_NORMAL, TC_NONE, &m.dp_proj));
  EV_TRY(ws.copy_vec("encoder.proj_w.norm_1.gamma", Fd, &m.dp_g1));
  EV_TRY(ws.copy_vec("encoder.proj_w.norm_1.beta", Fd, &m.dp_b1));
  EV_TRY(ws.copy_vec("encoder.proj_w.norm_2.gamma", Fd, &m.dp_g2));
  EV_TRY(ws.copy_vec("encoder.proj_w.norm_2.beta", Fd, &m.dp_b2));
  // RoPE tables: rotary width = half of a head (text_encoder.py:203-204)
  {
    const int rope_dim = (H / c.enc_heads) / 2;
    void* p;
    EV_TRY(device_alloc(ctx, (size_t)kRopeMaxT * (rope_dim / 2) * sizeof(float), &p, false, s));
    m.rope_cos = reinterpret_cast<float*>(p);
    EV_TRY(device_alloc(ctx, (size_t)kRopeMaxT * (rope_dim / 2) * sizeof(float), &p, false, s));
    m.rope_sin = reinterpret_cast<float*>(p);
    m.rope_T = kRopeMaxT;
    EV_CUDA(ctx, rope_tables(m.rope_cos, m.rope_sin, kRopeMaxT, rope_dim, 10000.0f, s));
  }
  // ---- estimator
  const std::string E = "decoder.estimator.";
  const int TD = 4 * D;
  EV_TRY(make_conv(ctx, ws, {E + "time_mlp.linear_1.weight"}, {E + "time_mlp.linear_1.bias"}, TD, dec_in, 1, 1, 0, 1, CONV_NORMAL, TC_NONE, &m.time1));
  EV_TRY(make_conv(ctx, ws, {E + "time_mlp.linear_2.weight"}, {E + "time_mlp.linear_2.bias"}, TD, TD, 1, 1, 0, 1, CONV_NORMAL, TC_NONE, &m.time2));
  const std::string rn_names[6] = {E + "down_blocks.0.0", E + "down_blocks.1.0", E + "mid_blocks.0.0", E + "mid_blocks.1.0",
                                   E + "up_blocks.0.0", E + "up_blocks.1.0"};
  const std::string tf_names[6] = {E + "down_blocks.0.1.0", E + "down_blocks.1.1.0", E + "mid_blocks.0.1.0",
                                   E + "mid_blocks.1.1.0", E + "up_blocks.0.1.0", E + "up_blocks.1.1.0"};
  const int rn_cin[6] = {dec_in, D, D, D, 2 * D, 2 * D};
  std::vector<std::string> mlp_w, mlp_b;
  for (int i = 0; i < 6; ++i) {
    EV_TRY(load_resnet(ctx, ws, rn_names[i], rn_cin[i], D, TD, &m.rn[i]));
    EV_TRY(load_transformer(ctx, ws, tf_names[i], D, inner, &m.tf[i]));
    mlp_w.push_back(rn_names[i] + ".mlp.1.weight");
    mlp_b.push_back(rn_names[i] + ".mlp.1.bias");
  }
  EV_TRY(make_conv(ctx, ws, mlp_w, mlp_b, D, TD, 1, 1, 0, 1, CONV_NORMAL, TC_NONE, &m.temb_proj));
  EV_TRY(make_conv(ctx, ws, {E + "down_blocks.0.2.conv.weight"}, {E + "down_blocks.0.2.conv.bias"}, D, D, 3, 2, 1, 1, CONV_NORMAL, TC_BF16, &m.down0));
  EV_TRY(make_conv(ctx, ws, {E + "down_blocks.1.2.weight"}, {E + "down_blocks.1.2.bias"}, D, D, 3, 1, 1, 1, CONV_NORMAL, TC_BF16, &m.down1_conv));
  EV_TRY(make_conv(ctx, ws, {E + "up_blocks.0.2.conv.weight"}, {E + "up_blocks.0.2.conv.bias"}, D, D, 4, 2, 1, 1, CONV_TRANSPOSED, TC_BF16, &m.up0));
  EV_TRY(make_conv(ctx, ws, {E + "up_blocks.1.2.weight"}, {E + "up_blocks.1.2.bias"}, D, D, 3, 1, 1, 1, CONV_NORMAL, TC_BF16, &m.up1_conv));
  EV_TRY(make_conv(ctx, ws, {E + "final_block.block.0.weight"}, {E + "final_block.block.0.bias"}, D, D, 3, 1, 1, 1, CONV_NORMAL, TC_BF16, &m.final_conv));
  EV_TRY(ws.copy_vec(E + "final_block.block.1.weight", D, &m.final_g));
  EV_TRY(ws.copy_vec(E + "final_block.block.1.bias", D, &m.final_b));
  EV_TRY(make_conv(ctx, ws, {E + "final_proj.weight"}, {E + "final_proj.bias"}, c.n_feats, D, 1, 1, 0, 1, CONV_NORMAL, TC_BF16, &m.final_proj));
  EV_CUDA(ctx, cudaStreamSynchronize(s));
  m.loaded = true;
  return 0;
}

// ================================================================================================ encoder
namespace {

struct EncBuffers {
  int* xlen32; float* h0; float* pa; float* pb; float* tmp; float* X; float* X1; float* qkv; float* att; float* F;
  float* mu_cl; float* D1; float* D2;
  float* split;   // [rows][2 * widest C_in]: the [hi | lo] operand of the 3xTF32 tensor-core convs
};

void plan_encode(const ev_matcha_cfg& c, int B, int Tx, Workspace& w, EncBuffers* e) {
  const size_t R = (size_t)B * Tx;
  const int H = c.enc_channels + (c.n_spks > 1 ? c.spk_emb_dim : 0);
  const int wide = std::max(std::max(H, c.enc_channels), c.enc_filter_channels_dp);
  e->xlen32 = w.take<int>(B);
  e->h0 = w.take<float>(R * c.enc_channels);
  e->pa = w.take<float>(R * c.enc_channels);
  e->pb = w.take<float>(R * c.enc_channels);
  e->tmp = w.take<float>(R * wide);
  e->X = w.take<float>(R * H);
  e->X1 = w.take<float>(R * H);
  e->qkv = w.take<float>(R * 3 * H);
  e->att = w.take<float>(R * H);
  e->F = w.take<float>(R * c.enc_filter_channels);
  e->mu_cl = w.take<float>(R * c.n_feats);
  e->D1 = w.take<float>(R * c.enc_filter_channels_dp);
  e->D2 = w.take<float>(R * c.enc_filter_channels_dp);
  e->split = w.take<float>(R * 2 * std::max(std::max(H, c.enc_filter_channels), c.enc_filter_channels_dp));
}

}  // namespace

extern "C" size_t ev_encode_workspace_bytes(const ev_ctx* ctx, int B, int Tx) {
  if (!ctx || !ctx->matcha.loaded || B <= 0 || Tx <= 0) return 0;
  Workspace w(nullptr, 0);
  EncBuffers e;
  plan_encode(ctx->matcha.cfg, B, Tx, w, &e);
  return w.off + 256;
}

extern "C" int ev_encode(ev_ctx* ctx, const int64_t* x, const int64_t* x_lengths, const int64_t* spks, int B, int Tx,
                         float length_scale, float* spk_emb, float* mu_x, float* logw, float* w_ceil, int64_t* y_lengths,
                         int64_t* summary, void* workspace, size_t workspace_bytes, void* stream) {
  if (!ctx) return EV_ERR_INVALID;
  if (!ctx->matcha.loaded) return fail(ctx, EV_ERR_STATE, "ev_encode: matcha weights not loaded");
  if (!x || !x_lengths || !mu_x || !logw || !w_ceil || !y_lengths || B <= 0 || Tx <= 0)
    return fail(ctx, EV_ERR_INVALID, "ev_encode: null argument or empty batch");
  const MatchaW& m = ctx->matcha;
  const ev_matcha_cfg& c = m.cfg;
  if (c.n_spks > 1 && (!spks || !spk_emb)) return fail(ctx, EV_ERR_INVALID, "ev_encode: multi-speaker model needs spks and spk_emb");
  if (Tx > m.rope_T) return fail(ctx, EV_ERR_INVALID, "ev_encode: text longer than the RoPE table (4096 tokens)");
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  Workspace w(workspace, workspace_bytes);
  EncBuffers e;
  plan_encode(c, B, Tx, w, &e);
  if (w.overflow || !workspace) return fail(ctx, EV_ERR_STATE, "ev_encode: workspace too small");
  ctx->prof_tag = "/enc";
  const int C = c.enc_channels, H = C + (c.n_spks > 1 ? c.spk_emb_dim : 0);
  const long long bsC = (long long)Tx * C, bsH = (long long)Tx * H;
  const double R = (double)B * Tx;
  EV_LAUNCH(ctx, s, "i64_to_i32", 0, 12.0 * B, i64_to_i32(reinterpret_cast<const long long*>(x_lengths), e.xlen32, B, s));
  const RowMask mask{e.xlen32, 0};
  long long* summ = reinterpret_cast<long long*>(summary);      // [0] max(y_lengths), [1] id-range flags
  if (summ) EV_CUDA(ctx, cudaMemsetAsync(summ, 0, 2 * sizeof(long long), s));
  if (c.n_spks > 1)
    EV_LAUNCH(ctx, s, "embed_speakers", 0, 8.0 * B * c.spk_emb_dim,
              embed_speakers(reinterpret_cast<const long long*>(spks), m.spk_table, B, c.spk_emb_dim, c.n_spks, spk_emb, summ ? summ + 1 : nullptr, s));
  EV_LAUNCH(ctx, s, "embed_tokens", 0, R * (8 + 8.0 * C),
            embed_tokens(reinterpret_cast<const long long*>(x), m.tok_emb, B, Tx, C, c.n_vocab, sqrtf((float)C), mask, e.h0, C, summ ? summ + 1 : nullptr, s));
  // Producers write the next 3xFP16 conv's [hi | lo] operand themselves (LayerNorm, the tcgen05 attention): 25 split launches less
  const bool ps = enc_split_f16() && ctx->enc_tc;
  if (c.enc_prenet) {
    // ConvReluNorm (text_encoder.py:60-67): 3 x [conv5(x*mask) -> LN -> ReLU], 1x1 proj, + x_org, * mask
    const float* cur = e.h0;
    float* pp[2] = {e.pa, e.pb};
    for (int i = 0; i < 3; ++i) {
      Epilogue ep;
      ep.out_f32 = e.tmp; ep.f32_ld = C; ep.f32_bs = bsC;
      EV_TRY(run_conv_tf32(ctx, m.pre_conv[i], cur, C, bsC, B, Tx, ep, e.split, s, ps && i > 0));
      LnArgs ln;
      ln.x = e.tmp; ln.x_ld = C; ln.gamma = m.pre_g[i]; ln.beta = m.pre_b[i]; ln.eps = 1e-4f; ln.post_relu = 1; ln.mask = mask;
      ln.out_f32 = pp[i & 1]; ln.f32_ld = C; ln.B = B; ln.T = Tx; ln.C = C; ln.split = ps ? e.split : nullptr;
      EV_LAUNCH(ctx, s, "layer_norm", 0, R * C * 8.0, layer_norm_rows<float>(ln, s));
      cur = pp[i & 1];
    }
    Epilogue ep;
    ep.res = e.h0; ep.res_ld = C; ep.res_bs = bsC;
    ep.out_act = e.X; ep.act_ld = H; ep.act_bs = bsH; ep.mask = mask; ep.mask_act = 1;
    EV_TRY(run_conv_tf32(ctx, m.pre_proj, cur, C, bsC, B, Tx, ep, e.split, s, ps));
  } else {
    EV_CUDA(ctx, cudaMemcpy2DAsync(e.X, (size_t)H * 4, e.h0, (size_t)C * 4, (size_t)C * 4, (size_t)B * Tx, cudaMemcpyDeviceToDevice, s));
  }
  if (c.n_spks > 1) {
    EV_LAUNCH(ctx, s, "fill_speaker", 0, R * c.spk_emb_dim * 4.0, fill_speaker_channels(spk_emb, B, Tx, c.spk_emb_dim, mask, e.X, H, C, s));
  }
  // Encoder (text_encoder.py:314-325), post-LN blocks.  Every stream is kept masked: padded rows never reach a valid
  // row (conv inputs are masked, padded keys get -1e4), so zeroing them early changes nothing that is observable.
  const int hd = H / c.enc_heads;
  for (int i = 0; i < c.enc_layers; ++i) {
    const EncLayerW& L = m.enc[i];
    Epilogue ep;
    ep.out_f32 = e.qkv; ep.f32_ld = 3 * H; ep.f32_bs = (long long)Tx * 3 * H;
    // 1x1 convs without a mask in the epilogue see the batch as ONE sequence of B*Tx rows (the tensors are dense): 128-row
    // tiles then straddle utterances instead of leaving every utterance's last tile mostly empty (Tx = 177: 45 m-tiles, not 64).
    // Row-wise the arithmetic is unchanged, so the results are bit-identical.
    EV_TRY(run_conv_tf32(ctx, L.qkv, e.X, H, bsH * B, 1, B * Tx, ep, e.split, s, ps && i > 0));
    AttnArgs at;
    at.q = e.qkv; at.k = e.qkv + H; at.v = e.qkv + 2 * H; at.ld = 3 * H; at.bs = (long long)Tx * 3 * H;
    at.B = B; at.T = Tx; at.H = c.enc_heads; at.D = hd; at.scale = 1.0f / sqrtf((float)hd);
    at.lens = e.xlen32; at.len_shift = 0; at.mode = 0;
    at.rope_cos = m.rope_cos; at.rope_sin = m.rope_sin; at.rope_dim = hd / 2;
    at.out = e.att; at.out_ld = H; at.out_bs = bsH;
    // tcgen05 with split fp16 operands where the shape allows (head width 96 or 128; EV_ENC_ATTN=f32 keeps the CUDA-core
    // kernel); both are fp32-accurate
    static const bool enc_attn_tc = []() { const char* v = getenv("EV_ENC_ATTN"); return !(v && std::string(v) == "f32"); }();
    const bool att_tc = enc_attn_tc && attention_enc_tc_supported(at);
    if (att_tc) at.split = ps ? e.split : nullptr;
    if (att_tc)   // 3 products per contraction
      EV_LAUNCH(ctx, s, "attention_enc_tc", 3.0 * 4.0 * B * c.enc_heads * (double)Tx * Tx * hd, R * H * 16.0, attention_enc_tc(at, s));
    else
      EV_LAUNCH(ctx, s, "attention_enc_f32", 4.0 * B * c.enc_heads * (double)Tx * Tx * hd, R * H * 16.0, attention_rows<float>(at, s));
    Epilogue eo;  // x + y
    eo.res = e.X; eo.res_ld = H; eo.res_bs = bsH; eo.out_f32 = e.tmp; eo.f32_ld = H; eo.f32_bs = bsH;
    EV_TRY(run_conv_tf32(ctx, L.o, e.att, H, bsH * B, 1, B * Tx, eo, e.split, s, ps && att_tc));
    LnArgs l1;
    l1.x = e.tmp; l1.x_ld = H; l1.gamma = L.ln1_g; l1.beta = L.ln1_b; l1.eps = 1e-4f; l1.mask = mask;
    l1.out_f32 = e.X1; l1.f32_ld = H; l1.B = B; l1.T = Tx; l1.C = H; l1.split = ps ? e.split : nullptr;
    EV_LAUNCH(ctx, s, "layer_norm", 0, R * H * 8.0, layer_norm_rows<float>(l1, s));
    Epilogue e1;  // relu(conv_1(x*mask)) * mask
    e1.act = ACT_RELU; e1.mask = mask; e1.mask_act = 1;
    e1.out_act = e.F; e1.act_ld = c.enc_filter_channels; e1.act_bs = (long long)Tx * c.enc_filter_channels;
    EV_TRY(run_conv_tf32(ctx, L.ffn1, e.X1, H, bsH, B, Tx, e1, e.split, s, ps));
    Epilogue e2;  // x + conv_2(..)*mask
    e2.mask = mask; e2.mask_pre = 1; e2.res = e.X1; e2.res_ld = H; e2.res_bs = bsH;
    e2.out_f32 = e.tmp; e2.f32_ld = H; e2.f32_bs = bsH;
    EV_TRY(run_conv_tf32(ctx, L.ffn2, e.F, c.enc_filter_channels, (long long)Tx * c.enc_filter_channels, B, Tx, e2, e.split, s));
    LnArgs l2 = l1;
    l2.gamma = L.ln2_g; l2.beta = L.ln2_b; l2.out_f32 = e.X;
    EV_LAUNCH(ctx, s, "layer_norm", 0, R * H * 8.0, layer_norm_rows<float>(l2, s));
  }
  {  // mu = proj_m(x) * mask  (text_encoder.py:405) -> channel-first output
    Epilogue ep;
    ep.mask = mask; ep.mask_pre = 1; ep.out_f32 = e.mu_cl; ep.f32_ld = c.n_feats; ep.f32_bs = (long long)Tx * c.n_feats;
    EV_TRY(run_conv_tf32(ctx, m.proj_m, e.X, H, bsH, B, Tx, ep, e.split, s, ps && c.enc_layers > 0));
    EV_LAUNCH(ctx, s, "cl_to_cf", 0, R * c.n_feats * 8.0, cl_to_cf(e.mu_cl, c.n_feats, (long long)Tx * c.n_feats, B, c.n_feats, Tx, mu_x, 1.0f, 0.0f, s));
  }
  {  // DurationPredictor (text_encoder.py:84-94): conv -> relu -> LN (x2), 1x1 proj, masks in between
    const int Fd = c.enc_filter_channels_dp;
    const long long bsF = (long long)Tx * Fd;
    Epilogue ep;
    ep.out_f32 = e.tmp; ep.f32_ld = Fd; ep.f32_bs = bsF;
    EV_TRY(run_conv_tf32(ctx, m.dp_conv1, e.X, H, bsH, B, Tx, ep, e.split, s, ps && c.enc_layers > 0));   // the operand proj_m used
    LnArgs ln;
    ln.x = e.tmp; ln.x_ld = Fd; ln.pre_relu = 1; ln.gamma = m.dp_g1; ln.beta = m.dp_b1; ln.eps = 1e-4f; ln.mask = mask;
    ln.out_f32 = e.D1; ln.f32_ld = Fd; ln.B = B; ln.T = Tx; ln.C = Fd; ln.split = ps ? e.split : nullptr;
    EV_LAUNCH(ctx, s, "layer_norm", 0, R * Fd * 8.0, layer_norm_rows<float>(ln, s));
    EV_TRY(run_conv_tf32(ctx, m.dp_conv2, e.D1, Fd, bsF, B, Tx, ep, e.split, s, ps));
    ln.gamma = m.dp_g2; ln.beta = m.dp_b2; ln.out_f32 = e.D2; ln.split = nullptr;
    EV_LAUNCH(ctx, s, "layer_norm", 0, R * Fd * 8.0, layer_norm_rows<float>(ln, s));
    Epilogue el;
    el.mask = mask; el.mask_pre = 1; el.out_f32 = logw; el.f32_ld = 1; el.f32_bs = Tx;
    EV_TRY(run_conv_tf32(ctx, m.dp_proj, e.D2, Fd, bsF, B, Tx, el, e.split, s));
    EV_LAUNCH(ctx, s, "durations", 0, R * 8.0, durations(logw, e.xlen32, B, Tx, length_scale, w_ceil, reinterpret_cast<long long*>(y_lengths), summ, s));
  }
  return 0;
}

// ================================================================================================ alignment
extern "C" size_t ev_align_workspace_bytes(const ev_ctx* ctx, int B, int Tx, int T_pad) {
  if (!ctx || B <= 0 || Tx <= 0 || T_pad <= 0) return 0;
  return align_up(((size_t)2 * B + (size_t)B * T_pad) * sizeof(int), 256) + 256;   // lengths as int32 + frame->token map
}

extern "C" int ev_align(ev_ctx* ctx, const float* w_ceil, const int64_t* x_lengths, const int64_t* y_lengths,
                        const float* mu_x, int B, int Tx, int T_pad, float* attn, float* mu_y, float* y_mask,
                        void* workspace, size_t workspace_bytes, void* stream) {
  if (!ctx) return EV_ERR_INVALID;
  if (!ctx->matcha.loaded) return fail(ctx, EV_ERR_STATE, "ev_align: matcha weights not loaded");
  if (!w_ceil || !x_lengths || !y_lengths || !mu_x || !attn || !mu_y || !y_mask || B <= 0 || Tx <= 0 || T_pad <= 0)
    return fail(ctx, EV_ERR_INVALID, "ev_align: null argument or empty shape");
  if (!workspace || workspace_bytes < ev_align_workspace_bytes(ctx, B, Tx, T_pad) - 256)
    return fail(ctx, EV_ERR_STATE, "ev_align: workspace too small");
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  int* scratch = reinterpret_cast<int*>(workspace);
  int* xl = scratch; int* yl = scratch + B; int* tok = scratch + 2 * B;
  const int Fm = ctx->matcha.cfg.n_feats;
  EV_LAUNCH(ctx, s, "i64_to_i32", 0, 12.0 * B, i64_to_i32(reinterpret_cast<const long long*>(x_lengths), xl, B, s));
  EV_LAUNCH(ctx, s, "i64_to_i32", 0, 12.0 * B, i64_to_i32(reinterpret_cast<const long long*>(y_lengths), yl, B, s));
  EV_LAUNCH(ctx, s, "generate_path", 0, 4.0 * B * (double)Tx * T_pad, generate_path(w_ceil, xl, yl, B, Tx, T_pad, attn, tok, s));
  EV_LAUNCH(ctx, s, "gather_mu", 0, 8.0 * B * (double)Fm * T_pad, gather_mu(mu_x, tok, yl, B, Fm, Tx, T_pad, mu_y, y_mask, s));
  return 0;
}

// ================================================================================================ decoder
namespace {

template <typename ActT>
struct DecBuffers {
  int* ylen32; float* t_steps; float* sinus; float* th1; float* th2; float* tproj;
  float* xstate; ActT* xin; ActT* cat0; ActT* cat1; ActT* din;
  float* h; float* r; float* xr; ActT* a; ActT* n; float* qkv; ActT* att; ActT* ff; double* gn_partial;
  double* gn_fused; size_t gn_fused_count;   // [n_steps][13][B][8][2] sums written by the conv epilogues (bf16 path)
  int* ff_tiles[2];                          // compact lists of the 128-row tiles with a valid row, at T and T/2 (ff_tc.cu)
  int* rag_arena; size_t rag_ints;           // tile lists of the convs whose padded output rows nobody reads (out-projection)
};

template <typename ActT>
void plan_decode(const ev_matcha_cfg& c, int B, int T, int n_steps, Workspace& w, DecBuffers<ActT>* d) {
  const size_t R = (size_t)B * T, R2 = (size_t)B * (T / 2);
  const int D = c.dec_channels, inner = c.dec_heads * c.dec_head_dim;
  const int dec_in = 2 * c.n_feats + (c.n_spks > 1 ? c.spk_emb_dim : 0);
  d->ylen32 = w.take<int>(B);
  d->t_steps = w.take<float>(n_steps);
  d->sinus = w.take<float>((size_t)n_steps * dec_in);
  d->th1 = w.take<float>((size_t)n_steps * 4 * D);
  d->th2 = w.take<float>((size_t)n_steps * 4 * D);
  d->tproj = w.take<float>((size_t)n_steps * 6 * D);
  d->xstate = w.take<float>(R * c.n_feats);
  d->xin = w.take<ActT>(R * dec_in);
  d->cat0 = w.take<ActT>(R * 2 * D);
  d->cat1 = w.take<ActT>(R2 * 2 * D);
  d->din = w.take<ActT>(R2 * D);
  d->h = w.take<float>(R * D);
  d->r = w.take<float>(R * D);
  d->xr = w.take<float>(R * D);
  d->a = w.take<ActT>(R * D);
  d->n = w.take<ActT>(R * D);
  d->qkv = w.take<float>(R * 3 * inner);
  d->att = w.take<ActT>(R * inner);
  d->ff = w.take<ActT>(R * 4 * D);
  d->gn_partial = w.take<double>((size_t)B * ceil_div(T, 32) * 8 * 2);
  d->gn_fused_count = (size_t)n_steps * 13 * B * 8 * 2;
  d->gn_fused = w.take<double>(d->gn_fused_count);
  d->ff_tiles[0] = w.take<int>((size_t)B * ceil_div(T, 128) + 64);
  d->ff_tiles[1] = w.take<int>((size_t)B * ceil_div(T / 2, 128) + 64);
  d->rag_ints = (size_t)8 * ((size_t)B * ceil_div(T, 128) + 64);
  d->rag_arena = w.take<int>(d->rag_ints);
}

// Fixed-step Euler times exactly as flow_matching.py:52,68-83 computes them in float32 (t_span = linspace(0,1,n+1),
// t += dt, dt = t_span[k+1] - t).  torch.linspace(float32): step=(end-start)/(steps-1); the first half counts up from
// `start`, the second half counts down from `end`.
void euler_schedule(int n, std::vector<float>* t_of_step, std::vector<float>* dt_of_step) {
  std::vector<float> span(n + 1);
  const int steps = n + 1;
  volatile float step = 1.0f / (float)(steps - 1);
  const int halfway = steps / 2;
  for (int i = 0; i < steps; ++i) {
    // ATen's CPU kernel evaluates both halves as one fused multiply-add (verified against torch.linspace for
    // n in {1,2,4,10,50}: tests/test_host_logic.py)
    if (i < halfway) span[i] = std::fmaf(step, (float)i, 0.0f);
    else span[i] = std::fmaf(-step, (float)(steps - i - 1), 1.0f);
  }
  volatile float t = span[0];
  volatile float dt = span[1] - span[0];
  t_of_step->resize(n);
  dt_of_step->resize(n);
  for (int k = 1; k <= n; ++k) {
    (*t_of_step)[k - 1] = t;
    (*dt_of_step)[k - 1] = dt;
    t = t + dt;
    if (k < n) dt = span[k + 1] - t;
  }
}

template <typename ActT>
struct Decoder {
  ev_ctx* ctx; const MatchaW& m; DecBuffers<ActT>& d; int B, T; cudaStream_t s; int D, inner;
  int gn_slot = 0;   // next free [B][8][2] slot of d.gn_fused
  bool xr_is_cf = false;       // d.xr of the current block holds the residual stream channel-first (written by resnet_tc for ff_tc's tail mode)
  bool qkv_done = false;       // the fused ResNet kernel of the current block has already written q|k|v (bf16) into d.qkv
  bool use_ff_tiles = false;   // d.ff_tiles hold this call's tile lists
  RaggedPlanner rag;           // planner state (table cache) of this call's ragged convs
  cudaStream_t side_stream = nullptr;   // side branch for res_conv (single-lane decoding), see resnet()
  cudaEvent_t temb_event = nullptr;     // time embeddings are produced on another side branch: waited for at their first use
  long long temb_bs = 0;                // item stride of the time embeddings (0: one t for the batch; ev_estimator: one t per item)
  bool estimator_only = false;          // ev_estimator: the final projection writes v * mask instead of the Euler update
  // GroupNorm statistics: fused into the producing conv's epilogue on the tensor-core path (32 channels per group),
  // a separate reduction kernel otherwise.  Returns the (partial, n_chunks) pair gn_apply reads.
  bool fuse_gn() const { return std::is_same<ActT, bf16>::value && D == 256; }
  double* next_gn_slot() { double* p = d.gn_fused + (size_t)(gn_slot++) * B * 8 * 2; return p; }
  // One launch for the whole ResNet block + pre-LN (resnet_tc.cu) when every tile of the level fits one co-resident wave
  // ff_tc's attention tail mode (out-projection + residual + LayerNorm3 + feed-forward in one launch) reads the residual stream
  // channel-first: it is used when the block's ResNet half is the fused kernel, which can write it that way
  bool fuse_tail(int k) const {
    if constexpr (!std::is_same<ActT, bf16>::value) return false;
    static const bool on = []() { const char* v = getenv("EV_TAIL_FUSE"); return !(v && atoi(v) == 0); }();
    static const int dbg_skip = []() { const char* v = getenv("EV_DEC_DEBUG_SKIP"); return v ? atoi(v) : 0; }();
    const TransformerW& w = m.tf[k];
    return on && D == 256 && inner == 128 && !dbg_skip && ff_tc_supported(w.ff1, w.ff2) && ff_tc_oproj_supported(w.out);
  }
  bool fuse_resnet(const ResnetW& w, int Tl) const {
    if constexpr (!std::is_same<ActT, bf16>::value) return false;
    return D == 256 && resnet_tc_supported(w.conv1, &w.conv2, &w.res, B, Tl);
  }
  int launch_resnet_tc(const ResnetTcArgs& ra, double flops, double bytes, const char* name) {
    std::string err;
    cudaError_t ce;
    { LaunchScope ls(ctx, s, name, flops, bytes); ce = resnet_tc_launch(ra, s, &err); }
    if (ce != cudaSuccess) return err.empty() ? cuda_fail(ctx, ce, name) : fail(ctx, EV_ERR_CUDA, err);
    return 0;
  }

  // ResnetBlock1D (decoder.py:46-61) followed by the pre-LN of the transformer block; in: masked operand tensor
  int resnet(int k, const ActT* in, long long in_ld, int Tl, int shift, const float* temb) {
    const ResnetW& w = m.rn[k];
    const RowMask mask{d.ylen32, shift};
    const long long bsD = (long long)Tl * D, in_bs = (long long)Tl * in_ld;
    if constexpr (std::is_same<ActT, bf16>::value) {
      if (fuse_resnet(w, Tl)) {
        if (temb_event) { EV_CUDA(ctx, cudaStreamWaitEvent(s, temb_event, 0)); temb_event = nullptr; }
        ResnetTcArgs ra;
        ra.x = in; ra.x_ld = in_ld; ra.x_bs = in_bs;
        ra.conv1 = &w.conv1; ra.conv2 = &w.conv2; ra.res = &w.res;
        ra.gn_g1 = w.gn1_g; ra.gn_b1 = w.gn1_b; ra.gn_g2 = w.gn2_g; ra.gn_b2 = w.gn2_b; ra.temb = temb; ra.temb_bs = temb_bs;
        ra.ln_g = m.tf[k].ln1_g; ra.ln_b = m.tf[k].ln1_b;
        ra.lens = d.ylen32; ra.len_shift = shift; ra.B = B; ra.T = Tl;
        ra.n_out = d.n;                      // conv2's operand stays in shared memory
        xr_is_cf = fuse_tail(k);
        if (xr_is_cf) ra.xr_cf = d.xr; else ra.xr = d.xr;
        qkv_done = xr_is_cf && resnet_tc_qkv_supported(m.tf[k].qkv);    // the q|k|v projection of the block's attention rides along
        if (qkv_done) { ra.qkv = &m.tf[k].qkv; ra.qkv_out = reinterpret_cast<bf16*>(d.qkv); ra.n_out = nullptr; }
        const double rows = (double)B * Tl;
        return launch_resnet_tc(ra, 2.0 * rows * D * (4.0 * w.c_in + 3.0 * D + (qkv_done ? 3.0 * inner : 0.0)),
                                rows * (2.0 * w.c_in + 6.0 * D + (qkv_done ? 6.0 * inner - 2.0 * D : 0.0)), "resnet_tc");
      }
    }
    xr_is_cf = false;
    qkv_done = false;
    Epilogue e1; e1.out_f32 = d.h; e1.f32_ld = D; e1.f32_bs = bsD;
    const double* part = d.gn_partial;
    if (fuse_gn()) { e1.gn_sum = next_gn_slot(); e1.gn_groups = 8; part = e1.gn_sum; }
    // res_conv(x * mask) depends only on the block's input: it runs as a side branch (a parallel branch of a captured graph),
    // filling the SMs that conv1 -> GroupNorm -> conv2 leave idle, and is joined before the residual add
    const bool side = side_stream != nullptr && !ctx->profiling;
    cudaStream_t sr = side ? side_stream : s;
    if (side) {
      EV_CUDA(ctx, cudaEventRecord(ctx->side_fork, s));
      EV_CUDA(ctx, cudaStreamWaitEvent(sr, ctx->side_fork, 0));
    }
    {
      Epilogue er; er.out_f32 = d.r; er.f32_ld = D; er.f32_bs = bsD;
      EV_TRY(run_conv<ActT>(ctx, w.res, in, in_ld, in_bs, B, Tl, er, sr));
    }
    if (side) EV_CUDA(ctx, cudaEventRecord(ctx->side_join, sr));
    EV_TRY(run_conv<ActT>(ctx, w.conv1, in, in_ld, in_bs, B, Tl, e1, s));
    int chunks = 1;
    const double RD = (double)B * Tl * D;
    if (!fuse_gn()) EV_LAUNCH(ctx, s, "gn_stats", 0, RD * 4.0, group_norm_stats(d.h, B, Tl, D, 8, d.gn_partial, &chunks, s));
    GnApplyArgs g1;
    g1.x = d.h; g1.partial = part; g1.n_chunks = chunks; g1.gamma = w.gn1_g; g1.beta = w.gn1_b;
    g1.B = B; g1.T = Tl; g1.C = D; g1.mask = mask; g1.temb = temb; g1.temb_bs = temb_bs; g1.out_act = d.a; g1.act_ld = D;
    static const int dbg_skip = []() { const char* v = getenv("EV_DEC_DEBUG_SKIP"); return v ? atoi(v) : 0; }();
    if (temb_event) { EV_CUDA(ctx, cudaStreamWaitEvent(s, temb_event, 0)); temb_event = nullptr; }
    if (!(dbg_skip & 8)) EV_LAUNCH(ctx, s, "gn_apply", 0, RD * (4.0 + sizeof(ActT)), group_norm_apply<ActT>(g1, s));
    if (fuse_gn()) { e1.gn_sum = next_gn_slot(); part = e1.gn_sum; }
    EV_TRY(run_conv<ActT>(ctx, w.conv2, d.a, D, bsD, B, Tl, e1, s));
    if (side) EV_CUDA(ctx, cudaStreamWaitEvent(s, ctx->side_join, 0));      // r is needed from here on
    if (!fuse_gn()) EV_LAUNCH(ctx, s, "gn_stats", 0, RD * 4.0, group_norm_stats(d.h, B, Tl, D, 8, d.gn_partial, &chunks, s));
    GnApplyArgs g2;
    g2.x = d.h; g2.partial = part; g2.n_chunks = chunks; g2.gamma = w.gn2_g; g2.beta = w.gn2_b;
    g2.B = B; g2.T = Tl; g2.C = D; g2.mask = mask; g2.res = d.r; g2.res_ld = D; g2.out_f32 = d.xr; g2.f32_ld = D;
    g2.ln_gamma = m.tf[k].ln1_g; g2.ln_beta = m.tf[k].ln1_b; g2.out_ln = d.n; g2.ln_ld = D;
    EV_LAUNCH(ctx, s, "gn_apply_ln", 0, RD * (12.0 + sizeof(ActT)), group_norm_apply<ActT>(g2, s));
    return 0;
  }

  // BasicTransformerBlock (transformer.py:243-316); expects d.xr (stream) and d.n = LN1(xr); writes x*mask to `out`
  int transformer(int k, int Tl, int shift, ActT* out, long long out_ld) {
    const TransformerW& w = m.tf[k];
    static const int dbg_skip = []() { const char* v = getenv("EV_DEC_DEBUG_SKIP"); return v ? atoi(v) : 0; }();   // timing experiments only (wrong results)
    const RowMask mask{d.ylen32, shift};
    const long long bsD = (long long)Tl * D;
    const int Hh = m.cfg.dec_heads, hd = m.cfg.dec_head_dim;
    const double attn_flops = 4.0 * B * Hh * (double)Tl * Tl * hd;
    // rows that the skips below leave unwritten are only safe behind the fused feed-forward, which masks with selects and
    // zero-fills the tiles it does not compute; the unfused fallback (D != 256) computes every row
    const bool ff_fused = std::is_same<ActT, bf16>::value && D == 256 && !(dbg_skip & 3) && ff_tc_supported(w.ff1, w.ff2);
    if constexpr (std::is_same<ActT, bf16>::value) {
      // bf16 q|k|v straight from the projection epilogue -> tcgen05 attention (attention_tc.cu)
      bf16* qkv16 = reinterpret_cast<bf16*>(d.qkv);
      if (!qkv_done) {
        Epilogue eq; eq.out_act = qkv16; eq.act_ld = 3 * inner; eq.act_bs = (long long)Tl * 3 * inner;
        EV_TRY(run_conv<ActT>(ctx, w.qkv, d.n, D, bsD, B, Tl, eq, s));
      }
      AttnTcArgs at;
      at.qkv = qkv16; at.ld = 3 * inner; at.bs = (long long)Tl * 3 * inner;
      at.B = B; at.T = Tl; at.H = Hh; at.D = hd; at.inner = inner; at.scale = 1.0f / sqrtf((float)hd);
      at.lens = d.ylen32; at.len_shift = shift;
      at.out = d.att; at.out_ld = inner; at.out_bs = (long long)Tl * inner;
      // Queries in the padding: their attention output only feeds rows of the residual stream that the block's masked
      // output discards, so whole padded query blocks are skipped (keys / values of padded frames still take part, H1)
      at.skip_padded_queries = (use_ff_tiles && ff_fused) ? 1 : 0;
      std::string err;
      cudaError_t ce;
      if (dbg_skip & 4) ce = cudaSuccess; else
      { LaunchScope ls(ctx, s, "attention_tc", attn_flops, (double)B * Tl * inner * 8.0); ce = attention_tc(at, s, &err); }
      if (ce != cudaSuccess) return err.empty() ? cuda_fail(ctx, ce, "attention_tc") : fail(ctx, EV_ERR_CUDA, err);
    } else {
      Epilogue eq; eq.out_f32 = d.qkv; eq.f32_ld = 3 * inner; eq.f32_bs = (long long)Tl * 3 * inner;
      EV_TRY(run_conv<ActT>(ctx, w.qkv, d.n, D, bsD, B, Tl, eq, s));
      AttnArgs at;
      at.q = d.qkv; at.k = d.qkv + inner; at.v = d.qkv + 2 * inner; at.ld = 3 * inner; at.bs = (long long)Tl * 3 * inner;
      at.B = B; at.T = Tl; at.H = Hh; at.D = hd; at.scale = 1.0f / sqrtf((float)hd);
      at.lens = d.ylen32; at.len_shift = shift; at.mode = 1;
      at.out = d.att; at.out_ld = inner; at.out_bs = (long long)Tl * inner;
      EV_LAUNCH(ctx, s, "attention_dec", attn_flops, (double)B * Tl * inner * (12.0 + sizeof(ActT)), attention_rows<ActT>(at, s));
    }
    if constexpr (std::is_same<ActT, bf16>::value) {
      if (xr_is_cf) {
        // out-projection + residual + LayerNorm3 + ff1 + SnakeBeta + ff2 + residual + mask: ONE launch (ff_tc.cu, tail mode)
        FfTcArgs fa;
        fa.att = d.att; fa.att_ld = inner; fa.att_bs = (long long)Tl * inner; fa.oproj = &w.out; fa.xr_cf = d.xr;
        fa.ln_g = w.ln3_g; fa.ln_b = w.ln3_b; fa.eps = 1e-5f; fa.ff1 = &w.ff1; fa.ff2 = &w.ff2;
        fa.snake_a = w.snake_a; fa.snake_invb = w.snake_invb;
        fa.out = out; fa.out_ld = out_ld; fa.out_bs = (long long)Tl * out_ld; fa.lens = d.ylen32; fa.len_shift = shift;
        fa.B = B; fa.T = Tl;
        fa.tiles = use_ff_tiles ? d.ff_tiles[shift] : nullptr;
        std::string err;
        cudaError_t ce;
        { LaunchScope ls(ctx, s, "ff_tc", 4.0 * B * (double)Tl * D * (w.ff1.N + inner / 2), (double)B * Tl * (D * 6.0 + inner * 2.0) + 4.0 * D * w.ff1.N);
          ce = ff_tc_launch(fa, s, &err); }
        if (ce != cudaSuccess) return err.empty() ? cuda_fail(ctx, ce, "ff_tc") : fail(ctx, EV_ERR_CUDA, err);
        return 0;
      }
    }
    Epilogue eo; eo.res = d.xr; eo.res_ld = D; eo.res_bs = bsD; eo.out_f32 = d.xr; eo.f32_ld = D; eo.f32_bs = bsD;
    if (use_ff_tiles && ff_fused) {   // out-projection: tiles without a valid row are skipped (same argument; the planner caches one table per level)
      rag.rows_per_frame = 1; rag.len_shift = shift;
      ctx->rag = rag;
    }
    const int rc_out = run_conv<ActT>(ctx, w.out, d.att, inner, (long long)Tl * inner, B, Tl, eo, s);
    if (use_ff_tiles && ff_fused) { rag = ctx->rag; ctx->rag = RaggedPlanner(); }
    EV_TRY(rc_out);
    if constexpr (std::is_same<ActT, bf16>::value) {
      // LayerNorm3 + ff1 + SnakeBeta + ff2 + residual + mask as ONE kernel: the 1024-wide hidden tensor stays on the SM (ff_tc.cu)
      if (ff_fused) {
        FfTcArgs fa;
        fa.x = d.xr; fa.ln_g = w.ln3_g; fa.ln_b = w.ln3_b; fa.eps = 1e-5f; fa.ff1 = &w.ff1; fa.ff2 = &w.ff2;
        fa.snake_a = w.snake_a; fa.snake_invb = w.snake_invb;
        fa.out = out; fa.out_ld = out_ld; fa.out_bs = (long long)Tl * out_ld; fa.lens = d.ylen32; fa.len_shift = shift;
        fa.B = B; fa.T = Tl;
        fa.tiles = use_ff_tiles ? d.ff_tiles[shift] : nullptr;
        std::string err;
        cudaError_t ce;
        { LaunchScope ls(ctx, s, "ff_tc", 4.0 * B * (double)Tl * D * w.ff1.N, (double)B * Tl * D * 10.0 + 4.0 * D * w.ff1.N);
          ce = ff_tc_launch(fa, s, &err); }
        if (ce != cudaSuccess) return err.empty() ? cuda_fail(ctx, ce, "ff_tc") : fail(ctx, EV_ERR_CUDA, err);
        return 0;
      }
    }
    LnArgs ln;
    ln.x = d.xr; ln.x_ld = D; ln.gamma = w.ln3_g; ln.beta = w.ln3_b; ln.eps = 1e-5f; ln.out_act = d.n; ln.act_ld = D;
    ln.B = B; ln.T = Tl; ln.C = D;
    EV_LAUNCH(ctx, s, "layer_norm", 0, (double)B * Tl * D * (4.0 + sizeof(ActT)), layer_norm_rows<ActT>(ln, s));
    Epilogue e1; e1.act = ACT_SNAKE; e1.snake_a = w.snake_a; e1.snake_invb = w.snake_invb;
    e1.out_act = d.ff; e1.act_ld = 4 * D; e1.act_bs = (long long)Tl * 4 * D;
    if (!(dbg_skip & 1)) EV_TRY(run_conv<ActT>(ctx, w.ff1, d.n, D, bsD, B, Tl, e1, s));
    Epilogue e2; e2.res = d.xr; e2.res_ld = D; e2.res_bs = bsD;
    e2.out_act = out; e2.act_ld = out_ld; e2.act_bs = (long long)Tl * out_ld; e2.mask = mask; e2.mask_act = 1;
    if (!(dbg_skip & 2)) EV_TRY(run_conv<ActT>(ctx, w.ff2, d.ff, 4 * D, (long long)Tl * 4 * D, B, Tl, e2, s));
    return 0;
  }

  int step(const float* temb_step, float dt) {
    const int T2 = T / 2;
    const int dec_in = (int)m.rn[0].c_in;
    const RowMask mask0{d.ylen32, 0}, mask1{d.ylen32, 1};
    const long long bs0 = (long long)T * 2 * D, bs1 = (long long)T2 * 2 * D;
    // down 0 (T): resnet, transformer -> skip0 (masked) ; stride-2 conv -> din (T/2, masked by mask[::2])
    EV_TRY(resnet(0, d.xin, dec_in, T, 0, temb_step + 0 * D));
    EV_TRY(transformer(0, T, 0, d.cat0 + D, 2 * D));
    { Epilogue e; e.out_act = d.din; e.act_ld = D; e.act_bs = (long long)T2 * D; e.mask = mask1; e.mask_act = 1;
      EV_TRY(run_conv<ActT>(ctx, m.down0, d.cat0 + D, 2 * D, bs0, B, T, e, s)); }
    // down 1 (T/2): resnet, transformer -> skip1 ; conv3 -> din
    EV_TRY(resnet(1, d.din, D, T2, 1, temb_step + 1 * D));
    EV_TRY(transformer(1, T2, 1, d.cat1 + D, 2 * D));
    { Epilogue e; e.out_act = d.din; e.act_ld = D; e.act_bs = (long long)T2 * D; e.mask = mask1; e.mask_act = 1;
      EV_TRY(run_conv<ActT>(ctx, m.down1_conv, d.cat1 + D, 2 * D, bs1, B, T2, e, s)); }
    // mid blocks (T/2)
    EV_TRY(resnet(2, d.din, D, T2, 1, temb_step + 2 * D));
    EV_TRY(transformer(2, T2, 1, d.din, D));
    EV_TRY(resnet(3, d.din, D, T2, 1, temb_step + 3 * D));
    EV_TRY(transformer(3, T2, 1, d.cat1, 2 * D));
    // up 0 (T/2): resnet on [x | skip1], transformer, transposed conv -> cat0[:, :, :D] (T)
    EV_TRY(resnet(4, d.cat1, 2 * D, T2, 1, temb_step + 4 * D));
    EV_TRY(transformer(4, T2, 1, d.a, D));
    { Epilogue e; e.out_act = d.cat0; e.act_ld = 2 * D; e.act_bs = bs0; e.mask = mask0; e.mask_act = 1;
      EV_TRY(run_conv<ActT>(ctx, m.up0, d.a, D, (long long)T2 * D, B, T2, e, s)); }
    // up 1 (T): resnet on [x | skip0], transformer, conv3 -> n (masked: final_block multiplies by mask)
    EV_TRY(resnet(5, d.cat0, 2 * D, T, 0, temb_step + 5 * D));
    EV_TRY(transformer(5, T, 0, d.a, D));
    { Epilogue e; e.out_act = d.n; e.act_ld = D; e.act_bs = (long long)T * D; e.mask = mask0; e.mask_act = 1;
      EV_TRY(run_conv<ActT>(ctx, m.up1_conv, d.a, D, (long long)T * D, B, T, e, s)); }
    // final_block (conv3 -> GN -> Mish -> *mask), final_proj fused with the Euler update x += dt * (proj*mask)
    bool final_fused = false;
    if constexpr (std::is_same<ActT, bf16>::value) {
      if (D == 256 && resnet_tc_supported(m.final_conv, nullptr, nullptr, B, T)) {   // conv -> GN -> Mish -> mask in one launch
        ResnetTcArgs ra;
        ra.x = d.n; ra.x_ld = D; ra.x_bs = (long long)T * D;
        ra.conv1 = &m.final_conv; ra.gn_g1 = m.final_g; ra.gn_b1 = m.final_b;
        ra.lens = d.ylen32; ra.len_shift = 0; ra.B = B; ra.T = T;
        ra.a_buf = d.a; ra.a_ld = D; ra.a_bs = (long long)T * D;
        EV_TRY(launch_resnet_tc(ra, 2.0 * B * T * D * 3.0 * D, (double)B * T * 4.0 * D, "final_block_tc"));
        final_fused = true;
      }
    }
    if (!final_fused) {
    const double* part = d.gn_partial;
    { Epilogue e; e.out_f32 = d.h; e.f32_ld = D; e.f32_bs = (long long)T * D;
      if (fuse_gn()) { e.gn_sum = next_gn_slot(); e.gn_groups = 8; part = e.gn_sum; }
      EV_TRY(run_conv<ActT>(ctx, m.final_conv, d.n, D, (long long)T * D, B, T, e, s)); }
    int chunks = 1;
    const double RD = (double)B * T * D;
    if (!fuse_gn()) EV_LAUNCH(ctx, s, "gn_stats", 0, RD * 4.0, group_norm_stats(d.h, B, T, D, 8, d.gn_partial, &chunks, s));
    GnApplyArgs g;
    g.x = d.h; g.partial = part; g.n_chunks = chunks; g.gamma = m.final_g; g.beta = m.final_b;
    g.B = B; g.T = T; g.C = D; g.mask = mask0; g.out_act = d.a; g.act_ld = D;
    EV_LAUNCH(ctx, s, "gn_apply", 0, RD * (4.0 + sizeof(ActT)), group_norm_apply<ActT>(g, s));
    }
    const int F = m.cfg.n_feats;
    Epilogue e; e.mask = mask0; e.mask_pre = 1; e.alpha = dt;
    e.out_f32 = d.xstate; e.f32_ld = F; e.f32_bs = (long long)T * F;
    if (!estimator_only) {     // Euler update x += dt * v * mask, and the next step's operand
      e.res = d.xstate; e.res_ld = F; e.res_bs = (long long)T * F;
      e.out_act = d.xin; e.act_ld = dec_in; e.act_bs = (long long)T * dec_in; e.mask_act = 1;
    }
    EV_TRY(run_conv<ActT>(ctx, m.final_proj, d.a, D, (long long)T * D, B, T, e, s));
    return 0;
  }
};

// Batch slices ("lanes") the decoder runs concurrently: every per-item quantity of the estimator (GroupNorm statistics,
// attention, masks) is independent of the other items of the batch, so slices of the batch are exact.
int decode_lane_count(const ev_ctx* ctx, int B) {
  if (ctx->profiling) return 1;            // per-launch event timing wants one serial stream
  return std::max(1, std::min(ctx->dec_lanes, B / 4));
}

template <typename ActT>
int decode_impl(ev_ctx* ctx, const float* mu_y, const int64_t* y_lengths, const float* z, const float* spk_emb, int B,
                int T, int n_steps, float temperature, float* decoder_out, float* mel, void* workspace, size_t ws_bytes,
                cudaStream_t s, const float* t_items = nullptr) {
  // t_items != nullptr (ev_estimator): ONE evaluation of the estimator with its own time t_items[b] per item; `z` is the point
  // it is evaluated at and decoder_out receives v * mask (decoder.py:363-443 as flow_matching.py:114 calls it)
  const bool est = t_items != nullptr;
  const int n_rows = est ? B : n_steps;     // rows of the time-embedding chain
  const MatchaW& m = ctx->matcha;
  const ev_matcha_cfg& c = m.cfg;
  Workspace w(workspace, ws_bytes);
  const int n_lanes = est ? 1 : decode_lane_count(ctx, B);
  int lane_b0[ev_ctx::kMaxLanes], lane_nb[ev_ctx::kMaxLanes];
  DecBuffers<ActT> dl[ev_ctx::kMaxLanes];
  for (int l = 0, b0 = 0; l < n_lanes; ++l) {
    lane_b0[l] = b0;
    lane_nb[l] = B / n_lanes + (l < B % n_lanes ? 1 : 0);
    b0 += lane_nb[l];
    plan_decode<ActT>(c, lane_nb[l], T, n_rows, w, &dl[l]);
  }
  if (w.overflow || !workspace) return fail(ctx, EV_ERR_STATE, "ev_decode: workspace too small");
  ctx->prof_tag = "/dec";
  const int D = c.dec_channels, F = c.n_feats, S = c.n_spks > 1 ? c.spk_emb_dim : 0, dec_in = 2 * F + S;
  DecBuffers<ActT>& d = dl[0];
  // time embeddings of all steps at once (they do not depend on the batch): sinusoid -> Linear -> SiLU -> Linear,
  // then Mish -> the six resnet mlp Linears stacked along N (decoder.py:381-382, :49,58)
  std::vector<float> ts, dts;
  euler_schedule(n_steps, &ts, &dts);
  // The time-embedding chain depends on nothing but n_steps: with one lane it runs as a side branch (second lane stream) next
  // to the input packing and the first ResNet conv, and is joined where the first time embedding is consumed.
  const bool temb_side = n_lanes == 1 && ctx->dec_side && !ctx->profiling && std::is_same<ActT, bf16>::value;
  cudaStream_t st = temb_side ? ctx->lane_stream[1] : s;
  if (temb_side) {
    EV_CUDA(ctx, cudaEventRecord(ctx->lane_fork, s));
    EV_CUDA(ctx, cudaStreamWaitEvent(st, ctx->lane_fork, 0));
  }
  if (est) {
    EV_CUDA(ctx, cudaMemcpyAsync(d.t_steps, t_items, (size_t)B * sizeof(float), cudaMemcpyDeviceToDevice, st));
  } else {
    EV_LAUNCH(ctx, st, "upload_floats", 0, 4.0 * n_steps, upload_floats(d.t_steps, ts.data(), n_steps, st));
    ctx->launches += ceil_div(n_steps, 32) - 1;
  }
  EV_LAUNCH(ctx, st, "time_sinusoid", 0, 4.0 * n_rows * dec_in, time_sinusoid(d.t_steps, n_rows, dec_in, d.sinus, st));
  { Epilogue e; e.act = ACT_SILU; e.out_act = d.th1; e.act_ld = 4 * D; e.act_bs = 0;
    EV_TRY(run_conv<float>(ctx, m.time1, d.sinus, dec_in, 0, 1, n_rows, e, st)); }
  { Epilogue e; e.act = ACT_MISH; e.out_act = d.th2; e.act_ld = 4 * D; e.act_bs = 0;
    EV_TRY(run_conv<float>(ctx, m.time2, d.th1, 4 * D, 0, 1, n_rows, e, st)); }
  { Epilogue e; e.out_f32 = d.tproj; e.f32_ld = 6 * D; e.f32_bs = 0;
    EV_TRY(run_conv<float>(ctx, m.temb_proj, d.th2, 4 * D, 0, 1, n_rows, e, st)); }
  if (temb_side) EV_CUDA(ctx, cudaEventRecord(ctx->lane_join[1], st));
  // fork: lane 0 stays on the caller's stream, the others wait for the time embeddings on their own streams
  cudaStream_t ls[ev_ctx::kMaxLanes];
  ls[0] = s;
  if (n_lanes > 1) EV_CUDA(ctx, cudaEventRecord(ctx->lane_fork, s));
  for (int l = 1; l < n_lanes; ++l) {
    ls[l] = ctx->lane_stream[l - 1];
    EV_CUDA(ctx, cudaStreamWaitEvent(ls[l], ctx->lane_fork, 0));
  }
  std::vector<Decoder<ActT>> dec;
  dec.reserve(n_lanes);
  const long long item = (long long)F * T;
  for (int l = 0; l < n_lanes; ++l) {
    const int b0 = lane_b0[l], nb = lane_nb[l];
    DecBuffers<ActT>& q = dl[l];
    EV_LAUNCH(ctx, ls[l], "i64_to_i32", 0, 12.0 * nb, i64_to_i32(reinterpret_cast<const long long*>(y_lengths) + b0, q.ylen32, nb, ls[l]));
    const RowMask mask0{q.ylen32, 0};
    EV_LAUNCH(ctx, ls[l], "decoder_pack_input", 0, (double)nb * T * (12.0 * F + sizeof(ActT) * dec_in),
              (decoder_pack_input<ActT>(z + b0 * item, mu_y + b0 * item, spk_emb ? spk_emb + (long long)b0 * S : nullptr, nb, F, S, T,
                                        temperature, mask0, q.xstate, q.xin, dec_in, ls[l])));
    dec.push_back(Decoder<ActT>{ctx, m, q, nb, T, ls[l], D, c.dec_heads * c.dec_head_dim});
    if (n_lanes == 1 && ctx->dec_side && std::is_same<ActT, bf16>::value) dec.back().side_stream = ctx->lane_stream[ev_ctx::kMaxLanes - 2];
    if (temb_side) dec.back().temb_event = ctx->lane_join[1];
    if (est) { dec.back().temb_bs = 6LL * D; dec.back().estimator_only = true; }
    if (std::is_same<ActT, bf16>::value && nb <= kRaggedMaxB) {
      static const bool on = []() { const char* v = getenv("EV_FF_RAGGED"); return !(v && atoi(v) == 0); }();
      if (on) {
        EV_LAUNCH(ctx, ls[l], "ragged_table", 0, 8.0 * nb, ragged_build_table(q.ylen32, nb, 0, 1, 0, 128, T, q.ff_tiles[0], ls[l]));
        EV_LAUNCH(ctx, ls[l], "ragged_table", 0, 8.0 * nb, ragged_build_table(q.ylen32, nb, 0, 1, 1, 128, T / 2, q.ff_tiles[1], ls[l]));
        dec.back().use_ff_tiles = true;
        RaggedPlanner& r = dec.back().rag;
        r.lens = q.ylen32; r.B = nb; r.margin = 0; r.arena = q.rag_arena; r.arena_ints = q.rag_ints; r.launch_counter = &ctx->launches;
      }
    }
    if (dec.back().fuse_gn()) {
      EV_CUDA(ctx, cudaMemsetAsync(q.gn_fused, 0, q.gn_fused_count * sizeof(double), ls[l]));
    }
  }
  // launches interleave across lanes step by step so that eager (un-captured) calls overlap as well
  if (est) EV_TRY(dec[0].step(d.tproj, 1.0f));      // item b reads row b of tproj (temb_bs)
  for (int k = 0; k < n_steps && !est; ++k)
    for (int l = 0; l < n_lanes; ++l) EV_TRY(dec[l].step(d.tproj + (size_t)k * 6 * D, dts[k]));
  for (int l = 0; l < n_lanes; ++l) {
    const int b0 = lane_b0[l], nb = lane_nb[l];
    DecBuffers<ActT>& q = dl[l];
    EV_LAUNCH(ctx, ls[l], "cl_to_cf", 0, 8.0 * nb * T * F, cl_to_cf(q.xstate, F, (long long)T * F, nb, F, T, decoder_out + b0 * item, 1.0f, 0.0f, ls[l]));
    if (mel) EV_LAUNCH(ctx, ls[l], "cl_to_cf", 0, 8.0 * nb * T * F, cl_to_cf(q.xstate, F, (long long)T * F, nb, F, T, mel + b0 * item, c.mel_std, c.mel_mean, ls[l]));
    if (l > 0) {
      EV_CUDA(ctx, cudaEventRecord(ctx->lane_join[l - 1], ls[l]));
      EV_CUDA(ctx, cudaStreamWaitEvent(s, ctx->lane_join[l - 1], 0));
    }
  }
  return 0;
}

}  // namespace

extern "C" size_t ev_decode_workspace_bytes(const ev_ctx* ctx, int B, int T_pad, int n_timesteps) {
  if (!ctx || !ctx->matcha.loaded || B <= 0 || T_pad <= 0 || n_timesteps <= 0) return 0;
  Workspace w(nullptr, 0);
  DecBuffers<float> d;  // fp32 operands are the larger plan; it also covers bf16
  const int n_lanes = std::min(std::max(ctx->dec_lanes, 1), std::max(1, B / 4));   // upper bound of decode_lane_count
  for (int l = 0; l < n_lanes; ++l) plan_decode<float>(ctx->matcha.cfg, B / n_lanes + (l < B % n_lanes ? 1 : 0), T_pad, n_timesteps, w, &d);
  size_t lanes_bytes = w.off;
  Workspace w1(nullptr, 0);                // the single-lane plan (profiling mode) must fit too
  plan_decode<float>(ctx->matcha.cfg, B, T_pad, n_timesteps, w1, &d);
  return std::max(lanes_bytes, w1.off) + 256;
}

extern "C" int ev_decode(ev_ctx* ctx, const float* mu_y, const int64_t* y_lengths, const float* z, const float* spk_emb,
                         int B, int T_pad, int n_timesteps, float temperature, int precision, float* decoder_out,
                         float* mel, void* workspace, size_t workspace_bytes, void* stream) {
  if (!ctx) return EV_ERR_INVALID;
  if (!ctx->matcha.loaded) return fail(ctx, EV_ERR_STATE, "ev_decode: matcha weights not loaded");
  if (!mu_y || !y_lengths || !z || !decoder_out || B <= 0 || T_pad <= 0 || n_timesteps <= 0)
    return fail(ctx, EV_ERR_INVALID, "ev_decode: null argument or empty shape");
  if (T_pad % 4) return fail(ctx, EV_ERR_INVALID, "ev_decode: T_pad must be a multiple of 4 (fix_len_compatibility)");
  if (ctx->matcha.cfg.n_spks > 1 && !spk_emb) return fail(ctx, EV_ERR_INVALID, "ev_decode: spk_emb required");
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = as_stream(stream);
  if (precision == EV_PREC_FP32)
    return decode_impl<float>(ctx, mu_y, y_lengths, z, spk_emb, B, T_pad, n_timesteps, temperature, decoder_out, mel, workspace, workspace_bytes, s);
  if (precision == EV_PREC_BF16)
    return decode_impl<bf16>(ctx, mu_y, y_lengths, z, spk_emb, B, T_pad, n_timesteps, temperature, decoder_out, mel, workspace, workspace_bytes, s);
  return fail(ctx, EV_ERR_INVALID, "ev_decode: unknown precision");
}

extern "C" size_t ev_estimator_workspace_bytes(const ev_ctx* ctx, int B, int T_pad) {
  return ev_decode_workspace_bytes(ctx, B, T_pad, std::max(B, 1));
}

// One evaluation of the flow-matching estimator (decoder.py:363-443) with one time per item, as the training loss calls it
// (flow_matching.py:114): v = estimator(y, mask, mu, t, spks).  All tensors channel-first like the reference's.
extern "C" int ev_estimator(ev_ctx* ctx, const float* y, const int64_t* y_lengths, const float* mu, const float* t, const float* spk_emb,
                            int B, int T_pad, int precision, float* v_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!ctx) return EV_ERR_INVALID;
  if (!ctx->matcha.loaded) return fail(ctx, EV_ERR_STATE, "ev_estimator: matcha weights not loaded");
  if (!y || !y_lengths || !mu || !t || !v_out || B <= 0 || T_pad <= 0) return fail(ctx, EV_ERR_INVALID, "ev_estimator: null argument or empty shape");
  if (T_pad % 4) return fail(ctx, EV_ERR_INVALID, "ev_estimator: T_pad must be a multiple of 4 (the U-Net halves the length twice)");
  if (ctx->matcha.cfg.n_spks > 1 && !spk_emb) return fail(ctx, EV_ERR_INVALID, "ev_estimator: spk_emb required");
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = as_stream(stream);
  if (precision == EV_PREC_FP32)
    return decode_impl<float>(ctx, mu, y_lengths, y, spk_emb, B, T_pad, 1, 1.0f, v_out, nullptr, workspace, workspace_bytes, s, t);
  if (precision == EV_PREC_BF16)
    return decode_impl<bf16>(ctx, mu, y_lengths, y, spk_emb, B, T_pad, 1, 1.0f, v_out, nullptr, workspace, workspace_bytes, s, t);
  return fail(ctx, EV_ERR_INVALID, "ev_estimator: unknown precision");
}

// test hook: the Euler schedule as the library computes it (pure host code)
extern "C" int ev_test_euler_schedule(int n, float* t_host, float* dt_host) {
  if (n <= 0 || !t_host || !dt_host) return EV_ERR_INVALID;
  std::vector<float> t, dt;
  euler_schedule(n, &t, &dt);
  for (int i = 0; i < n; ++i) { t_host[i] = t[i]; dt_host[i] = dt[i]; }
  return 0;
}
