// HiFi-GAN v1 generator on the GPU (hifigan/models.py:148-206): conv_pre, 4 x [LeakyReLU, polyphase transposed
// conv, mean of three dilated ResBlock1 branches], LeakyReLU(0.01), conv_post, tanh, clamp.  Every conv is the
// shared implicit GEMM; activations/residual adds/MRF mean are fused into its epilogue (see DESIGN.md).
#include <cstdlib>

#include "ctx.cuh"

using namespace ev;

namespace {
cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
constexpr float kSlope = 0.1f;  // LRELU_SLOPE, hifigan/models.py:11

__global__ void fold_weight_norm_kernel(const float* __restrict__ g, const float* __restrict__ v, int rows, int cols,
                                        float* __restrict__ w) {
  // torch.nn.utils.weight_norm, dim=0: w[r,:] = g[r] * v[r,:] / ||v[r,:]||   (one block per row)
  __shared__ float red[32];
  const int r = blockIdx.x;
  const float* vr = v + (long long)r * cols;
  float s = 0.0f;
  for (int i = threadIdx.x; i < cols; i += blockDim.x) s += vr[i] * vr[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0f;
    t = warp_sum(t);
    if (threadIdx.x == 0) red[0] = t;
  }
  __syncthreads();
  const float scale = g[r] / sqrtf(red[0]);
  for (int i = threadIdx.x; i < cols; i += blockDim.x) w[(long long)r * cols + i] = vr[i] * scale;
}

__global__ void bias_cumsum_kernel(const float* b0, const float* b1, const float* b2, int C, float* o0, float* o1, float* o2) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) { const float s0 = b0[c], s1 = s0 + b1[c]; o0[c] = s0; o1[c] = s1; o2[c] = s1 + b2[c]; }
}

__global__ void pack_post_kernel(const float* src, int C, int K, float* dst) {  // (1,C,K) -> [K][C]
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < C * K) { const int j = i / C, c = i - j * C; dst[i] = src[c * K + j]; }
}

// Accept either plain `name.weight` or the checkpoint form `name.weight_g` + `name.weight_v` (feel_me.py:161-167 loads
// the latter and then calls remove_weight_norm()).  Returns a tensor record pointing at a folded copy when needed.
int resolve_weight(ev_ctx* ctx, WeightStore& ws, const std::string& base, long long d0, long long d1, long long d2,
                   std::vector<ev_tensor>* extra, std::vector<std::string>* extra_names) {
  if (ws.has(base + ".weight")) return 0;
  if (!ws.has(base + ".weight_g") || !ws.has(base + ".weight_v")) return fail(ctx, EV_ERR_MISSING, "missing weight tensor: " + base + ".weight");
  const ev_tensor* g = ws.get(base + ".weight_g", {d0});
  const ev_tensor* v = ws.get(base + ".weight_v", {d0, d1, d2});
  if (!g || !v) return EV_ERR_INVALID;
  void* p;
  EV_TRY(device_alloc(ctx, (size_t)(d0 * d1 * d2) * sizeof(float), &p, false, ws.stream));
  fold_weight_norm_kernel<<<(int)d0, 256, 0, ws.stream>>>(g->data, v->data, (int)d0, (int)(d1 * d2), reinterpret_cast<float*>(p));
  EV_CUDA(ctx, cudaGetLastError());
  extra_names->push_back(base + ".weight");
  ev_tensor t{};
  t.data = reinterpret_cast<float*>(p);
  t.ndim = 3; t.shape[0] = d0; t.shape[1] = d1; t.shape[2] = d2;
  extra->push_back(t);
  return 0;
}
}  // namespace

namespace ev {

int load_resblock(ev_ctx* ctx, WeightStore& ws, const std::string& prefix, int C, int k, const int dil[3], ConvWeights c1[3],
                  ConvWeights c2[3], float* bacc[3], cudaStream_t s) {
  for (int l = 0; l < 3; ++l) {
    const std::string a = prefix + "convs1." + std::to_string(l), b = prefix + "convs2." + std::to_string(l);
    // get_padding(k, d) = (k*d - d)/2  (hifigan/xutils.py:37-38)
    EV_TRY(make_conv(ctx, ws, {a + ".weight"}, {a + ".bias"}, C, C, k, 1, (k * dil[l] - dil[l]) / 2, dil[l], CONV_NORMAL, TC_BF16, &c1[l]));
    EV_TRY(make_conv(ctx, ws, {b + ".weight"}, {b + ".bias"}, C, C, k, 1, (k - 1) / 2, 1, CONV_NORMAL, TC_BF16, &c2[l]));
  }
  for (int l = 0; l < 3; ++l) {
    void* q;
    EV_TRY(device_alloc(ctx, (size_t)align_up(C, 4) * sizeof(float), &q, true, s));
    bacc[l] = reinterpret_cast<float*>(q);
  }
  if (c2[0].bias && c2[1].bias && c2[2].bias) {
    bias_cumsum_kernel<<<ceil_div(C, 128), 128, 0, s>>>(c2[0].bias, c2[1].bias, c2[2].bias, C, bacc[0], bacc[1], bacc[2]);
    EV_CUDA(ctx, cudaGetLastError());
  }
  return 0;
}

template <typename ActT>
int run_resblock(ev_ctx* ctx, const ResBlockArgs<ActT>& a, cudaStream_t s) {
  const int C = a.C;
  const long long bs = (long long)a.L * C;
  if (a.fused) {
    if constexpr (std::is_same<ActT, bf16>::value) {
      // fused ResBlock: six convs in one kernel, residual stream resident in TMEM (resblock_tc.cu)
      if (a.mode > 2) return fail(ctx, EV_ERR_INVALID, "resblock_tc: a lone branch (mode 3) runs layer by layer");
      const double fl = 3 * 2.0 * 2.0 * a.B * (double)a.L * C * (double)C * a.k;
      std::string msg;
      cudaError_t ce;
      {
        char nm[48];
        snprintf(nm, sizeof nm, "resblock_tc/voc c%d k%d", C, a.k);
        LaunchScope ls(ctx, s, ctx->prof_detail ? nm : "resblock_tc/voc", fl, (double)a.B * a.L * C * (4.0 + (a.mode ? 8.0 : 4.0)));
        ce = resblock_tc_launch(C, a.k, a.c1, a.c2, a.bacc, a.x, a.sum, a.act_out, a.B, a.L, a.mode, a.inv_n, a.slope_out, a.write_f32, s,
                                &msg, ctx->rag.active() ? &ctx->rag : nullptr, a.sched, a.info);
      }
      if (ce == cudaErrorInvalidValue && !msg.empty()) return fail(ctx, EV_ERR_INVALID, msg);
      if (ce != cudaSuccess) return fail(ctx, EV_ERR_CUDA, "resblock_tc_launch: " + (msg.empty() ? std::string(cudaGetErrorString(ce)) : msg));
      return 0;
    } else {
      return fail(ctx, EV_ERR_INVALID, "resblock_tc: the fused ResBlock runs with bf16 operands only");
    }
  }
  const float* in_f32 = a.x;
  const ActT* in_act = a.x_act;
  for (int l = 0; l < 3; ++l) {  // ResBlock1.forward (hifigan/models.py:90-97)
    Epilogue e1; e1.act = ACT_LRELU; e1.slope = kSlope; e1.out_act = a.mid; e1.act_ld = C; e1.act_bs = bs;
    EV_TRY(run_conv<ActT>(ctx, *a.c1[l], in_act, C, bs, a.B, a.L, e1, s));
    Epilogue e2; e2.res = in_f32; e2.res_ld = C; e2.res_bs = bs;
    if (l < 2) {
      e2.out_f32 = a.xb; e2.f32_ld = C; e2.f32_bs = bs;
      e2.act = ACT_LRELU; e2.slope = kSlope; e2.out_act = a.xba; e2.act_ld = C; e2.act_bs = bs;
    } else {  // branch output joins the MRF sum; the last branch divides by n_kernels (hifigan/models.py:186-192)
      if (a.mode == 1 || a.mode == 2) { e2.res2 = a.sum; e2.res2_ld = C; e2.res2_bs = bs; }
      if (a.mode < 2 || a.write_f32) { e2.out_f32 = a.sum; e2.f32_ld = C; e2.f32_bs = bs; }
      if (a.mode >= 2) {
        e2.div = 1.0f / a.inv_n;
        if (a.act_out) { e2.act = ACT_LRELU; e2.slope = a.slope_out; e2.out_act = a.act_out; e2.act_ld = C; e2.act_bs = bs; }
      }
    }
    EV_TRY(run_conv<ActT>(ctx, *a.c2[l], a.mid, C, bs, a.B, a.L, e2, s));
    in_f32 = a.xb;
    in_act = a.xba;
  }
  return 0;
}
template int run_resblock<float>(ev_ctx*, const ResBlockArgs<float>&, cudaStream_t);
template int run_resblock<bf16>(ev_ctx*, const ResBlockArgs<bf16>&, cudaStream_t);

}  // namespace ev

extern "C" int ev_load_hifigan(ev_ctx* ctx, const ev_tensor* weights, int n_weights, const ev_hifigan_cfg* cfg, void* stream) {
  if (!ctx || !weights || !cfg) return EV_ERR_INVALID;
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  if (ctx->hifigan.loaded) return fail(ctx, EV_ERR_STATE, "hifigan weights already loaded in this context");
  const ev_hifigan_cfg& c = *cfg;
  if (c.n_ups <= 0 || c.n_ups > 8 || c.n_kernels <= 0 || c.n_kernels > 4 || (c.num_mels & 7) || (c.upsample_initial_channel >> c.n_ups) < 16)
    return fail(ctx, EV_ERR_INVALID, "unsupported HiFi-GAN configuration");
  HifiganW& h = ctx->hifigan;
  h.cfg = c;
  // pass 1: fold weight-norm checkpoints into plain weights, extend the tensor list with the folded copies
  std::vector<ev_tensor> all(weights, weights + n_weights);
  {
    WeightStore ws0(ctx, weights, n_weights, s);
    std::vector<ev_tensor> extra;
    std::vector<std::string> names;
    const int c0 = c.upsample_initial_channel;
    EV_TRY(resolve_weight(ctx, ws0, "conv_pre", c0, c.num_mels, 7, &extra, &names));
    for (int i = 0; i < c.n_ups; ++i) {
      const int cin = c0 >> i, ch = c0 >> (i + 1);
      EV_TRY(resolve_weight(ctx, ws0, "ups." + std::to_string(i), cin, ch, c.upsample_kernel_sizes[i], &extra, &names));
      for (int j = 0; j < c.n_kernels; ++j)
        for (int l = 0; l < 3; ++l) {
          const std::string rb = "resblocks." + std::to_string(i * c.n_kernels + j);
          EV_TRY(resolve_weight(ctx, ws0, rb + ".convs1." + std::to_string(l), ch, ch, c.resblock_kernel_sizes[j], &extra, &names));
          EV_TRY(resolve_weight(ctx, ws0, rb + ".convs2." + std::to_string(l), ch, ch, c.resblock_kernel_sizes[j], &extra, &names));
        }
    }
    EV_TRY(resolve_weight(ctx, ws0, "conv_post", 1, c0 >> c.n_ups, 7, &extra, &names));
    static thread_local std::vector<std::string> keep;  // keeps the c_str() of synthesized names alive for `all`
    keep = names;
    for (size_t i = 0; i < extra.size(); ++i) { extra[i].name = keep[i].c_str(); all.push_back(extra[i]); }
  }
  WeightStore ws(ctx, all.data(), (int)all.size(), s);
  const int c0 = c.upsample_initial_channel;
  EV_TRY(make_conv(ctx, ws, {"conv_pre.weight"}, {"conv_pre.bias"}, c0, c.num_mels, 7, 1, 3, 1, CONV_NORMAL, TC_BF16, &h.conv_pre));
  h.total_up = 1;
  for (int i = 0; i < c.n_ups; ++i) {
    const int cin = c0 >> i, ch = c0 >> (i + 1);
    const int u = c.upsample_rates[i], k = c.upsample_kernel_sizes[i];
    h.total_up *= u;
    const std::string up = "ups." + std::to_string(i);
    EV_TRY(make_conv(ctx, ws, {up + ".weight"}, {up + ".bias"}, ch, cin, k, u, (k - u) / 2, 1, CONV_TRANSPOSED, TC_BF16, &h.ups[i]));
    for (int j = 0; j < c.n_kernels; ++j)
      EV_TRY(load_resblock(ctx, ws, "resblocks." + std::to_string(i * c.n_kernels + j) + ".", ch, c.resblock_kernel_sizes[j],
                           c.resblock_dilation_sizes[j], h.c1[i][j], h.c2[i][j], h.bacc[i][j], s));
  }
  h.c_last = c0 >> c.n_ups;
  if (h.c_last != 32 && h.c_last != 16) return fail(ctx, EV_ERR_INVALID, "conv_post supports 16 or 32 input channels");
  {
    const ev_tensor* t = ws.get("conv_post.weight", {1, (long long)h.c_last, 7});
    if (!t) return EV_ERR_MISSING;
    void* p;
    EV_TRY(device_alloc(ctx, (size_t)7 * h.c_last * sizeof(float), &p, false, s));
    h.post_w = reinterpret_cast<float*>(p);
    pack_post_kernel<<<ceil_div(7 * h.c_last, 128), 128, 0, s>>>(t->data, h.c_last, 7, h.post_w);
    EV_CUDA(ctx, cudaGetLastError());
    EV_TRY(ws.copy_vec("conv_post.bias", 1, &h.post_b));
  }
  EV_CUDA(ctx, cudaStreamSynchronize(s));
  h.loaded = true;
  return 0;
}

namespace {

template <typename ActT>
struct VocBuffers {
  ActT* mel; ActT* stage_in; float* x0; ActT* x0a; float* xb; ActT* xba; ActT* mid; float* sum;
  int* lens32; int* rag_arena; size_t rag_ints;
};

// How far past an utterance's end each layer must still be correct for the last valid sample to be exact, per stage, in mel
// frames.  Walks the generator backwards in samples of each stage's rate: conv_post looks 3 samples ahead; the widest
// ResBlock1 of a stage sum_l (k-1)/2 * (d_l + 1); a transposed conv output t reads inputs floor((t + p) / s) and the
// (k/s - 1) before it (bounded by ceil(h / s) + ceil(k / s)).  One spare frame is added everywhere.
struct VocMargins { int stage[8]; int up[8]; int pre; };
VocMargins vocoder_margins(const ev_hifigan_cfg& c) {
  VocMargins m{};
  long long rate[8], r = 1;
  for (int i = 0; i < c.n_ups; ++i) { r *= c.upsample_rates[i]; rate[i] = r; }
  long long h = 3;
  for (int i = c.n_ups - 1; i >= 0; --i) {
    long long rb = 0;
    for (int j = 0; j < c.n_kernels; ++j) {
      long long q = 0;
      for (int l = 0; l < 3; ++l) q += (long long)(c.resblock_kernel_sizes[j] - 1) / 2 * (c.resblock_dilation_sizes[j][l] + 1);
      rb = std::max(rb, q);
    }
    h += rb;                                                   // rows of the stage's input (= upsampler output) still needed
    m.stage[i] = (int)((h + rate[i] - 1) / rate[i]) + 1;       // safe for every conv inside the stage
    const int u = c.upsample_rates[i], k = c.upsample_kernel_sizes[i];
    h = (h + u - 1) / u + (k + u - 1) / u;                     // rows of the upsampler's input
    const long long rin = i > 0 ? rate[i - 1] : 1;
    m.up[i] = (int)((h + rin - 1) / rin) + 1;
  }
  m.pre = (int)h + 1;
  return m;
}

template <typename ActT>
void plan_vocode(const HifiganW& h, int B, int T, Workspace& w, VocBuffers<ActT>* v) {
  const ev_hifigan_cfg& c = h.cfg;
  size_t big = (size_t)T * c.upsample_initial_channel, L = T;
  for (int i = 0; i < c.n_ups; ++i) {
    L *= c.upsample_rates[i];
    big = std::max(big, L * (size_t)(c.upsample_initial_channel >> (i + 1)));
  }
  big *= B;
  v->mel = w.take<ActT>((size_t)B * T * c.num_mels);
  v->stage_in = w.take<ActT>(big);
  v->x0 = w.take<float>(big);
  v->x0a = w.take<ActT>(big);
  v->xb = w.take<float>(big);
  v->xba = w.take<ActT>(big);
  v->mid = w.take<ActT>(big);
  v->sum = w.take<float>(big);
  // ragged batches: int32 lengths + the compact tile lists (at most 32 geometries of <= B * ceil(L/128) + 64 entries)
  v->lens32 = w.take<int>((size_t)B);
  v->rag_ints = std::min<size_t>((size_t)32 * ((size_t)B * ((L + 127) / 128) + 64), (size_t)16 << 20);
  v->rag_arena = w.take<int>(v->rag_ints);
}

template <typename ActT>
int vocode_impl(ev_ctx* ctx, const float* mel, const long long* mel_lengths, int B, int T, float* wav, void* workspace,
                size_t ws_bytes, cudaStream_t s) {
  const HifiganW& h = ctx->hifigan;
  const ev_hifigan_cfg& c = h.cfg;
  Workspace w(workspace, ws_bytes);
  VocBuffers<ActT> v;
  plan_vocode<ActT>(h, B, T, w, &v);
  if (w.overflow || !workspace) return fail(ctx, EV_ERR_STATE, "ev_vocode: workspace too small");
  ctx->prof_tag = "/voc";
  const RowMask none{nullptr, 0};
  // Ragged batch: tiles that start past (len_b + margin) frames are skipped by the tensor-core kernels; the waveform of
  // item b is bit-identical to the dense computation on [0, len_b * hop) and zero beyond.
  struct RagGuard {
    ev_ctx* c;
    ~RagGuard() { c->rag = RaggedPlanner(); c->prof_scale = 1.0; }
  } guard{ctx};
  const int* lens32 = nullptr;
  const VocMargins margins = vocoder_margins(c);
  if (mel_lengths) {
    EV_LAUNCH(ctx, s, "i64_to_i32", 0, 12.0 * B, i64_to_i32(mel_lengths, v.lens32, B, s));
    lens32 = v.lens32;
    RaggedPlanner& r = ctx->rag;
    r = RaggedPlanner();
    r.lens = lens32; r.B = B; r.margin = margins.pre;
    r.arena = v.rag_arena; r.arena_ints = v.rag_ints;
    r.launch_counter = &ctx->launches;
    if (ctx->dec_side && !ctx->profiling && std::is_same<ActT, bf16>::value) {   // tile lists are built on a side branch as soon as the lengths are there
      r.side = ctx->lane_stream[ev_ctx::kMaxLanes - 2]; r.ready = ctx->side_join;
      EV_CUDA(ctx, cudaEventRecord(ctx->side_fork, s));
      EV_CUDA(ctx, cudaStreamWaitEvent(r.side, ctx->side_fork, 0));
    }
    if (ctx->profiling) {   // algorithmic work = the valid frames only (instrumented eager step: a host copy is fine here)
      std::vector<long long> hl(B);
      EV_CUDA(ctx, cudaMemcpyAsync(hl.data(), mel_lengths, sizeof(long long) * B, cudaMemcpyDeviceToHost, s));
      EV_CUDA(ctx, cudaStreamSynchronize(s));
      double valid = 0.0;
      for (int b = 0; b < B; ++b) valid += (double)std::min<long long>(std::max<long long>(hl[b], 0), T);
      ctx->prof_scale = valid / ((double)B * T);
    }
  }
  EV_LAUNCH(ctx, s, "cf_to_cl", 0, (double)B * T * c.num_mels * (4.0 + sizeof(ActT)),
            (cf_to_cl<ActT>(mel, B, c.num_mels, T, v.mel, c.num_mels, (long long)T * c.num_mels, 1.0f, none, s)));
  int C = c.upsample_initial_channel;
  long long L = T;
  {  // x = conv_pre(mel); the loop's first leaky_relu is fused here
    Epilogue e; e.act = ACT_LRELU; e.slope = kSlope; e.out_act = v.stage_in; e.act_ld = C; e.act_bs = L * C;
    EV_TRY(run_conv<ActT>(ctx, h.conv_pre, v.mel, c.num_mels, (long long)T * c.num_mels, B, T, e, s));
  }
  for (int i = 0; i < c.n_ups; ++i) {
    const int Cin = C;
    const long long Lin = L;
    C = Cin / 2;
    L = Lin * c.upsample_rates[i];
    const long long bs = L * C;
    ctx->rag.rows_per_frame = (int)(Lin / T);   // the transposed conv's GEMM rows are its input rows
    ctx->rag.margin = margins.up[i];
    {  // x = ups[i](leaky_relu(x)) -> fp32 residual stream x0 and its activated operand copy
      Epilogue e; e.out_f32 = v.x0; e.f32_ld = C; e.f32_bs = bs; e.act = ACT_LRELU; e.slope = kSlope;
      e.out_act = v.x0a; e.act_ld = C; e.act_bs = bs;
      EV_TRY(run_conv<ActT>(ctx, h.ups[i], v.stage_in, Cin, Lin * Cin, B, (int)Lin, e, s));
    }
    const bool last_stage = (i == c.n_ups - 1);
    ctx->rag.rows_per_frame = (int)(L / T);
    ctx->rag.margin = margins.stage[i];
    for (int j = 0; j < c.n_kernels; ++j) {   // the MRF branches: sum = mean_j ResBlock_j(x), lrelu(sum) -> next stage's operand
      ResBlockArgs<ActT> a;
      a.C = C; a.k = c.resblock_kernel_sizes[j];
      for (int l = 0; l < 3; ++l) { a.c1[l] = &h.c1[i][j][l]; a.c2[l] = &h.c2[i][j][l]; a.bacc[l] = h.bacc[i][j][l]; }
      a.x = v.x0; a.x_act = v.x0a; a.xb = v.xb; a.xba = v.xba; a.mid = v.mid; a.sum = v.sum;
      a.B = B; a.L = (int)L;
      const bool last_branch = j == c.n_kernels - 1;
      a.mode = last_branch ? (j == 0 ? 3 : 2) : (j == 0 ? 0 : 1);
      a.write_f32 = last_stage ? 1 : 0;   // only conv_post reads the mean in fp32
      a.act_out = (last_branch && !last_stage) ? v.stage_in : nullptr;
      a.inv_n = 1.0f / (float)c.n_kernels; a.slope_out = kSlope;
      a.fused = std::is_same<ActT, bf16>::value && h.fuse_resblocks && c.n_kernels >= 2 && L >= 1024 &&
                resblock_tc_supported(C, a.k, c.resblock_dilation_sizes[j]);
      EV_TRY(run_resblock<ActT>(ctx, a, s));
    }
  }
  if (ctx->rag.side) {   // join the side branch whatever happened on it (a captured graph must not end with unjoined work)
    EV_CUDA(ctx, cudaEventRecord(ctx->rag.ready, ctx->rag.side));
    EV_CUDA(ctx, cudaStreamWaitEvent(s, ctx->rag.ready, 0));
  }
  EV_LAUNCH(ctx, s, "conv_post_tanh", 2.0 * B * (double)L * C * 7, (double)B * L * (4.0 * C + 4.0),
            conv_post_tanh(v.sum, B, (int)L, C, h.post_w, h.post_b, wav, lens32, h.total_up, s));
  return 0;
}
}  // namespace

// host-only: the per-layer margins (mel frames) ev_vocode_ragged uses for this configuration; stage[i] / up[i] for i < n_ups
extern "C" int ev_test_vocoder_margins(const ev_hifigan_cfg* cfg, int32_t* stage, int32_t* up, int32_t* pre) {
  if (!cfg || !stage || !up || !pre || cfg->n_ups <= 0 || cfg->n_ups > 8 || cfg->n_kernels <= 0 || cfg->n_kernels > 4) return EV_ERR_INVALID;
  const VocMargins m = vocoder_margins(*cfg);
  for (int i = 0; i < cfg->n_ups; ++i) { stage[i] = m.stage[i]; up[i] = m.up[i]; }
  *pre = m.pre;
  return EV_OK;
}

extern "C" size_t ev_vocode_workspace_bytes(const ev_ctx* ctx, int B, int T) {
  if (!ctx || !ctx->hifigan.loaded || B <= 0 || T <= 0) return 0;
  Workspace w(nullptr, 0);
  VocBuffers<float> v;
  plan_vocode<float>(ctx->hifigan, B, T, w, &v);
  return w.off + 256;
}

extern "C" int ev_vocode_ragged(ev_ctx* ctx, const float* mel, const int64_t* mel_lengths, int B, int T, int precision, float* wav,
                                void* workspace, size_t workspace_bytes, void* stream) {
  if (!ctx) return EV_ERR_INVALID;
  if (!ctx->hifigan.loaded) return fail(ctx, EV_ERR_STATE, "ev_vocode: hifigan weights not loaded");
  if (!mel || !wav || B <= 0 || T <= 0) return fail(ctx, EV_ERR_INVALID, "ev_vocode: null argument or empty shape");
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t s = as_stream(stream);
  const long long* ml = reinterpret_cast<const long long*>(mel_lengths);
  if (precision == EV_PREC_FP32) return vocode_impl<float>(ctx, mel, ml, B, T, wav, workspace, workspace_bytes, s);
  if (precision == EV_PREC_BF16) return vocode_impl<bf16>(ctx, mel, ml, B, T, wav, workspace, workspace_bytes, s);
  return fail(ctx, EV_ERR_INVALID, "ev_vocode: unknown precision");
}

extern "C" int ev_vocode(ev_ctx* ctx, const float* mel, int B, int T, int precision, float* wav, void* workspace,
                         size_t workspace_bytes, void* stream) {
  return ev_vocode_ragged(ctx, mel, nullptr, B, T, precision, wav, workspace, workspace_bytes, stream);
}
