// Context lifetime, bookkeeping and the single-kernel unit-test hooks of the C ABI (include/emojivoice_b200.h).
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "ctx.cuh"

using namespace ev;

namespace ev {
bool pdl_enabled() {
  static const bool on = []() { const char* v = getenv("EV_PDL"); return !(v && atoi(v) == 0); }();
  return on;
}
}  // namespace ev

namespace {
thread_local std::string g_create_error;
cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
}  // namespace

extern "C" int ev_version(void) { return 100; }

extern "C" const char* ev_last_error(const ev_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int ev_create(ev_ctx** out, int device) {
  if (!out) return EV_ERR_INVALID;
  *out = nullptr;
  int n = 0;
  cudaError_t ce = cudaGetDeviceCount(&n);
  if (ce != cudaSuccess || n == 0) {
    g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(ce);
    return EV_ERR_NO_DEVICE;
  }
  if (device < 0 || device >= n) { g_create_error = "device index out of range"; return EV_ERR_INVALID; }
  cudaDeviceProp prop;
  if ((ce = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) { g_create_error = cudaGetErrorString(ce); return EV_ERR_CUDA; }
  if (prop.major != 10) {
    g_create_error = std::string("emojivoice_b200 needs an sm_100-class GPU (B200); found ") + prop.name + " sm_" +
                     std::to_string(prop.major) + std::to_string(prop.minor) + " -- there is no fallback path";
    return EV_ERR_NO_DEVICE;
  }
  if ((ce = cudaSetDevice(device)) != cudaSuccess) { g_create_error = cudaGetErrorString(ce); return EV_ERR_CUDA; }
  std::string msg;
  if (!conv_tc_init(&msg)) { g_create_error = msg; return EV_ERR_CUDA; }
  ev_ctx* ctx = new ev_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  { const char* v = getenv("EV_ENC_TC"); ctx->enc_tc = !(v && atoi(v) == 0); }
  { const char* v = getenv("EV_DEC_LANES"); if (v) ctx->dec_lanes = std::min(std::max(atoi(v), 1), (int)ev_ctx::kMaxLanes); }
  // lane streams / events are created here: stream creation is not allowed while a caller captures a CUDA graph
  { const char* v = getenv("EV_DEC_SIDE"); ctx->dec_side = !(v && atoi(v) == 0); }
  ce = cudaEventCreateWithFlags(&ctx->lane_fork, cudaEventDisableTiming);
  if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&ctx->side_fork, cudaEventDisableTiming);
  if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&ctx->side_join, cudaEventDisableTiming);
  for (int i = 0; i < ev_ctx::kMaxLanes - 1 && ce == cudaSuccess; ++i) {
    ce = cudaStreamCreateWithFlags(&ctx->lane_stream[i], cudaStreamNonBlocking);
    if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&ctx->lane_join[i], cudaEventDisableTiming);
  }
  if (ce != cudaSuccess) { g_create_error = std::string("lane streams: ") + cudaGetErrorString(ce); delete ctx; return EV_ERR_CUDA; }
  *out = ctx;
  return EV_OK;
}

extern "C" int ev_destroy(ev_ctx* ctx) {
  if (!ctx) return EV_OK;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (void* p : ctx->owned) cudaFree(p);
  for (int i = 0; i < ev_ctx::kMaxLanes - 1; ++i) {
    if (ctx->lane_stream[i]) cudaStreamDestroy(ctx->lane_stream[i]);
    if (ctx->lane_join[i]) cudaEventDestroy(ctx->lane_join[i]);
  }
  if (ctx->lane_fork) cudaEventDestroy(ctx->lane_fork);
  if (ctx->side_fork) cudaEventDestroy(ctx->side_fork);
  if (ctx->side_join) cudaEventDestroy(ctx->side_join);
  delete ctx;
  return EV_OK;
}

extern "C" int64_t ev_launch_count(const ev_ctx* ctx, int reset) {
  if (!ctx) return 0;
  const int64_t v = ctx->launches;
  if (reset) const_cast<ev_ctx*>(ctx)->launches = 0;
  return v;
}

extern "C" int ev_profile_begin(ev_ctx* ctx) {
  if (!ctx) return EV_ERR_INVALID;
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  EV_CUDA(ctx, cudaDeviceSynchronize());
  for (auto& r : ctx->prof) { ctx->event_pool.push_back(r.e0); ctx->event_pool.push_back(r.e1); }
  ctx->prof.clear();
  ctx->profiling = true;
  { const char* d = getenv("EV_PROF_DETAIL"); ctx->prof_detail = d && atoi(d) != 0; }
  return EV_OK;
}

extern "C" int ev_profile_end(ev_ctx* ctx, ev_kernel_stat* out, int max_entries, int* n_out) {
  if (!ctx || !out || !n_out) return EV_ERR_INVALID;
  ctx->profiling = false;
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  EV_CUDA(ctx, cudaDeviceSynchronize());
  const int nk = (int)ctx->kernel_names.size();
  std::vector<ev_kernel_stat> agg(nk);
  for (int i = 0; i < nk; ++i) {
    memset(&agg[i], 0, sizeof(ev_kernel_stat));
    strncpy(agg[i].name, ctx->kernel_names[i].c_str(), sizeof(agg[i].name) - 1);
  }
  for (auto& r : ctx->prof) {
    float ms = 0.0f;
    if (cudaEventElapsedTime(&ms, r.e0, r.e1) == cudaSuccess) {
      agg[r.kid].launches++;
      agg[r.kid].total_ms += ms;
      agg[r.kid].flops += r.flops;
      agg[r.kid].bytes += r.bytes;
    }
    ctx->event_pool.push_back(r.e0);
    ctx->event_pool.push_back(r.e1);
  }
  ctx->prof.clear();
  int n = 0;
  for (int i = 0; i < nk && n < max_entries; ++i)
    if (agg[i].launches > 0) out[n++] = agg[i];
  *n_out = n;
  return EV_OK;
}

// ------------------------------------------------------------------------------------------------ test hooks
extern "C" int ev_test_conv1d(ev_ctx* ctx, const float* x, const float* w, const float* bias, int B, int Cin, int T,
                              int Cout, int K, int stride, int padding, int dilation, int transposed, int precision,
                              float* y, void* stream) {
  if (!ctx || !x || !w || !y) return EV_ERR_INVALID;
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t mark = ctx->owned.size();
  auto release = [&]() {
    cudaStreamSynchronize(s);
    for (size_t i = mark; i < ctx->owned.size(); ++i) cudaFree(ctx->owned[i]);
    ctx->owned.resize(mark);
  };
  ev_tensor tw{}, tb{};
  tw.name = "w"; tw.data = w; tw.ndim = 3;
  tw.shape[0] = transposed ? Cin : Cout; tw.shape[1] = transposed ? Cout : Cin; tw.shape[2] = K;
  tb.name = "b"; tb.data = bias; tb.ndim = 1; tb.shape[0] = Cout;
  ev_tensor list[2] = {tw, tb};
  WeightStore ws(ctx, list, bias ? 2 : 1, s);
  ConvWeights cw;
  int rc = make_conv(ctx, ws, {"w"}, bias ? std::vector<std::string>{"b"} : std::vector<std::string>{}, Cout, Cin, K, stride,
                     padding, dilation, transposed ? CONV_TRANSPOSED : CONV_NORMAL, precision == 2 ? TC_TF32X3 : TC_BF16, &cw);
  if (!rc && precision == 2 && !cw.w_tf32) rc = fail(ctx, EV_ERR_INVALID, "ev_test_conv1d: this shape has no 3xTF32 path");
  if (rc) { release(); return rc; }
  ConvGeom g;
  const int T_out = conv_geometry(cw, B, T, &g);
  void *xa = nullptr, *yo = nullptr;
  const size_t esz = precision == EV_PREC_BF16 ? 2 : 4;
  if ((rc = device_alloc(ctx, (size_t)B * T * Cin * esz, &xa, false, s)) || (rc = device_alloc(ctx, (size_t)B * T_out * Cout * 4, &yo, false, s))) { release(); return rc; }
  Epilogue e;
  e.out_f32 = reinterpret_cast<float*>(yo); e.f32_ld = Cout; e.f32_bs = (long long)T_out * Cout;
  const RowMask none{nullptr, 0};
  cudaError_t ce;
  if (precision == EV_PREC_BF16) {
    ce = cf_to_cl<bf16>(x, B, Cin, T, reinterpret_cast<bf16*>(xa), Cin, (long long)T * Cin, 1.0f, none, s);
    if (ce == cudaSuccess) rc = run_conv<bf16>(ctx, cw, reinterpret_cast<bf16*>(xa), Cin, (long long)T * Cin, B, T, e, s);
  } else if (precision == 2) {
    void* sc = nullptr;
    if ((rc = device_alloc(ctx, (size_t)B * T * Cin * 8, &sc, false, s))) { release(); return rc; }
    ce = cf_to_cl<float>(x, B, Cin, T, reinterpret_cast<float*>(xa), Cin, (long long)T * Cin, 1.0f, none, s);
    const bool keep = ctx->enc_tc;
    ctx->enc_tc = true;
    if (ce == cudaSuccess) rc = run_conv_tf32(ctx, cw, reinterpret_cast<float*>(xa), Cin, (long long)T * Cin, B, T, e, reinterpret_cast<float*>(sc), s);
    ctx->enc_tc = keep;
  } else {
    ce = cf_to_cl<float>(x, B, Cin, T, reinterpret_cast<float*>(xa), Cin, (long long)T * Cin, 1.0f, none, s);
    if (ce == cudaSuccess) rc = run_conv<float>(ctx, cw, reinterpret_cast<float*>(xa), Cin, (long long)T * Cin, B, T, e, s);
  }
  if (ce != cudaSuccess) { release(); return cuda_fail(ctx, ce, "cf_to_cl"); }
  if (rc) { release(); return rc; }
  ce = cl_to_cf(reinterpret_cast<float*>(yo), Cout, (long long)T_out * Cout, B, Cout, T_out, y, 1.0f, 0.0f, s);
  if (ce != cudaSuccess) { release(); return cuda_fail(ctx, ce, "cl_to_cf"); }
  ce = cudaStreamSynchronize(s);
  release();
  if (ce != cudaSuccess) return cuda_fail(ctx, ce, "ev_test_conv1d");
  return EV_OK;
}

namespace {
__global__ void f32_to_bf16_kernel(const float* in, bf16* out, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __float2bfloat16_rn(in[i]);
}
__global__ void bf16_to_f32_kernel(const bf16* in, float* out, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __bfloat162float(in[i]);
}
}  // namespace

// Decoder attention alone: qkv (B, 3*H*64, T) channel-first fp32 [q | k | v sections], y_lengths (B) int64 or NULL.
extern "C" int ev_test_attention(ev_ctx* ctx, const float* qkv, const int64_t* y_lengths, int B, int T, int H, int len_shift,
                                 int precision, float* out, void* stream) {
  if (!ctx || !qkv || !out || B <= 0 || T <= 0 || H <= 0) return EV_ERR_INVALID;
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  const int inner = H * 64;
  const size_t mark = ctx->owned.size();
  auto release = [&]() {
    cudaStreamSynchronize(s);
    for (size_t i = mark; i < ctx->owned.size(); ++i) cudaFree(ctx->owned[i]);
    ctx->owned.resize(mark);
  };
  void *xa = nullptr, *yo = nullptr, *yf = nullptr, *li = nullptr;
  const size_t esz = precision == EV_PREC_BF16 ? 2 : 4;
  int rc;
  if ((rc = device_alloc(ctx, (size_t)B * T * 3 * inner * esz, &xa, false, s)) || (rc = device_alloc(ctx, (size_t)B * T * inner * esz, &yo, false, s)) ||
      (rc = device_alloc(ctx, (size_t)B * T * inner * 4, &yf, false, s)) || (rc = device_alloc(ctx, (size_t)B * 4, &li, false, s))) { release(); return rc; }
  int* lens = nullptr;
  cudaError_t ce = cudaSuccess;
  if (y_lengths) { lens = reinterpret_cast<int*>(li); ce = i64_to_i32(reinterpret_cast<const long long*>(y_lengths), lens, B, s); }
  const RowMask none{nullptr, 0};
  const float scale = 0.125f;
  std::string err;
  if (ce == cudaSuccess && precision == EV_PREC_BF16) {
    ce = cf_to_cl<bf16>(qkv, B, 3 * inner, T, reinterpret_cast<bf16*>(xa), 3 * inner, (long long)T * 3 * inner, 1.0f, none, s);
    AttnTcArgs at;
    at.qkv = reinterpret_cast<bf16*>(xa); at.ld = 3 * inner; at.bs = (long long)T * 3 * inner;
    at.B = B; at.T = T; at.H = H; at.D = 64; at.inner = inner; at.scale = scale; at.lens = lens; at.len_shift = len_shift;
    at.out = reinterpret_cast<bf16*>(yo); at.out_ld = inner; at.out_bs = (long long)T * inner;
    if (ce == cudaSuccess) ce = attention_tc(at, s, &err);
    const long long n = (long long)B * T * inner;
    if (ce == cudaSuccess) { bf16_to_f32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(reinterpret_cast<bf16*>(yo), reinterpret_cast<float*>(yf), n); ce = cudaGetLastError(); }
  } else if (ce == cudaSuccess) {
    ce = cf_to_cl<float>(qkv, B, 3 * inner, T, reinterpret_cast<float*>(xa), 3 * inner, (long long)T * 3 * inner, 1.0f, none, s);
    AttnArgs at;
    const float* q = reinterpret_cast<float*>(xa);
    at.q = q; at.k = q + inner; at.v = q + 2 * inner; at.ld = 3 * inner; at.bs = (long long)T * 3 * inner;
    at.B = B; at.T = T; at.H = H; at.D = 64; at.scale = scale; at.lens = lens; at.len_shift = len_shift; at.mode = 1;
    at.out = yf; at.out_ld = inner; at.out_bs = (long long)T * inner;
    if (ce == cudaSuccess) ce = attention_rows<float>(at, s);
  }
  if (ce == cudaSuccess) ce = cl_to_cf(reinterpret_cast<float*>(yf), inner, (long long)T * inner, B, inner, T, out, 1.0f, 0.0f, s);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
  release();
  if (ce != cudaSuccess) return err.empty() ? cuda_fail(ctx, ce, "ev_test_attention") : fail(ctx, EV_ERR_CUDA, err);
  return EV_OK;
}

// Text-encoder attention alone (text_encoder.py:223-246, head width hd, RoPE on the first hd / 2 features): qkv (B, T, 3*H*hd)
// CHANNEL-LAST fp32 [q | k | v], x_lengths (B) int64 or NULL, out (B, T, H*hd).  impl 0: fp32 CUDA cores (attention.cu,
// hd 64 / 96 / 128), 1: tcgen05 with 3xFP16 split operands (attention_enc_tc.cu, hd 96 / 128).  repeat / avg_us_host as
// ev_test_ff_block.
extern "C" int ev_test_encoder_attention_hd(ev_ctx* ctx, const float* qkv, const int64_t* x_lengths, int B, int T, int H, int hd,
                                            int impl, float* out, int repeat, float* avg_us_host, void* stream) {
  if (!ctx || !qkv || !out || B <= 0 || T <= 0 || H <= 0) return EV_ERR_INVALID;
  if (hd != 96 && hd != 128 && (impl == 1 || hd != 64))
    return fail(ctx, EV_ERR_INVALID, "ev_test_encoder_attention_hd: no kernel for this head width / impl");
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  const int inner = H * hd, rope_dim = hd / 2;
  const size_t mark = ctx->owned.size();
  auto release = [&]() {
    cudaStreamSynchronize(s);
    for (size_t i = mark; i < ctx->owned.size(); ++i) cudaFree(ctx->owned[i]);
    ctx->owned.resize(mark);
  };
  void *li = nullptr, *rc = nullptr, *rs = nullptr;
  int rcode;
  if ((rcode = device_alloc(ctx, (size_t)B * 4, &li, false, s)) || (rcode = device_alloc(ctx, (size_t)T * (rope_dim / 2) * 4, &rc, false, s)) ||
      (rcode = device_alloc(ctx, (size_t)T * (rope_dim / 2) * 4, &rs, false, s))) { release(); return rcode; }
  int* lens = nullptr;
  cudaError_t ce = cudaSuccess;
  if (x_lengths) { lens = reinterpret_cast<int*>(li); ce = i64_to_i32(reinterpret_cast<const long long*>(x_lengths), lens, B, s); }
  if (ce == cudaSuccess) ce = rope_tables(reinterpret_cast<float*>(rc), reinterpret_cast<float*>(rs), T, rope_dim, 10000.0f, s);
  AttnArgs at;
  at.q = qkv; at.k = qkv + inner; at.v = qkv + 2 * inner; at.ld = 3 * inner; at.bs = (long long)T * 3 * inner;
  at.B = B; at.T = T; at.H = H; at.D = hd; at.scale = 1.0f / sqrtf((float)hd); at.lens = lens; at.len_shift = 0; at.mode = 0;
  at.rope_cos = reinterpret_cast<float*>(rc); at.rope_sin = reinterpret_cast<float*>(rs); at.rope_dim = rope_dim;
  at.out = out; at.out_ld = inner; at.out_bs = (long long)T * inner;
  if (impl == 1 && !attention_enc_tc_supported(at)) { release(); return fail(ctx, EV_ERR_INVALID, "ev_test_encoder_attention: shape not supported by the tcgen05 kernel"); }
  auto run = [&]() { return impl == 1 ? attention_enc_tc(at, s) : attention_rows<float>(at, s); };
  if (ce == cudaSuccess) ce = run();
  if (ce == cudaSuccess && repeat > 0 && avg_us_host) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0, s);
    for (int i = 0; i < repeat && ce == cudaSuccess; ++i) ce = run();
    cudaEventRecord(e1, s);
    cudaEventSynchronize(e1);
    float ms = 0.0f;
    cudaEventElapsedTime(&ms, e0, e1);
    *avg_us_host = 1e3f * ms / (float)repeat;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
  }
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
  release();
  if (ce != cudaSuccess) return cuda_fail(ctx, ce, "ev_test_encoder_attention");
  return EV_OK;
}

extern "C" int ev_test_encoder_attention(ev_ctx* ctx, const float* qkv, const int64_t* x_lengths, int B, int T, int H, int impl,
                                         float* out, int repeat, float* avg_us_host, void* stream) {
  return ev_test_encoder_attention_hd(ctx, qkv, x_lengths, B, T, H, 128, impl, out, repeat, avg_us_host, stream);
}

// Fused transformer feed-forward alone (ff_tc.cu): x (B, T, 256) CHANNEL-LAST fp32; w1 (inner, 256), w2 (256, inner) as
// nn.Linear stores them; snake_a = exp(alpha), snake_invb = 1 / (exp(beta) + 1e-9); out (B, T, 256) fp32 (the kernel's
// bf16 result widened).  y_lengths (B) int64 or NULL: rows with (t << len_shift) >= y_lengths[b] come out as zero.
static int test_ff_block(ev_ctx* ctx, const float* x, const float* att, const float* wo, const float* bo, const float* ln_g, const float* ln_b,
                         const float* w1, const float* b1, const float* snake_a, const float* snake_invb, const float* w2, const float* b2,
                         const int64_t* y_lengths, int B, int T, int inner, int len_shift, float* out, int repeat, float* avg_us_host,
                         void* stream);

extern "C" int ev_test_ff_block(ev_ctx* ctx, const float* x, const float* ln_g, const float* ln_b, const float* w1, const float* b1,
                                const float* snake_a, const float* snake_invb, const float* w2, const float* b2,
                                const int64_t* y_lengths, int B, int T, int inner, int len_shift, float* out, int repeat,
                                float* avg_us_host, void* stream) {
  return test_ff_block(ctx, x, nullptr, nullptr, nullptr, ln_g, ln_b, w1, b1, snake_a, snake_invb, w2, b2, y_lengths, B, T, inner, len_shift, out,
                       repeat, avg_us_host, stream);
}

// ff_tc's attention tail mode alone: xr (B, 256, T) CHANNEL-FIRST fp32 residual stream, att (B, T, 128) channel-last fp32 (rounded
// to bf16 inside), wo (256, 128) / bo (256) the out-projection; everything else as ev_test_ff_block.
// out = (x + W2 snake(W1 LN(x) + b1) + b2) * mask with x = xr + att Wo^T + bo.
extern "C" int ev_test_tf_tail(ev_ctx* ctx, const float* xr_cf, const float* att, const float* wo, const float* bo, const float* ln_g,
                               const float* ln_b, const float* w1, const float* b1, const float* snake_a, const float* snake_invb,
                               const float* w2, const float* b2, const int64_t* y_lengths, int B, int T, int inner, int len_shift,
                               float* out, int repeat, float* avg_us_host, void* stream) {
  if (!att || !wo || !bo) return EV_ERR_INVALID;
  return test_ff_block(ctx, xr_cf, att, wo, bo, ln_g, ln_b, w1, b1, snake_a, snake_invb, w2, b2, y_lengths, B, T, inner, len_shift, out, repeat,
                       avg_us_host, stream);
}

static int test_ff_block(ev_ctx* ctx, const float* x, const float* att, const float* wo, const float* bo, const float* ln_g, const float* ln_b,
                         const float* w1, const float* b1, const float* snake_a, const float* snake_invb, const float* w2, const float* b2,
                         const int64_t* y_lengths, int B, int T, int inner, int len_shift, float* out, int repeat, float* avg_us_host,
                         void* stream) {
  if (!ctx || !x || !ln_g || !ln_b || !w1 || !b1 || !snake_a || !snake_invb || !w2 || !b2 || !out || B <= 0 || T <= 0 || inner <= 0)
    return EV_ERR_INVALID;
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  const int D = 256;
  const size_t mark = ctx->owned.size();
  auto release = [&]() {
    cudaStreamSynchronize(s);
    for (size_t i = mark; i < ctx->owned.size(); ++i) cudaFree(ctx->owned[i]);
    ctx->owned.resize(mark);
  };
  ev_tensor t1{}, t2{}, tb1{}, tb2{};
  t1.name = "w1"; t1.data = w1; t1.ndim = 3; t1.shape[0] = inner; t1.shape[1] = D; t1.shape[2] = 1;
  t2.name = "w2"; t2.data = w2; t2.ndim = 3; t2.shape[0] = D; t2.shape[1] = inner; t2.shape[2] = 1;
  tb1.name = "b1"; tb1.data = b1; tb1.ndim = 1; tb1.shape[0] = inner;
  tb2.name = "b2"; tb2.data = b2; tb2.ndim = 1; tb2.shape[0] = D;
  ev_tensor two{}, tbo{};
  two.name = "wo"; two.data = wo; two.ndim = 3; two.shape[0] = D; two.shape[1] = 128; two.shape[2] = 1;
  tbo.name = "bo"; tbo.data = bo; tbo.ndim = 1; tbo.shape[0] = D;
  ev_tensor list[6] = {t1, t2, tb1, tb2, two, tbo};
  WeightStore ws(ctx, list, att ? 6 : 4, s);
  ConvWeights c1, c2, co;
  int rc = make_conv(ctx, ws, {"w1"}, {"b1"}, inner, D, 1, 1, 0, 1, CONV_NORMAL, TC_BF16, &c1);
  if (!rc) rc = make_conv(ctx, ws, {"w2"}, {"b2"}, D, inner, 1, 1, 0, 1, CONV_NORMAL, TC_BF16, &c2);
  if (!rc && att) rc = make_conv(ctx, ws, {"wo"}, {"bo"}, D, 128, 1, 1, 0, 1, CONV_NORMAL, TC_BF16, &co);
  if (!rc && att && !ff_tc_oproj_supported(co)) rc = fail(ctx, EV_ERR_INVALID, "ev_test_tf_tail: out-projection not served by the fused kernel");
  void* att16 = nullptr;
  if (!rc && att) rc = device_alloc(ctx, (size_t)B * T * 128 * 2, &att16, false, s);
  if (!rc && !ff_tc_supported(c1, c2)) rc = fail(ctx, EV_ERR_INVALID, "ev_test_ff_block: shape not served by the fused kernel");
  void *yo = nullptr, *li = nullptr, *tb = nullptr;
  if (!rc) rc = device_alloc(ctx, (size_t)B * T * D * 2, &yo, false, s);
  if (!rc) rc = device_alloc(ctx, (size_t)B * 4, &li, false, s);
  if (!rc) rc = device_alloc(ctx, ((size_t)B * ceil_div(T, 128) + 64) * 4, &tb, false, s);
  if (rc) { release(); return rc; }
  cudaError_t ce = cudaMemsetAsync(yo, 0xff, (size_t)B * T * D * 2, s);   // NaN patterns: every output row must be written
  int* lens = nullptr;
  const int* tiles = nullptr;
  if (ce == cudaSuccess && y_lengths) {
    lens = reinterpret_cast<int*>(li);
    ce = i64_to_i32(reinterpret_cast<const long long*>(y_lengths), lens, B, s);
    const char* v = getenv("EV_FF_RAGGED");
    if (ce == cudaSuccess && !(v && atoi(v) == 0) && B <= kRaggedMaxB) {   // as the decoder does: only tiles with a valid row are computed
      ce = ragged_build_table(lens, B, 0, 1, len_shift, 128, T, reinterpret_cast<int*>(tb), s);
      tiles = reinterpret_cast<int*>(tb);
    }
  }
  FfTcArgs fa;
  if (att) {
    const long long na = (long long)B * T * 128;
    if (ce == cudaSuccess) { f32_to_bf16_kernel<<<(unsigned)((na + 255) / 256), 256, 0, s>>>(att, reinterpret_cast<bf16*>(att16), na); ce = cudaGetLastError(); }
    fa.att = reinterpret_cast<bf16*>(att16); fa.att_ld = 128; fa.att_bs = (long long)T * 128; fa.oproj = &co; fa.xr_cf = x;
  } else {
    fa.x = x;
  }
  fa.ln_g = ln_g; fa.ln_b = ln_b; fa.eps = 1e-5f; fa.ff1 = &c1; fa.ff2 = &c2; fa.snake_a = snake_a; fa.snake_invb = snake_invb;
  fa.out = reinterpret_cast<bf16*>(yo); fa.out_ld = D; fa.out_bs = (long long)T * D; fa.lens = lens; fa.len_shift = len_shift;
  fa.B = B; fa.T = T; fa.tiles = tiles;
  std::string err;
  if (ce == cudaSuccess) ce = ff_tc_launch(fa, s, &err);
  if (ce == cudaSuccess && repeat > 0 && avg_us_host) {   // timing aid: `repeat` more back-to-back launches between two events
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0, s);
    for (int i = 0; i < repeat && ce == cudaSuccess; ++i) ce = ff_tc_launch(fa, s, &err);
    cudaEventRecord(e1, s);
    if (ce == cudaSuccess) ce = cudaEventSynchronize(e1);
    float ms = 0.0f;
    if (ce == cudaSuccess) cudaEventElapsedTime(&ms, e0, e1);
    *avg_us_host = ms * 1e3f / (float)repeat;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
  }
  const long long n = (long long)B * T * D;
  if (ce == cudaSuccess) { bf16_to_f32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(reinterpret_cast<bf16*>(yo), out, n); ce = cudaGetLastError(); }
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
  release();
  if (ce != cudaSuccess) return err.empty() ? cuda_fail(ctx, ce, "ev_test_ff_block") : fail(ctx, EV_ERR_CUDA, err);
  return EV_OK;
}

// Fused ResnetBlock1D (+ pre-LN) alone (resnet_tc.cu).  `weights`: conv1.weight (256, C_in, 3), conv1.bias, gn1.weight, gn1.bias,
// and -- for the full block -- temb (256), conv2.weight (256, 256, 3), conv2.bias, gn2.weight, gn2.bias, res.weight (256, C_in, 1),
// res.bias, ln.weight, ln.bias, named like that.  x (B, C_in, T) channel-first fp32 (masked and rounded to bf16 inside).
// full != 0: out_a = conv2's operand, out_xr = the block's fp32 output, out_n = LayerNorm(out_xr), all (B, T, 256) channel-last
// fp32 (bf16 results widened); full == 0: conv -> GN -> Mish -> mask only, result in out_a.
extern "C" int ev_test_resnet_block(ev_ctx* ctx, const ev_tensor* weights, int n_weights, const float* x, const int64_t* y_lengths,
                                    int B, int T, int C_in, int len_shift, int full, float* out_a, float* out_xr, float* out_n,
                                    int repeat, float* avg_us_host, void* stream) {
  if (!ctx || !weights || !x || !out_a || B <= 0 || T <= 0 || C_in <= 0 || (full && (!out_xr || !out_n))) return EV_ERR_INVALID;
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  const int D = 256;
  const size_t mark = ctx->owned.size();
  auto release = [&]() {
    cudaStreamSynchronize(s);
    for (size_t i = mark; i < ctx->owned.size(); ++i) cudaFree(ctx->owned[i]);
    ctx->owned.resize(mark);
  };
  WeightStore ws(ctx, weights, n_weights, s);
  ConvWeights c1, c2, cr;
  float *g1 = nullptr, *b1 = nullptr, *g2 = nullptr, *b2 = nullptr, *te = nullptr, *lg = nullptr, *lb = nullptr;
  int rc = make_conv(ctx, ws, {"conv1.weight"}, {"conv1.bias"}, D, C_in, 3, 1, 1, 1, CONV_NORMAL, TC_BF16, &c1);
  if (!rc) rc = ws.copy_vec("gn1.weight", D, &g1);
  if (!rc) rc = ws.copy_vec("gn1.bias", D, &b1);
  if (!rc && full) {
    rc = make_conv(ctx, ws, {"conv2.weight"}, {"conv2.bias"}, D, D, 3, 1, 1, 1, CONV_NORMAL, TC_BF16, &c2);
    if (!rc) rc = make_conv(ctx, ws, {"res.weight"}, {"res.bias"}, D, C_in, 1, 1, 0, 1, CONV_NORMAL, TC_BF16, &cr);
    if (!rc) rc = ws.copy_vec("gn2.weight", D, &g2);
    if (!rc) rc = ws.copy_vec("gn2.bias", D, &b2);
    if (!rc) rc = ws.copy_vec("temb", D, &te);
    if (!rc) rc = ws.copy_vec("ln.weight", D, &lg);
    if (!rc) rc = ws.copy_vec("ln.bias", D, &lb);
  }
  if (!rc && !resnet_tc_supported(c1, full ? &c2 : nullptr, full ? &cr : nullptr, B, T))
    rc = fail(ctx, EV_ERR_INVALID, "ev_test_resnet_block: shape not served by the fused kernel (too many tiles for one wave?)");
  const int ld_in = (int)align_up((size_t)C_in, 8);
  const size_t n = (size_t)B * T * D;
  void *xin = nullptr, *ab = nullptr, *nb = nullptr, *li = nullptr;
  if (!rc) rc = device_alloc(ctx, (size_t)B * T * ld_in * 2, &xin, true, s);
  if (!rc) rc = device_alloc(ctx, n * 2, &ab, false, s);
  if (!rc) rc = device_alloc(ctx, n * 2, &nb, false, s);
  if (!rc) rc = device_alloc(ctx, (size_t)B * 4, &li, false, s);
  if (rc) { release(); return rc; }
  cudaError_t ce = cudaMemsetAsync(ab, 0xff, n * 2, s);      // NaN patterns: every output row must be written
  if (ce == cudaSuccess) ce = cudaMemsetAsync(nb, 0xff, n * 2, s);
  if (ce == cudaSuccess && full) ce = cudaMemsetAsync(out_xr, 0xff, n * 4, s);
  int* lens = nullptr;
  if (ce == cudaSuccess && y_lengths) {
    lens = reinterpret_cast<int*>(li);
    ce = i64_to_i32(reinterpret_cast<const long long*>(y_lengths), lens, B, s);
  }
  if (ce == cudaSuccess) ce = cf_to_cl<bf16>(x, B, C_in, T, reinterpret_cast<bf16*>(xin), ld_in, (long long)T * ld_in, 1.0f, RowMask{lens, len_shift}, s);
  ResnetTcArgs ra;
  ra.x = reinterpret_cast<bf16*>(xin); ra.x_ld = ld_in; ra.x_bs = (long long)T * ld_in;
  ra.conv1 = &c1; ra.gn_g1 = g1; ra.gn_b1 = b1;
  if (full) { ra.conv2 = &c2; ra.res = &cr; ra.gn_g2 = g2; ra.gn_b2 = b2; ra.temb = te; ra.ln_g = lg; ra.ln_b = lb; }
  ra.lens = lens; ra.len_shift = len_shift; ra.B = B; ra.T = T;
  ra.a_buf = reinterpret_cast<bf16*>(ab); ra.a_ld = D; ra.a_bs = (long long)T * D;
  ra.n_out = reinterpret_cast<bf16*>(nb);
  void* xcf = nullptr;
  if (full == 2) {                       // the stream channel-first (what ff_tc's tail mode reads); handed back channel-last
    rc = device_alloc(ctx, n * 4, &xcf, false, s);
    if (rc) { release(); return rc; }
    if (ce == cudaSuccess) ce = cudaMemsetAsync(xcf, 0xff, n * 4, s);
    ra.xr_cf = reinterpret_cast<float*>(xcf);
  } else {
    ra.xr = out_xr;
  }
  std::string err;
  auto once = [&]() { return resnet_tc_launch(ra, s, &err); };
  if (ce == cudaSuccess) ce = once();
  if (ce == cudaSuccess && repeat > 0 && avg_us_host) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0, s);
    for (int i = 0; i < repeat && ce == cudaSuccess; ++i) ce = once();
    cudaEventRecord(e1, s);
    if (ce == cudaSuccess) ce = cudaEventSynchronize(e1);
    float ms = 0.0f;
    if (ce == cudaSuccess) cudaEventElapsedTime(&ms, e0, e1);
    *avg_us_host = ms * 1e3f / (float)repeat;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
  }
  if (ce == cudaSuccess) { bf16_to_f32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(reinterpret_cast<bf16*>(ab), out_a, (long long)n); ce = cudaGetLastError(); }
  if (ce == cudaSuccess && full) { bf16_to_f32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(reinterpret_cast<bf16*>(nb), out_n, (long long)n); ce = cudaGetLastError(); }
  if (ce == cudaSuccess && full == 2) ce = cf_to_cl<float>(reinterpret_cast<float*>(xcf), B, D, T, out_xr, D, (long long)T * D, 1.0f, RowMask{nullptr, 0}, s);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
  release();
  if (ce != cudaSuccess) return err.empty() ? cuda_fail(ctx, ce, "ev_test_resnet_block") : fail(ctx, EV_ERR_CUDA, err);
  return EV_OK;
}

namespace {
// (B, C, L) channel-first fp32 -> the vocoder's residual stream (B, L, C) fp32 and its operand lrelu(x, 0.1) as ActT
template <typename ActT>
__global__ void rb_input_kernel(const float* __restrict__ x, int C, int L, long long n, float* __restrict__ xs, ActT* __restrict__ xa) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = (int)(i % C);
  const long long bt = i / C, b = bt / L, t = bt - b * L;
  const float v = x[(b * C + c) * L + t];
  xs[i] = v;
  xa[i] = ActT(v > 0.0f ? v : v * 0.1f);
}

template <typename ActT>
int test_resblock(ev_ctx* ctx, const ev_tensor* weights, int n_weights, int C, int k, const float* x, const float* sum_in, int B, int L, int mode,
                  float inv_n, float slope_out, int write_f32, int want_act, const int64_t* lengths, int rows_per_frame, int margin, int impl,
                  const int32_t* schedule, float* sum, float* act_out, int32_t* report, cudaStream_t s) {
  const size_t mark = ctx->owned.size();
  struct Release {   // frees this call's allocations and leaves the context's ragged planner inactive, on every return path
    ev_ctx* c; cudaStream_t s; size_t mark;
    ~Release() {
      cudaStreamSynchronize(s);
      for (size_t i = mark; i < c->owned.size(); ++i) cudaFree(c->owned[i]);
      c->owned.resize(mark);
      c->rag = RaggedPlanner();
    }
  } release{ctx, s, mark};
  WeightStore ws(ctx, weights, n_weights, s);
  const int dil[3] = {1, 3, 5};
  ConvWeights c1[3], c2[3];
  float* bacc[3] = {};
  EV_TRY(load_resblock(ctx, ws, "", C, k, dil, c1, c2, bacc, s));
  // outputs live `guard` rows inside NaN-filled buffers: a row written before item 0 or after item B-1 is caught below
  const long long n = (long long)B * L * C, guard = 1024LL * C;
  void *xs = nullptr, *xa = nullptr, *sb = nullptr, *ab = nullptr, *xb = nullptr, *xba = nullptr, *mid = nullptr, *li = nullptr, *arena = nullptr;
  EV_TRY(device_alloc(ctx, n * 4, &xs, false, s));
  EV_TRY(device_alloc(ctx, n * sizeof(ActT), &xa, false, s));
  EV_TRY(device_alloc(ctx, (n + 2 * guard) * 4, &sb, false, s));
  EV_TRY(device_alloc(ctx, (n + 2 * guard) * sizeof(ActT), &ab, false, s));
  if (!impl) {
    EV_TRY(device_alloc(ctx, n * 4, &xb, true, s));
    EV_TRY(device_alloc(ctx, n * sizeof(ActT), &xba, true, s));
    EV_TRY(device_alloc(ctx, n * sizeof(ActT), &mid, true, s));
  }
  float* sum_buf = reinterpret_cast<float*>(sb) + guard;
  ActT* act_buf = reinterpret_cast<ActT*>(ab) + guard;
  EV_CUDA(ctx, cudaMemsetAsync(sb, 0xff, (n + 2 * guard) * 4, s));
  EV_CUDA(ctx, cudaMemsetAsync(ab, 0xff, (n + 2 * guard) * sizeof(ActT), s));
  if (mode >= 1) EV_CUDA(ctx, cudaMemcpyAsync(sum_buf, sum_in, n * 4, cudaMemcpyDeviceToDevice, s));
  rb_input_kernel<ActT><<<(unsigned)((n + 255) / 256), 256, 0, s>>>(x, C, L, n, reinterpret_cast<float*>(xs), reinterpret_cast<ActT*>(xa));
  EV_CUDA(ctx, cudaGetLastError());
  if (lengths) {   // as ev_vocode_ragged sets it up: item b needs rows [0, (lengths[b] + margin) * rows_per_frame)
    const size_t arena_ints = 32 * ((size_t)B * ceil_div(L, 128) + 64);
    EV_TRY(device_alloc(ctx, (size_t)B * 4, &li, false, s));
    EV_TRY(device_alloc(ctx, arena_ints * 4, &arena, false, s));
    EV_CUDA(ctx, i64_to_i32(reinterpret_cast<const long long*>(lengths), reinterpret_cast<int*>(li), B, s));
    RaggedPlanner& r = ctx->rag;
    r = RaggedPlanner();
    r.lens = reinterpret_cast<int*>(li); r.B = B; r.margin = margin; r.rows_per_frame = rows_per_frame;
    r.arena = reinterpret_cast<int*>(arena); r.arena_ints = arena_ints;
    r.launch_counter = &ctx->launches;
  }
  ResBlockArgs<ActT> a;
  a.C = C; a.k = k;
  for (int l = 0; l < 3; ++l) { a.c1[l] = &c1[l]; a.c2[l] = &c2[l]; a.bacc[l] = bacc[l]; }
  a.x = reinterpret_cast<float*>(xs); a.x_act = reinterpret_cast<ActT*>(xa);
  a.xb = reinterpret_cast<float*>(xb); a.xba = reinterpret_cast<ActT*>(xba); a.mid = reinterpret_cast<ActT*>(mid);
  a.sum = sum_buf; a.act_out = want_act ? act_buf : nullptr;
  a.B = B; a.L = L; a.mode = mode; a.write_f32 = write_f32; a.inv_n = inv_n; a.slope_out = slope_out;
  a.fused = impl == 1;
  RbSchedule sched;
  if (schedule) { sched.cluster = schedule[0]; sched.occ2 = schedule[1]; sched.wave = schedule[2]; sched.resident = schedule[3]; }
  RbLaunchInfo info;
  a.sched = &sched; a.info = &info;
  EV_TRY(run_resblock<ActT>(ctx, a, s));
  if (report) {
    const int32_t r[9] = {info.cl, info.occ, info.wave, info.resident, info.w_slots, info.n_epi, info.grid, info.Wv, info.total_tiles};
    memcpy(report, r, sizeof r);
  }
  // the rows around the outputs must still hold the fill pattern
  std::vector<uint8_t> hs(guard * 4), ha(guard * sizeof(ActT));
  for (int side = 0; side < 2; ++side) {
    const long long off = side ? guard + n : 0;
    EV_CUDA(ctx, cudaMemcpyAsync(hs.data(), reinterpret_cast<float*>(sb) + off, hs.size(), cudaMemcpyDeviceToHost, s));
    EV_CUDA(ctx, cudaMemcpyAsync(ha.data(), reinterpret_cast<ActT*>(ab) + off, ha.size(), cudaMemcpyDeviceToHost, s));
    EV_CUDA(ctx, cudaStreamSynchronize(s));
    for (uint8_t v : hs) if (v != 0xff) return fail(ctx, EV_ERR_STATE, "ev_test_resblock: sum written outside its (B, L, C) rows");
    for (uint8_t v : ha) if (v != 0xff) return fail(ctx, EV_ERR_STATE, "ev_test_resblock: act_out written outside its (B, L, C) rows");
  }
  EV_CUDA(ctx, cudaMemcpyAsync(sum, sum_buf, n * 4, cudaMemcpyDeviceToDevice, s));
  if (act_out) {
    if constexpr (std::is_same<ActT, bf16>::value) {
      bf16_to_f32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(act_buf, act_out, n);
      EV_CUDA(ctx, cudaGetLastError());
    } else {
      EV_CUDA(ctx, cudaMemcpyAsync(act_out, act_buf, n * 4, cudaMemcpyDeviceToDevice, s));
    }
  }
  EV_CUDA(ctx, cudaStreamSynchronize(s));
  return EV_OK;
}
}  // namespace

// One HiFi-GAN ResBlock1 alone, through the code the vocoder runs (run_resblock, hifigan.cu).  See the header.
extern "C" int ev_test_resblock(ev_ctx* ctx, const ev_tensor* weights, int n_weights, int C, int k, const float* x, const float* sum_in, int B,
                                int L, int mode, float inv_n, float slope_out, int write_f32, int want_act, const int64_t* lengths,
                                int rows_per_frame, int margin, int impl, int precision, const int32_t* schedule, float* sum, float* act_out,
                                int32_t* report, void* stream) {
  if (!ctx || !weights || !x || !sum || B <= 0 || L <= 0 || C <= 0 || C % 8 || k <= 0 || mode < 0 || mode > 2 || (mode >= 1 && !sum_in) ||
      (impl != 0 && impl != 1) || (lengths && (rows_per_frame <= 0 || margin < 0)))
    return EV_ERR_INVALID;
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  if (report) memset(report, 0, 9 * sizeof(int32_t));
  if (precision == EV_PREC_BF16)
    return test_resblock<bf16>(ctx, weights, n_weights, C, k, x, sum_in, B, L, mode, inv_n, slope_out, write_f32, want_act, lengths, rows_per_frame,
                               margin, impl, schedule, sum, act_out, report, s);
  if (precision == EV_PREC_FP32)
    return test_resblock<float>(ctx, weights, n_weights, C, k, x, sum_in, B, L, mode, inv_n, slope_out, write_f32, want_act, lengths, rows_per_frame,
                                margin, impl, schedule, sum, act_out, report, s);
  return fail(ctx, EV_ERR_INVALID, "ev_test_resblock: unknown precision");
}

// One tensor-core conv with its fused epilogue, through run_conv / run_conv_tf32 (see the header).
extern "C" int ev_test_conv_epilogue(ev_ctx* ctx, const ev_conv_epilogue_test* a, void* stream) {
  static_assert(sizeof(TcSchedule) == 8 * sizeof(int32_t) && sizeof(TcLaunchInfo) == 19 * sizeof(int32_t), "the header's int32 arrays");
  if (!ctx || !a) return EV_ERR_INVALID;
  if (a->report_host) memset(a->report_host, 0, sizeof(TcLaunchInfo));
  if (!a->w || !a->x || a->B <= 0 || a->C_in <= 0 || a->T <= 0 || a->C_out <= 0 || a->K <= 0 || a->precision < 1 || a->precision > 3 ||
      (a->ragged_lengths && (a->precision != 1 || a->rows_per_frame <= 0 || a->ragged_margin < 0)))
    return fail(ctx, EV_ERR_INVALID, "ev_test_conv_epilogue: bad arguments");
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t mark = ctx->owned.size();
  struct Release {   // frees this call's allocations and leaves the context's ragged planner inactive, on every return path
    ev_ctx* c; cudaStream_t s; size_t mark;
    ~Release() {
      cudaStreamSynchronize(s);
      for (size_t i = mark; i < c->owned.size(); ++i) cudaFree(c->owned[i]);
      c->owned.resize(mark);
      c->rag = RaggedPlanner();
    }
  } release{ctx, s, mark};
  ev_tensor tw{}, tb{};
  tw.name = "w"; tw.data = a->w; tw.ndim = 3;
  tw.shape[0] = a->transposed ? a->C_in : a->C_out; tw.shape[1] = a->transposed ? a->C_out : a->C_in; tw.shape[2] = a->K;
  tb.name = "b"; tb.data = a->bias; tb.ndim = 1; tb.shape[0] = a->C_out;
  ev_tensor list[2] = {tw, tb};
  WeightStore ws(ctx, list, a->bias ? 2 : 1, s);
  ConvWeights cw;
  EV_TRY(make_conv(ctx, ws, {"w"}, a->bias ? std::vector<std::string>{"b"} : std::vector<std::string>{}, a->C_out, a->C_in, a->K, a->stride,
                   a->pad, a->dilation, a->transposed ? CONV_TRANSPOSED : CONV_NORMAL, a->precision == 1 ? TC_BF16 : TC_TF32X3, &cw));
  if (a->precision >= 2 && !cw.w_tf32) return fail(ctx, EV_ERR_INVALID, "ev_test_conv_epilogue: this layer has no split tensor-core path");
  if (a->precision == 2) cw.w_f16x3 = nullptr;   // the 3xTF32 products (what EV_ENC_SPLIT=tf32 selects)
  if (a->precision == 3 && !cw.w_f16x3) return fail(ctx, EV_ERR_INVALID, "ev_test_conv_epilogue: the 3xFP16 path needs C_in % 64 == 0");
  Epilogue e;
  e.res = a->res; e.res_ld = a->res_ld; e.res_bs = a->res_bs;
  e.res2 = a->res2; e.res2_ld = a->res2_ld; e.res2_bs = a->res2_bs;
  e.out_f32 = a->out_f32; e.f32_ld = a->f32_ld; e.f32_bs = a->f32_bs;
  e.out_act = a->out_act; e.act_ld = a->act_ld; e.act_bs = a->act_bs;
  e.mask_pre = a->mask_pre; e.mask_act = a->mask_act; e.alpha = a->alpha; e.div = a->div; e.f32_is_act = a->f32_is_act;
  e.act = a->act; e.slope = a->slope; e.snake_a = a->snake_a; e.snake_invb = a->snake_invb;
  e.gn_sum = a->gn_sum; e.gn_groups = a->gn_groups;
  if (a->lengths) {
    void* li = nullptr;
    EV_TRY(device_alloc(ctx, (size_t)a->B * 4, &li, false, s));
    EV_CUDA(ctx, i64_to_i32(reinterpret_cast<const long long*>(a->lengths), reinterpret_cast<int*>(li), a->B, s));
    e.mask = RowMask{reinterpret_cast<int*>(li), a->len_shift};
  }
  if (a->ragged_lengths) {   // as ev_vocode_ragged sets it up: item b needs rows [0, (lengths[b] + margin) * rows_per_frame)
    const size_t arena_ints = 32 * ((size_t)a->B * ceil_div(a->T + 1, 128) + 64);
    void *li = nullptr, *arena = nullptr;
    EV_TRY(device_alloc(ctx, (size_t)a->B * 4, &li, false, s));
    EV_TRY(device_alloc(ctx, arena_ints * 4, &arena, false, s));
    EV_CUDA(ctx, i64_to_i32(reinterpret_cast<const long long*>(a->ragged_lengths), reinterpret_cast<int*>(li), a->B, s));
    RaggedPlanner& r = ctx->rag;
    r = RaggedPlanner();
    r.lens = reinterpret_cast<int*>(li); r.B = a->B; r.margin = a->ragged_margin; r.rows_per_frame = a->rows_per_frame;
    r.arena = reinterpret_cast<int*>(arena); r.arena_ints = arena_ints;
    r.launch_counter = &ctx->launches;
  }
  TcSchedule sched;
  if (a->schedule_host) memcpy(&sched, a->schedule_host, sizeof sched);
  TcLaunchInfo info;
  if (a->precision == 1) {
    EV_TRY(run_conv<bf16>(ctx, cw, reinterpret_cast<const bf16*>(a->x), a->x_ld, a->x_bs, a->B, a->T, e, s, &sched, &info));
  } else {
    void* scratch = nullptr;
    EV_TRY(device_alloc(ctx, (size_t)a->B * a->T * a->C_in * 8, &scratch, false, s));
    const bool keep = ctx->enc_tc;
    ctx->enc_tc = true;
    const int rc = run_conv_tf32(ctx, cw, reinterpret_cast<const float*>(a->x), a->x_ld, a->x_bs, a->B, a->T, e, reinterpret_cast<float*>(scratch), s,
                                 false, &sched, &info);
    ctx->enc_tc = keep;
    EV_TRY(rc);
    if (info.grid > 0 && info.split != a->precision - 1)
      return fail(ctx, EV_ERR_INVALID, "ev_test_conv_epilogue: EV_ENC_SPLIT selects the other split path");
  }
  if (info.grid == 0) return fail(ctx, EV_ERR_INVALID, "ev_test_conv_epilogue: the layer ran on the CUDA-core kernel, not conv_tc");
  EV_CUDA(ctx, cudaStreamSynchronize(s));
  if (a->report_host) memcpy(a->report_host, &info, sizeof info);
  return EV_OK;
}

extern "C" int ev_test_resnet_trace(ev_ctx* ctx, uint64_t* out_host, int n) {
  if (!ctx || !out_host || n <= 0) return EV_ERR_INVALID;
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  EV_CUDA(ctx, cudaDeviceSynchronize());
  EV_CUDA(ctx, resnet_tc_read_trace(reinterpret_cast<unsigned long long*>(out_host), n));
  return EV_OK;
}

// diagnostic (EV_TC_TRACE=1): per-CTA clock stamps [n_cta][16] of the most recent conv_tc launch, host buffer
extern "C" int ev_test_conv_trace(ev_ctx* ctx, uint64_t* out_host, int n) {
  if (!ctx || !out_host || n <= 0) return EV_ERR_INVALID;
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  EV_CUDA(ctx, cudaDeviceSynchronize());
  EV_CUDA(ctx, conv_tc_read_trace(reinterpret_cast<unsigned long long*>(out_host), n));
  return EV_OK;
}

extern "C" int ev_test_ff_trace(ev_ctx* ctx, uint64_t* out_host, int n) {
  if (!ctx || !out_host || n <= 0) return EV_ERR_INVALID;
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  EV_CUDA(ctx, cudaDeviceSynchronize());
  EV_CUDA(ctx, ff_tc_read_trace(reinterpret_cast<unsigned long long*>(out_host), n));
  return EV_OK;
}

extern "C" int ev_test_row_sum(ev_ctx* ctx, const float* x, int B, int Tx, float* out, void* stream) {
  if (!ctx || !x || !out) return EV_ERR_INVALID;
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  EV_CUDA(ctx, row_sum_aten(x, B, Tx, out, as_stream(stream)));
  return EV_OK;
}
