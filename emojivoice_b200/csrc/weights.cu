// Weight packing (reference state_dict layouts -> kernel layouts, fp32 + bf16 twins) and the conv dispatch.
#include <cuda_fp16.h>

#include "ctx.cuh"

namespace ev {

int fail(ev_ctx* ctx, int code, const std::string& msg) {
  if (ctx) ctx->err = msg;
  return code;
}
int cuda_fail(ev_ctx* ctx, cudaError_t ce, const char* what) {
  return fail(ctx, EV_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(ce));
}

LaunchScope::LaunchScope(ev_ctx* c, cudaStream_t st, const char* name, double flops, double bytes) : ctx(c), s(st), idx(-1) {
  ctx->launches++;
  if (!ctx->profiling) return;
  int kid = -1;
  for (size_t i = 0; i < ctx->kernel_names.size(); ++i)
    if (ctx->kernel_names[i] == name) { kid = (int)i; break; }
  if (kid < 0) { kid = (int)ctx->kernel_names.size(); ctx->kernel_names.push_back(name); }
  ProfRecord r{kid, flops * ctx->prof_scale, bytes * ctx->prof_scale, nullptr, nullptr};
  for (cudaEvent_t* e : {&r.e0, &r.e1}) {
    if (!ctx->event_pool.empty()) { *e = ctx->event_pool.back(); ctx->event_pool.pop_back(); }
    else if (cudaEventCreate(e) != cudaSuccess) return;
  }
  cudaEventRecord(r.e0, s);
  idx = (int)ctx->prof.size();
  ctx->prof.push_back(r);
}
LaunchScope::~LaunchScope() {
  if (idx >= 0) cudaEventRecord(ctx->prof[idx].e1, s);
}

int device_alloc(ev_ctx* ctx, size_t bytes, void** out, bool zero, cudaStream_t s) {
  void* p = nullptr;
  EV_CUDA(ctx, cudaMalloc(&p, bytes ? bytes : 16));
  ctx->owned.push_back(p);
  if (zero) EV_CUDA(ctx, cudaMemsetAsync(p, 0, bytes ? bytes : 16, s));
  *out = p;
  return 0;
}

WeightStore::WeightStore(ev_ctx* c, const ev_tensor* w, int n, cudaStream_t s) : ctx(c), stream(s) {
  for (int i = 0; i < n; ++i)
    if (w[i].name) by_name[w[i].name] = &w[i];
}

const ev_tensor* WeightStore::get(const std::string& name, std::initializer_list<long long> shape) {
  auto it = by_name.find(name);
  if (it == by_name.end()) { fail(ctx, EV_ERR_MISSING, "missing weight tensor: " + name); return nullptr; }
  const ev_tensor* t = it->second;
  long long want = 1, have = 1;
  for (long long d : shape) want *= d;
  for (int i = 0; i < t->ndim; ++i) have *= t->shape[i];
  if (want != have || t->data == nullptr) {
    fail(ctx, EV_ERR_INVALID, "weight tensor " + name + " has " + std::to_string(have) + " elements, expected " + std::to_string(want));
    return nullptr;
  }
  return t;
}

int WeightStore::copy_vec(const std::string& name, long long n, float** out) {
  const ev_tensor* t = get(name, {n});
  if (!t) return ctx->err.find("missing") == 0 ? EV_ERR_MISSING : EV_ERR_INVALID;
  void* p;
  EV_TRY(device_alloc(ctx, (size_t)n * sizeof(float), &p, false, stream));
  EV_CUDA(ctx, cudaMemcpyAsync(p, t->data, (size_t)n * sizeof(float), cudaMemcpyDeviceToDevice, stream));
  *out = reinterpret_cast<float*>(p);
  return 0;
}

namespace {
// src is (C_out, C_in, K) [nn.Conv1d / nn.Linear with K=1] or (C_in, C_out, K) [nn.ConvTranspose1d].
// Ordinary conv:   GEMM column n = co,              tap j = kernel index j
// Transposed conv: GEMM column n = phase*C_out + co, tap e in {0,1} holds kernel index m = phase + s*e   (k == 2s)
__global__ void pack_conv_kernel(const float* __restrict__ src, int C_out, int C_in, int K, int transposed, int s,
                                 int taps, int n_local, int n_off, float* __restrict__ dst_f32, int N_pad,
                                 bf16* __restrict__ dst_bf16, int N_pad_tc, int K_pad) {
  const long long total = (long long)taps * C_in * n_local;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(idx % n_local);
    const int ci = (int)((idx / n_local) % C_in);
    const int tap = (int)(idx / ((long long)n_local * C_in));
    float v;
    if (!transposed) {
      v = src[((long long)n * C_in + ci) * K + tap];
    } else {
      const int phase = n / C_out, co = n - phase * C_out;
      v = src[((long long)ci * C_out + co) * K + phase + s * tap];
    }
    if (dst_f32) dst_f32[((long long)tap * C_in + ci) * N_pad + n_off + n] = v;
    if (dst_bf16) dst_bf16[((long long)tap * N_pad_tc + n_off + n) * K_pad + ci] = __float2bfloat16_rn(v);
  }
}
// 3xTF32 split of the fp32 weights, K-major: per (tap, n): [w_hi(K32) | w_lo(K32) | w_hi(K32)] with w_hi = w truncated to
// tf32 (10-bit mantissa, low 13 bits cleared) and w_lo = w - w_hi (exact).  Pairs with activations [x_hi | x_hi | x_lo].
__global__ void pack_conv_tf32_kernel(const float* __restrict__ src, int C_out, int C_in, int K, int taps, int n_local, int n_off,
                                      float* __restrict__ dst, int N_pad_tc, int K32) {
  const long long total = (long long)taps * C_in * n_local;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(idx % n_local);
    const int ci = (int)((idx / n_local) % C_in);
    const int tap = (int)(idx / ((long long)n_local * C_in));
    const float v = src[((long long)n * C_in + ci) * K + tap];
    const float hi = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
    const float lo = v - hi;
    float* row = dst + ((long long)tap * N_pad_tc + n_off + n) * (3LL * K32);
    row[ci] = hi;
    row[K32 + ci] = lo;
    row[2 * K32 + ci] = hi;
  }
}

// ---- 3xFP16 split: v = hi + lo with hi = fp16(v), lo = fp16(v - hi): 22 mantissa bits, products x_hi w_hi + x_hi w_lo + x_lo w_hi on
// kind::f16 MMAs (K = 16, half the operand bytes and less than half the tensor time of the tf32 products), fp32 accumulation.
// Values are pre-scaled by powers of two (exact) so that the lo halves are normal fp16 numbers; the epilogue undoes it.
__global__ void absmax_kernel(const float* __restrict__ src, long long n, unsigned int* __restrict__ cell) {
  unsigned int m = 0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    m = max(m, __float_as_uint(fabsf(src[i])));          // non-negative floats order like their bit patterns
  for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(cell, m);
}
__global__ void f16_scale_kernel(const unsigned int* __restrict__ cell, float* __restrict__ scale) {
  const float mx = __uint_as_float(*cell);
  int e = 0;
  if (mx > 0.0f && isfinite(mx)) { int ex; frexpf(mx, &ex); e = 14 - ex; }   // mx = f * 2^ex, f in [0.5, 1): mx * 2^e in [2^13, 2^14)
  e = max(-100, min(100, e));
  scale[0] = ldexpf(1.0f, e);
  scale[1] = ldexpf(1.0f, -e) / kF16ActScale;
}
__global__ void pack_conv_f16x3_kernel(const float* __restrict__ src, int C_out, int C_in, int K, int taps, int n_local, int n_off,
                                       __half* __restrict__ dst, int N_pad_tc, const float* __restrict__ scale) {
  const long long total = (long long)taps * C_in * n_local;
  const float sc = scale[0];
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(idx % n_local);
    const int ci = (int)((idx / n_local) % C_in);
    const int tap = (int)(idx / ((long long)n_local * C_in));
    const float v = src[((long long)n * C_in + ci) * K + tap] * sc;
    const __half hi = __float2half_rn(v);
    const __half lo = __float2half_rn(v - __half2float(hi));
    __half* row = dst + ((long long)tap * N_pad_tc + n_off + n) * (3LL * C_in);
    row[ci] = hi;
    row[C_in + ci] = lo;
    row[2 * C_in + ci] = hi;
  }
}
// x (rows x C fp32, row stride ld) -> [x_hi | x_lo] halves of x * kF16ActScale (rows x 2C): the A operand of the 3xFP16 path
__global__ void split_f16_kernel(const float* __restrict__ x, long long ld, int C, long long rows, __half* __restrict__ out) {
  const long long n4 = rows * (C >> 2);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / (C >> 2);
    const int c = (int)(i - r * (C >> 2)) << 2;
    float4 v = *reinterpret_cast<const float4*>(x + r * ld + c);
    v.x *= kF16ActScale; v.y *= kF16ActScale; v.z *= kF16ActScale; v.w *= kF16ActScale;
    const __half h0 = __float2half_rn(v.x), h1 = __float2half_rn(v.y), h2 = __float2half_rn(v.z), h3 = __float2half_rn(v.w);
    const __half2 ha = __halves2half2(h0, h1), hb = __halves2half2(h2, h3);
    const __half2 la = __floats2half2_rn(v.x - __half2float(h0), v.y - __half2float(h1));
    const __half2 lb = __floats2half2_rn(v.z - __half2float(h2), v.w - __half2float(h3));
    uint2 hv, lv;
    hv.x = *reinterpret_cast<const uint32_t*>(&ha); hv.y = *reinterpret_cast<const uint32_t*>(&hb);
    lv.x = *reinterpret_cast<const uint32_t*>(&la); lv.y = *reinterpret_cast<const uint32_t*>(&lb);
    *reinterpret_cast<uint2*>(out + r * 2 * C + c) = hv;
    *reinterpret_cast<uint2*>(out + r * 2 * C + C + c) = lv;
  }
}

// x (rows x C fp32, row stride ld) -> [x_hi | x_lo] (rows x 2C): the A operand of the 3xTF32 path
__global__ void split_tf32_kernel(const float* __restrict__ x, long long ld, int C, long long rows, float* __restrict__ out) {
  const long long n4 = rows * (C >> 2);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / (C >> 2);
    const int c = (int)(i - r * (C >> 2)) << 2;
    const float4 v = *reinterpret_cast<const float4*>(x + r * ld + c);
    float4 h;
    h.x = __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u); h.y = __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
    h.z = __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u); h.w = __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
    *reinterpret_cast<float4*>(out + r * 2 * C + c) = h;
    *reinterpret_cast<float4*>(out + r * 2 * C + C + c) = make_float4(v.x - h.x, v.y - h.y, v.z - h.z, v.w - h.w);
  }
}
}  // namespace

int make_conv(ev_ctx* ctx, WeightStore& ws, const std::vector<std::string>& weight_names,
              const std::vector<std::string>& bias_names, int c_out_each, int c_in, int ksize, int stride, int pad,
              int dilation, ConvKind kind, int tc_mode, ConvWeights* out) {
  const bool want_bf16 = tc_mode == TC_BF16, want_tf32 = tc_mode == TC_TF32X3 && kind == CONV_NORMAL && stride == 1 && c_in % 32 == 0;
  ConvWeights w;
  const int parts = (int)weight_names.size();
  w.transposed = kind == CONV_TRANSPOSED;
  w.ksize = ksize;
  w.C_in = c_in;
  w.conv_stride = w.transposed ? 1 : stride;
  w.dilation = dilation;
  w.pad = pad;
  int n_local;
  if (w.transposed) {
    if (ksize != 2 * stride || pad >= stride || parts != 1 || dilation != 1)
      return fail(ctx, EV_ERR_INVALID, "transposed conv must have kernel == 2*stride and padding < stride: " + weight_names[0]);
    w.taps = 2;
    w.up_s = stride;
    w.up_p = pad;
    w.C_out = c_out_each;
    n_local = stride * c_out_each;
  } else {
    if (ksize > kMaxTaps) return fail(ctx, EV_ERR_INVALID, "kernel too wide: " + weight_names[0]);
    w.taps = ksize;
    w.C_out = c_out_each * parts;
    n_local = c_out_each;
  }
  w.N = n_local * parts;
  w.N_pad = (w.N == 1) ? 4 : (int)align_up(w.N, 4);
  const int bn = conv_tc_pick_bn(w.N);
  w.N_pad_tc = (int)align_up(w.N, bn);
  w.K_pad = (int)align_up(c_in, 64);
  void* p;
  EV_TRY(device_alloc(ctx, (size_t)w.taps * c_in * w.N_pad * sizeof(float), &p, true, ws.stream));
  w.w_f32 = reinterpret_cast<float*>(p);
  if (want_bf16) {
    EV_TRY(device_alloc(ctx, (size_t)w.taps * w.N_pad_tc * w.K_pad * sizeof(bf16), &p, true, ws.stream));
    w.w_bf16 = reinterpret_cast<bf16*>(p);
  }
  if (want_tf32) {
    w.K32 = (int)align_up(c_in, 32);
    EV_TRY(device_alloc(ctx, (size_t)w.taps * w.N_pad_tc * 3 * w.K32 * sizeof(float), &p, true, ws.stream));
    w.w_tf32 = reinterpret_cast<float*>(p);
  }
  unsigned int* absmax_cell = nullptr;
  if (want_tf32 && c_in % 64 == 0) {        // the 3xFP16 operand set of the same layer
    EV_TRY(device_alloc(ctx, (size_t)w.taps * w.N_pad_tc * 3 * c_in * sizeof(__half), &p, true, ws.stream));
    w.w_f16x3 = p;
    EV_TRY(device_alloc(ctx, 4 * sizeof(float), &p, true, ws.stream));
    w.f16_scale = reinterpret_cast<float*>(p);
    absmax_cell = reinterpret_cast<unsigned int*>(w.f16_scale + 2);
    for (int i = 0; i < parts; ++i) {
      const ev_tensor* t = ws.get(weight_names[i], {(long long)c_out_each, (long long)c_in, (long long)ksize});
      if (!t) return ctx->err.rfind("missing", 0) == 0 ? EV_ERR_MISSING : EV_ERR_INVALID;
      const long long n = (long long)c_out_each * c_in * ksize;
      absmax_kernel<<<(int)std::min<long long>(1024, ceil_div_ll(n, 256)), 256, 0, ws.stream>>>(t->data, n, absmax_cell);
      EV_CUDA(ctx, cudaGetLastError());
    }
    f16_scale_kernel<<<1, 1, 0, ws.stream>>>(absmax_cell, w.f16_scale);
    EV_CUDA(ctx, cudaGetLastError());
  }
  for (int i = 0; i < parts; ++i) {
    const ev_tensor* t = ws.get(weight_names[i], {(long long)c_out_each, (long long)c_in, (long long)ksize});
    if (!t) return ctx->err.rfind("missing", 0) == 0 ? EV_ERR_MISSING : EV_ERR_INVALID;
    const long long total = (long long)w.taps * c_in * n_local;
    const int blocks = (int)std::min<long long>(4096, ceil_div_ll(total, 256));
    pack_conv_kernel<<<blocks, 256, 0, ws.stream>>>(t->data, c_out_each, c_in, ksize, w.transposed, stride, w.taps,
                                                    n_local, i * n_local, w.w_f32, w.N_pad, w.w_bf16, w.N_pad_tc, w.K_pad);
    EV_CUDA(ctx, cudaGetLastError());
    if (w.w_tf32) {
      pack_conv_tf32_kernel<<<blocks, 256, 0, ws.stream>>>(t->data, c_out_each, c_in, ksize, w.taps, n_local, i * n_local, w.w_tf32,
                                                           w.N_pad_tc, w.K32);
      EV_CUDA(ctx, cudaGetLastError());
    }
    if (w.w_f16x3) {
      pack_conv_f16x3_kernel<<<blocks, 256, 0, ws.stream>>>(t->data, c_out_each, c_in, ksize, w.taps, n_local, i * n_local,
                                                            reinterpret_cast<__half*>(w.w_f16x3), w.N_pad_tc, w.f16_scale);
      EV_CUDA(ctx, cudaGetLastError());
    }
  }
  if (!bias_names.empty()) {
    if ((int)bias_names.size() != parts) return fail(ctx, EV_ERR_INVALID, "bias list does not match weight list");
    EV_TRY(device_alloc(ctx, (size_t)align_up(w.C_out, 4) * sizeof(float), &p, true, ws.stream));
    w.bias = reinterpret_cast<float*>(p);
    for (int i = 0; i < parts; ++i) {
      const ev_tensor* t = ws.get(bias_names[i], {(long long)c_out_each});
      if (!t) return ctx->err.rfind("missing", 0) == 0 ? EV_ERR_MISSING : EV_ERR_INVALID;
      EV_CUDA(ctx, cudaMemcpyAsync(w.bias + (size_t)i * c_out_each, t->data, (size_t)c_out_each * sizeof(float),
                                   cudaMemcpyDeviceToDevice, ws.stream));
    }
  }
  *out = w;
  return 0;
}

int conv_geometry(const ConvWeights& w, int B, int T_in, ConvGeom* g) {
  g->B = B;
  g->N = w.N;
  g->C_in = w.C_in;
  g->taps = w.taps;
  g->T_in = T_in;
  g->conv_stride = w.conv_stride;
  int T_out;
  if (w.transposed) {
    // t_out + p = s*r + phase,  phase in [0,s);  tap e reads input row r - e  (weights.cu pack_conv_kernel)
    g->tap_off[0] = 0;
    g->tap_off[1] = -1;
    g->M = T_in + 1;
    T_out = (T_in - 1) * w.up_s - 2 * w.up_p + w.ksize;
  } else {
    for (int j = 0; j < w.taps; ++j) g->tap_off[j] = j * w.dilation - w.pad;
    T_out = (T_in + 2 * w.pad - w.dilation * (w.ksize - 1) - 1) / w.conv_stride + 1;
    g->M = T_out;
  }
  return T_out;
}

template <typename ActT>
int run_conv(ev_ctx* ctx, const ConvWeights& w, const ActT* x, long long x_ld, long long x_bs, int B, int T_in, Epilogue e,
             cudaStream_t s, const TcSchedule* sched, TcLaunchInfo* info) {
  ConvGeom g;
  const int T_out = conv_geometry(w, B, T_in, &g);
  e.bias = w.bias;
  e.T_out = T_out;
  e.phase_cout = w.transposed ? w.C_out : w.N;
  e.up_s = w.transposed ? w.up_s : 1;
  e.up_p = w.transposed ? w.up_p : 0;
  // algorithmic work of this launch: valid multiply-adds only (padding, polyphase zero taps excluded)
  const double taps_eff = w.transposed ? (double)w.ksize / w.up_s : (double)w.taps;
  const double flops = 2.0 * B * (double)T_out * w.C_out * taps_eff * w.C_in;
  const double esz = sizeof(ActT);
  double bytes = (double)B * T_in * w.C_in * esz + (double)w.taps * w.N * w.C_in * esz;
  if (e.out_f32) bytes += 4.0 * B * T_out * w.C_out;
  if (e.out_act) bytes += esz * B * T_out * w.C_out;
  if (e.res) bytes += 4.0 * B * T_out * w.C_out;
  if (e.res2) bytes += 4.0 * B * T_out * w.C_out;
  cudaError_t ce;
  if constexpr (std::is_same<ActT, float>::value) {
    const std::string nm = std::string("conv_simt_f32") + ctx->prof_tag;
    { LaunchScope ls(ctx, s, nm.c_str(), flops, bytes); ce = conv_simt_launch(g, x, x_ld, x_bs, w, e, s); }
    if (ce != cudaSuccess) return cuda_fail(ctx, ce, "conv_simt_launch");
  } else {
    if (!w.w_bf16) return fail(ctx, EV_ERR_STATE, "layer has no bf16 weights");
    std::string msg;
    static const char* names[4] = {"conv_tc_bn32", "conv_tc_bn64", "conv_tc_bn128", "conv_tc_bn256"};
    const int bn = conv_tc_pick_bn(w.N);
    std::string nm = std::string(names[bn == 32 ? 0 : bn == 64 ? 1 : bn == 128 ? 2 : 3]) + ctx->prof_tag;
    if (ctx->profiling && ctx->prof_detail) {   // EV_PROF_DETAIL=1: one class per layer shape
      char buf[64];
      snprintf(buf, sizeof buf, " c%d n%d k%d d%d m%d", w.C_in, w.N, w.taps, w.dilation, g.M);
      nm += buf;
    }
    { LaunchScope ls(ctx, s, nm.c_str(), flops, bytes); ce = conv_tc_launch(g, x, x_ld, x_bs, 0, w, e, s, &msg, ctx->rag.active() ? &ctx->rag : nullptr, sched, info); }
    if (ce == cudaErrorInvalidValue && !msg.empty()) return fail(ctx, EV_ERR_INVALID, msg);
    if (ce != cudaSuccess) return fail(ctx, EV_ERR_CUDA, "conv_tc_launch: " + (msg.empty() ? std::string(cudaGetErrorString(ce)) : msg));
  }
  return 0;
}
// fp32-accurate convolution on the tensor cores (3xTF32): x is split into [hi | lo] in `scratch` (B*T_in*2*C_in floats),
// then one tcgen05 GEMM over the concatenated K does x_hi*w_hi + x_hi*w_lo + x_lo*w_hi with fp32 accumulation.
// Falls back to the CUDA-core kernel when the layer has no split weights or the tile path cannot serve the epilogue.
bool enc_split_f16() {
  static const bool use_f16 = []() { const char* v = getenv("EV_ENC_SPLIT"); return !(v && std::string(v) == "tf32"); }();
  return use_f16;
}

int run_conv_tf32(ev_ctx* ctx, const ConvWeights& w, const float* x, long long x_ld, long long x_bs, int B, int T_in, Epilogue e,
                  float* scratch, cudaStream_t s, bool presplit, const TcSchedule* sched, TcLaunchInfo* info) {
  const bool aligned = (e.f32_ld % 4 == 0) && (e.f32_bs % 4 == 0) && (e.act_ld % 4 == 0) && (e.res_ld % 4 == 0) && w.N % 4 == 0;
  const bool act_ok = e.act == ACT_NONE || e.act == ACT_RELU || e.act == ACT_LRELU;
  if (!w.w_tf32 || !scratch || x_bs != (long long)T_in * x_ld || !aligned || !act_ok || (e.out_act && e.out_f32) || !ctx->enc_tc ||
      conv_tc_pick_bn(w.N) != 128)   // two-level accumulation is built for 128-wide tiles (one 32 x 32 block per epilogue warp)
    return run_conv<float>(ctx, w, x, x_ld, x_bs, B, T_in, e, s);
  ConvGeom g;
  const int T_out = conv_geometry(w, B, T_in, &g);
  e.bias = w.bias;
  e.T_out = T_out;
  e.phase_cout = w.N;
  e.up_s = 1;
  e.up_p = 0;
  if (e.out_act) {   // the fp32 graph's "activated" output becomes the fp32 output of the tensor-core epilogue
    e.out_f32 = reinterpret_cast<float*>(e.out_act); e.f32_ld = e.act_ld; e.f32_bs = e.act_bs; e.f32_is_act = 1;
    e.out_act = nullptr;
  }
  const long long rows = (long long)B * T_in;
  const double flops = 2.0 * B * (double)T_out * w.C_out * w.taps * w.C_in;
  const double bytes = 4.0 * (rows * w.C_in + (double)w.taps * w.N * w.C_in + (double)B * T_out * w.C_out * (e.res ? 2 : 1));
  // EV_ENC_SPLIT=tf32: the 3xTF32 products (round 1); default: 3xFP16 where the layer has that operand set
  const int split = (enc_split_f16() && w.w_f16x3) ? 2 : 1;
  if (!(presplit && split == 2)) {
    const int blocks = (int)std::min<long long>(2048, ceil_div_ll(rows * (w.C_in / 4), 256));
    cudaError_t ce;
    if (split == 2) {
      LaunchScope ls(ctx, s, "split_f16", 0, 8.0 * rows * w.C_in);
      split_f16_kernel<<<blocks, 256, 0, s>>>(x, x_ld, w.C_in, rows, reinterpret_cast<__half*>(scratch));
      ce = cudaGetLastError();
    } else {
      LaunchScope ls(ctx, s, "split_tf32", 0, 12.0 * rows * w.C_in); split_tf32_kernel<<<blocks, 256, 0, s>>>(x, x_ld, w.C_in, rows, scratch); ce = cudaGetLastError();
    }
    if (ce != cudaSuccess) return cuda_fail(ctx, ce, "split");
  }
  std::string msg;
  cudaError_t ce;
  std::string nm = std::string(split == 2 ? "conv_tc_f16x3" : "conv_tc_tf32x3") + ctx->prof_tag;
  if (ctx->profiling && ctx->prof_detail) {   // EV_PROF_DETAIL=1: one class per layer shape
    char buf[64];
    snprintf(buf, sizeof buf, " c%d n%d k%d m%d", w.C_in, w.N, w.taps, g.M);
    nm += buf;
  }
  { LaunchScope ls(ctx, s, nm.c_str(), flops, bytes); ce = conv_tc_launch(g, scratch, 2LL * w.C_in, (long long)T_in * 2 * w.C_in, split, w, e, s, &msg, nullptr, sched, info); }
  if (ce == cudaErrorInvalidValue && !msg.empty()) return fail(ctx, EV_ERR_INVALID, msg);
  if (ce != cudaSuccess) return fail(ctx, EV_ERR_CUDA, "conv_tc_launch(tf32x3): " + (msg.empty() ? std::string(cudaGetErrorString(ce)) : msg));
  return 0;
}

template int run_conv<float>(ev_ctx*, const ConvWeights&, const float*, long long, long long, int, int, Epilogue, cudaStream_t, const TcSchedule*,
                             TcLaunchInfo*);
template int run_conv<bf16>(ev_ctx*, const ConvWeights&, const bf16*, long long, long long, int, int, Epilogue, cudaStream_t, const TcSchedule*,
                            TcLaunchInfo*);

}  // namespace ev
