// Coalesced / vectorised / warp-shuffle kernels around the GEMMs: layout glue, embeddings, LayerNorm, GroupNorm,
// Mish, the decoder input pack, the sinusoidal time embedding and HiFi-GAN's conv_post+tanh tail.
#include <cstdlib>
#include <type_traits>

#include "kernels.cuh"

namespace ev {
namespace {

// ---------------------------------------------------------------------------------------------- transposes
template <typename OutT>
__global__ void cf_to_cl_kernel(const float* __restrict__ in, int C, int T, OutT* __restrict__ out, long long out_ld,
                                long long out_bs, float scale, RowMask mask) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const float* inb = in + (long long)b * C * T;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, t = t0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && t < T) ? inb[(long long)c * T + t] : 0.0f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int t = t0 + i, c = c0 + threadIdx.x;
    if (t < T && c < C) out[b * out_bs + (long long)t * out_ld + c] = from_float<OutT>(tile[threadIdx.x][i] * scale * mask.at(b, t));
  }
}

__global__ void cl_to_cf_kernel(const float* __restrict__ in, long long in_ld, long long in_bs, int C, int T,
                                float* __restrict__ out, float mul, float add) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int t = t0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && t < T) ? in[b * in_bs + (long long)t * in_ld + c] : 0.0f;
  }
  __syncthreads();
  float* outb = out + (long long)b * C * T;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, t = t0 + threadIdx.x;
    if (c < C && t < T) outb[(long long)c * T + t] = tile[threadIdx.x][i] * mul + add;
  }
}

__global__ void i64_to_i32_kernel(const long long* in, int* out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (int)in[i];
}

struct Vals32 { float v[32]; };
__global__ void upload_kernel(float* dst, Vals32 vals, int n) {
  if ((int)threadIdx.x < n) dst[threadIdx.x] = vals.v[threadIdx.x];
}
struct Words { uint32_t w[kUploadWords]; };
__global__ void upload_words_kernel(uint32_t* dst, Words words, int n) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = words.w[i];
}

// ---------------------------------------------------------------------------------------------- embeddings
__global__ void embed_tokens_kernel(const long long* __restrict__ ids, const float* __restrict__ emb, int Tx, int C,
                                    int n_vocab, float scale, RowMask mask, float* __restrict__ out, long long out_ld,
                                    long long* flags) {
  const int row = blockIdx.x, b = row / Tx, t = row - b * Tx;
  long long id = ids[row];
  const float m = mask.at(b, t);
  if ((id < 0 || id >= n_vocab) && flags && threadIdx.x == 0) atomicOr(reinterpret_cast<unsigned long long*>(flags), 1ull);
  id = id < 0 ? 0 : (id >= n_vocab ? n_vocab - 1 : id);
  for (int c = threadIdx.x; c < C; c += blockDim.x) out[(long long)row * out_ld + c] = emb[id * C + c] * scale * m;
}

__global__ void embed_speakers_kernel(const long long* ids, const float* table, int dim, int n_spks, float* out, long long* flags) {
  const int b = blockIdx.x;
  long long id = ids[b];
  if ((id < 0 || id >= n_spks) && flags && threadIdx.x == 0) atomicOr(reinterpret_cast<unsigned long long*>(flags), 2ull);
  id = id < 0 ? 0 : (id >= n_spks ? n_spks - 1 : id);
  for (int c = threadIdx.x; c < dim; c += blockDim.x) out[b * dim + c] = table[id * dim + c];
}

__global__ void fill_speaker_kernel(const float* spk, int T, int dim, RowMask mask, float* buf, long long ld, int c0) {
  const int row = blockIdx.x, b = row / T, t = row - b * T;
  const float m = mask.at(b, t);
  for (int c = threadIdx.x; c < dim; c += blockDim.x) buf[(long long)row * ld + c0 + c] = spk[b * dim + c] * m;
}

// ---------------------------------------------------------------------------------------------- LayerNorm (warp per row)
template <typename ActT, int VPL>  // VPL = ceil(C/32) values per lane
__global__ void __launch_bounds__(256) layer_norm_kernel(LnArgs a) {
  pdl_trigger();
  pdl_wait();
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int rows = a.B * a.T;
  if (warp >= rows) return;
  const int b = warp / a.T, t = warp - b * a.T;
  const float* x = a.x + (long long)warp * a.x_ld;
  const float* ad = a.add ? a.add + (long long)warp * a.add_ld : nullptr;
  float v[VPL];
  float sum = 0.0f;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int c = lane + 32 * i;
    float xv = 0.0f;
    if (c < a.C) {
      xv = x[c];
      if (ad) xv += ad[c];
      if (a.pre_relu) xv = fmaxf(xv, 0.0f);
    }
    v[i] = xv;
    sum += xv;
  }
  const float mean = warp_sum(sum) / (float)a.C;
  float sq = 0.0f;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int c = lane + 32 * i;
    const float d = (c < a.C) ? v[i] - mean : 0.0f;
    sq += d * d;
  }
  const float var = warp_sum(sq) / (float)a.C;
  const float rstd = 1.0f / sqrtf(var + a.eps);
  const float m = a.mask.at(b, t);
  ActT* oa = a.out_act ? reinterpret_cast<ActT*>(a.out_act) + (long long)warp * a.act_ld : nullptr;
  float* of = a.out_f32 ? a.out_f32 + (long long)warp * a.f32_ld : nullptr;
  __half* sp = a.split ? reinterpret_cast<__half*>(a.split) + (long long)warp * 2 * a.C : nullptr;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int c = lane + 32 * i;
    if (c < a.C) {
      float y = (v[i] - mean) * rstd * a.gamma[c] + a.beta[c];
      if (a.post_relu) y = fmaxf(y, 0.0f);
      y *= m;
      if (of) of[c] = y;
      if (oa) oa[c] = from_float<ActT>(y);
      if (sp) {   // exactly what split_f16_kernel computes from the stored value
        const float ys = y * kF16ActScale;
        const __half hi = __float2half_rn(ys);
        sp[c] = hi;
        sp[a.C + c] = __float2half_rn(ys - __half2float(hi));
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------- time embedding
__global__ void time_sinusoid_kernel(const float* t_steps, int n, int dim, float* out) {
  const int s = blockIdx.x, half = dim / 2;
  // decoder.py:23-26: exp(arange(half) * -(log(1e4)/(half-1))), then (1000*t)*freq, all in float32
  const float neg = (float)(-(log(10000.0) / (double)(half - 1)));
  const float tt = __fmul_rn(1000.0f, t_steps[s]);
  for (int i = threadIdx.x; i < half; i += blockDim.x) {
    const float freq = (float)exp((double)__fmul_rn((float)i, neg));
    const float arg = __fmul_rn(tt, freq);
    out[s * dim + i] = (float)sin((double)arg);
    out[s * dim + half + i] = (float)cos((double)arg);
  }
}

template <typename ActT>
__global__ void decoder_pack_kernel(const float* __restrict__ z, const float* __restrict__ mu, const float* __restrict__ spk,
                                    int F, int S, int T, float temperature, const float* __restrict__ temperatures,
                                    RowMask mask, float* __restrict__ x_state, ActT* __restrict__ xin, long long xin_ld) {
  // one block per (b, 32-frame tile): transposes z and mu through shared memory
  extern __shared__ float sh[];  // [2][F][33]
  const int b = blockIdx.y, t0 = blockIdx.x * 32;
  if (temperatures) temperature = temperatures[b];
  float* zs = sh;
  float* ms = sh + F * 33;
  for (int idx = threadIdx.x; idx < F * 32; idx += blockDim.x) {
    const int c = idx >> 5, tt = idx & 31, t = t0 + tt;
    const long long g = ((long long)b * F + c) * T + t;
    zs[c * 33 + tt] = t < T ? z[g] * temperature : 0.0f;
    ms[c * 33 + tt] = t < T ? mu[g] : 0.0f;
  }
  __syncthreads();
  const int C = 2 * F + S;
  for (int idx = threadIdx.x; idx < 32 * C; idx += blockDim.x) {
    const int tt = idx / C, c = idx - tt * C, t = t0 + tt;
    if (t >= T) continue;
    const float m = mask.at(b, t);
    float v;
    if (c < F) {
      v = zs[c * 33 + tt];
      x_state[((long long)b * T + t) * F + c] = v;
    } else if (c < 2 * F) {
      v = ms[(c - F) * 33 + tt];
    } else {
      v = spk[b * S + (c - 2 * F)];
    }
    xin[((long long)b * T + t) * xin_ld + c] = from_float<ActT>(v * m);
  }
}

// ---------------------------------------------------------------------------------------------- GroupNorm
constexpr int GN_ROWS = 32;  // frames per statistics block
// partial[b][chunk][group][2] (sum, sum of squares) in double; blockDim = C threads (C <= 1024, 32 ch per group)
__global__ void gn_stats_kernel(const float* __restrict__ x, int T, int C, int cpg, double* __restrict__ partial) {
  const int b = blockIdx.y, chunk = blockIdx.x, c = threadIdx.x;
  const int t0 = chunk * GN_ROWS, t1 = min(T, t0 + GN_ROWS);
  float s = 0.0f, q = 0.0f;
  const float* xb = x + ((long long)b * T) * C;
  for (int t = t0; t < t1; ++t) {
    const float v = xb[(long long)t * C + c];
    s += v;
    q += v * v;
  }
  // reduce over the cpg channels of the group (cpg is a power of two <= 32, groups are lane-aligned)
  double ds = (double)s, dq = (double)q;
  for (int o = cpg >> 1; o > 0; o >>= 1) {
    ds += __shfl_xor_sync(0xffffffffu, ds, o);
    dq += __shfl_xor_sync(0xffffffffu, dq, o);
  }
  if ((c % cpg) == 0) {
    const int g = c / cpg, G = C / cpg;
    double* p = partial + (((long long)b * gridDim.x + chunk) * G + g) * 2;
    p[0] = ds;
    p[1] = dq;
  }
}

// Mish for the bf16-operand path: x*tanh(softplus(x)) = x*w/(w+2) with w = e^x (e^x + 2); one ex2 + one fast divide
// (relative error ~1e-6, far inside the bf16 tolerance).  The fp32 parity path keeps the exact formulation.
template <typename ActT> __device__ __forceinline__ float mish_sel(float x) { return mish_f(x); }
template <> __device__ __forceinline__ float mish_sel<bf16>(float x) {
  const float n = __expf(fminf(x, 20.0f));
  const float w = n * (n + 2.0f);
  return x > 20.0f ? x : x * __fdividef(w, w + 2.0f);
}

template <typename ActT> __device__ __forceinline__ void store_act4(ActT* p, float4 v);
template <> __device__ __forceinline__ void store_act4<float>(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
template <> __device__ __forceinline__ void store_act4<bf16>(bf16* p, float4 v) {
  __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
  uint2 pk;
  pk.x = *reinterpret_cast<uint32_t*>(&lo);
  pk.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(p) = pk;
}

constexpr int GN_APPLY_ROWS = 4;   // rows per warp

template <typename ActT, int V4>
__global__ void __launch_bounds__(256) gn_apply_kernel(GnApplyArgs a) {
  pdl_trigger();
  pdl_wait();
  // warp per (b,t) row, GN_APPLY_ROWS rows per warp; lane owns the float4 channel groups 4*(lane + 32*i), each inside
  // one GroupNorm group (channels-per-group is a multiple of 4)
  extern __shared__ float stat[];  // [G][2] mean, rstd for this block's batch item
  const int b = blockIdx.y;
  const int G = a.groups, cpg = a.C / G;
  if ((int)threadIdx.x < G) {
    double s = 0.0, q = 0.0;
    for (int ch = 0; ch < a.n_chunks; ++ch) {
      const double* p = a.partial + (((long long)b * a.n_chunks + ch) * G + threadIdx.x) * 2;
      s += p[0];
      q += p[1];
    }
    const double n = (double)cpg * (double)a.T;
    const double mean = s / n;
    double var = q / n - mean * mean;
    if (var < 0.0) var = 0.0;
    stat[2 * threadIdx.x] = (float)mean;
    stat[2 * threadIdx.x + 1] = (float)(1.0 / sqrt(var + (double)a.eps));
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // per-lane constants of its channel groups: scale = rstd*gamma, shift = beta - mean*rstd*gamma
  float4 sc[V4], sh[V4], te[V4], lg[V4], lb[V4];
#pragma unroll
  for (int i = 0; i < V4; ++i) {
    const int c = 4 * (lane + 32 * i);
    sc[i] = sh[i] = te[i] = lg[i] = lb[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < a.C) {
      const int g = c / cpg;
      const float mean = stat[2 * g], rstd = stat[2 * g + 1];
      const float4 ga = *reinterpret_cast<const float4*>(a.gamma + c), be = *reinterpret_cast<const float4*>(a.beta + c);
      sc[i] = make_float4(rstd * ga.x, rstd * ga.y, rstd * ga.z, rstd * ga.w);
      sh[i] = make_float4(be.x - mean * sc[i].x, be.y - mean * sc[i].y, be.z - mean * sc[i].z, be.w - mean * sc[i].w);
      if (a.temb) te[i] = *reinterpret_cast<const float4*>(a.temb + b * a.temb_bs + c);
      if (a.out_ln) { lg[i] = *reinterpret_cast<const float4*>(a.ln_gamma + c); lb[i] = *reinterpret_cast<const float4*>(a.ln_beta + c); }
    }
  }
  const int t_base = (blockIdx.x * (blockDim.x >> 5) + warp) * GN_APPLY_ROWS;
#pragma unroll 1
  for (int rr = 0; rr < GN_APPLY_ROWS; ++rr) {
    const int t = t_base + rr;
    if (t >= a.T) return;
    const long long row = (long long)b * a.T + t;
    const float* x = a.x + row * a.C;
    const float m = a.mask.at(b, t);
    float4 y[V4];
    float sum = 0.0f;
#pragma unroll
    for (int i = 0; i < V4; ++i) {
      const int c = 4 * (lane + 32 * i);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c < a.C) {
        const float4 xv = *reinterpret_cast<const float4*>(x + c);
        // same operation order as the reference: ((x - mean) * rstd) * gamma + beta is refactored only in bf16 mode
        if (sizeof(ActT) == 4) {
          const int g = c / cpg;
          const float mean = stat[2 * g], rstd = stat[2 * g + 1];
          const float4 ga = *reinterpret_cast<const float4*>(a.gamma + c), be = *reinterpret_cast<const float4*>(a.beta + c);
          v.x = (xv.x - mean) * rstd * ga.x + be.x; v.y = (xv.y - mean) * rstd * ga.y + be.y;
          v.z = (xv.z - mean) * rstd * ga.z + be.z; v.w = (xv.w - mean) * rstd * ga.w + be.w;
        } else {
          v.x = fmaf(xv.x, sc[i].x, sh[i].x); v.y = fmaf(xv.y, sc[i].y, sh[i].y);
          v.z = fmaf(xv.z, sc[i].z, sh[i].z); v.w = fmaf(xv.w, sc[i].w, sh[i].w);
        }
        v.x = mish_sel<ActT>(v.x) * m; v.y = mish_sel<ActT>(v.y) * m;      // Block1D: Mish then *mask (decoder.py:41-43)
        v.z = mish_sel<ActT>(v.z) * m; v.w = mish_sel<ActT>(v.w) * m;
        if (a.temb) {                                                       // h += mlp(t); next Block1D multiplies by mask again
          v.x = (v.x + te[i].x) * m; v.y = (v.y + te[i].y) * m; v.z = (v.z + te[i].z) * m; v.w = (v.w + te[i].w) * m;
        }
        if (a.res) {
          const float4 r = *reinterpret_cast<const float4*>(a.res + row * a.res_ld + c);
          v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
        }
        if (a.out_f32) *reinterpret_cast<float4*>(a.out_f32 + row * a.f32_ld + c) = v;
        if (a.out_act) store_act4<ActT>(reinterpret_cast<ActT*>(a.out_act) + row * a.act_ld + c, v);
      }
      y[i] = v;
      sum += (v.x + v.y) + (v.z + v.w);
    }
    if (a.out_ln) {  // fused pre-LN of the transformer block that follows (transformer.py:262), eps 1e-5
      const float mean = warp_sum(sum) / (float)a.C;
      float sq = 0.0f;
#pragma unroll
      for (int i = 0; i < V4; ++i) {
        if (4 * (lane + 32 * i) < a.C) {
          const float d0 = y[i].x - mean, d1 = y[i].y - mean, d2 = y[i].z - mean, d3 = y[i].w - mean;
          sq += (d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3);
        }
      }
      const float rstd = 1.0f / sqrtf(warp_sum(sq) / (float)a.C + 1e-5f);
#pragma unroll
      for (int i = 0; i < V4; ++i) {
        const int c = 4 * (lane + 32 * i);
        if (c < a.C) {
          const float4 o = make_float4((y[i].x - mean) * rstd * lg[i].x + lb[i].x, (y[i].y - mean) * rstd * lg[i].y + lb[i].y,
                                       (y[i].z - mean) * rstd * lg[i].z + lb[i].z, (y[i].w - mean) * rstd * lg[i].w + lb[i].w);
          store_act4<ActT>(reinterpret_cast<ActT*>(a.out_ln) + row * a.ln_ld + c, o);
        }
      }
    }
  }
}

// Specialised bf16-operand variant for the decoder's width (C = 256, 8 groups of 32 channels): one compile-time MODE per
// call site instead of runtime feature tests, constants fetched before the programmatic-dependency wait, two rows of a warp
// in flight at a time, padded rows never read from x, four blocks per SM.  The generic kernel above spent ~58 issued
// instructions per element at 27 % occupancy (ncu, profiles/r01_ncu_full_gn_apply_v22.txt).
//   MODE 0: block1 of a ResNet block   y = (Mish(GN(x)) * m + temb) * m            -> bf16 operand
//   MODE 1: block2 + residual + pre-LN y = Mish(GN(x)) * m + res -> fp32 stream;  LN(y) -> bf16 operand
//   MODE 2: final block                y = Mish(GN(x)) * m                         -> bf16 operand
template <int MODE>
__global__ void __launch_bounds__(256, MODE == 1 ? 3 : 4) gn_apply256_kernel(GnApplyArgs a) {   // MODE 1 spills at 64 registers (measured: 1.13 -> 1.01 ms per step at 80)
  constexpr int C = 256;
  __shared__ float stat[16];
  pdl_trigger();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int c0 = 4 * lane, c1 = 128 + 4 * lane;          // this lane's two float4 channel groups (groups lane/8 and 4 + lane/8)
  // weights: not written by any kernel of the stream
  const float4 ga0 = __ldg(reinterpret_cast<const float4*>(a.gamma + c0)), ga1 = __ldg(reinterpret_cast<const float4*>(a.gamma + c1));
  const float4 be0 = __ldg(reinterpret_cast<const float4*>(a.beta + c0)), be1 = __ldg(reinterpret_cast<const float4*>(a.beta + c1));
  float4 lg0, lg1, lb0, lb1;
  if (MODE == 1) {
    lg0 = __ldg(reinterpret_cast<const float4*>(a.ln_gamma + c0)); lg1 = __ldg(reinterpret_cast<const float4*>(a.ln_gamma + c1));
    lb0 = __ldg(reinterpret_cast<const float4*>(a.ln_beta + c0)); lb1 = __ldg(reinterpret_cast<const float4*>(a.ln_beta + c1));
  }
  pdl_wait();
  if (threadIdx.x < 8) {
    double s = 0.0, q = 0.0;
    for (int ch = 0; ch < a.n_chunks; ++ch) {
      const double* p = a.partial + (((long long)b * a.n_chunks + ch) * 8 + threadIdx.x) * 2;
      s += p[0];
      q += p[1];
    }
    const double n = 32.0 * (double)a.T;
    const double mean = s / n;
    double var = q / n - mean * mean;
    if (var < 0.0) var = 0.0;
    stat[2 * threadIdx.x] = (float)mean;
    stat[2 * threadIdx.x + 1] = (float)(1.0 / sqrt(var + (double)a.eps));
  }
  const int len_b = a.mask.lens ? __ldg(a.mask.lens + b) : 0x7fffffff;
  const int t_base = (blockIdx.x * 8 + warp) * GN_APPLY_ROWS;
  float4 te0, te1;
  if (MODE == 0) { te0 = *reinterpret_cast<const float4*>(a.temb + b * a.temb_bs + c0); te1 = *reinterpret_cast<const float4*>(a.temb + b * a.temb_bs + c1); }
  __syncthreads();
  float4 sc0, sc1, sh0, sh1;
  {
    const float m0 = stat[2 * (lane >> 3)], r0 = stat[2 * (lane >> 3) + 1], m1 = stat[8 + 2 * (lane >> 3)], r1 = stat[9 + 2 * (lane >> 3)];
    sc0 = make_float4(r0 * ga0.x, r0 * ga0.y, r0 * ga0.z, r0 * ga0.w);
    sc1 = make_float4(r1 * ga1.x, r1 * ga1.y, r1 * ga1.z, r1 * ga1.w);
    sh0 = make_float4(be0.x - m0 * sc0.x, be0.y - m0 * sc0.y, be0.z - m0 * sc0.z, be0.w - m0 * sc0.w);
    sh1 = make_float4(be1.x - m1 * sc1.x, be1.y - m1 * sc1.y, be1.z - m1 * sc1.z, be1.w - m1 * sc1.w);
  }
  auto mish4 = [](float4 x, float4 sc, float4 sh) {
    return make_float4(mish_sel<bf16>(fmaf(x.x, sc.x, sh.x)), mish_sel<bf16>(fmaf(x.y, sc.y, sh.y)),
                       mish_sel<bf16>(fmaf(x.z, sc.z, sh.z)), mish_sel<bf16>(fmaf(x.w, sc.w, sh.w)));
  };
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
  for (int pair = 0; pair < GN_APPLY_ROWS; pair += 2) {
    float4 x0[2], x1[2], r0[2], r1[2];
    bool valid[2], live[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {                          // both rows' loads are issued before any arithmetic
      const int t = t_base + pair + k;
      live[k] = t < a.T;
      valid[k] = live[k] && (t << a.mask.shift) < len_b;
      const long long row = (long long)b * a.T + t;
      x0[k] = x1[k] = r0[k] = r1[k] = zero4;
      if (valid[k]) {                                      // a padded row is Mish(.) * 0: x is not read
        x0[k] = *reinterpret_cast<const float4*>(a.x + row * C + c0);
        x1[k] = *reinterpret_cast<const float4*>(a.x + row * C + c1);
      }
      if (MODE == 1 && live[k]) {
        r0[k] = *reinterpret_cast<const float4*>(a.res + row * a.res_ld + c0);
        r1[k] = *reinterpret_cast<const float4*>(a.res + row * a.res_ld + c1);
      }
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (!live[k]) continue;
      const long long row = (long long)b * a.T + t_base + pair + k;
      float4 v0 = zero4, v1 = zero4;
      if (valid[k]) {
        v0 = mish4(x0[k], sc0, sh0); v1 = mish4(x1[k], sc1, sh1);
        if (MODE == 0) {
          v0.x += te0.x; v0.y += te0.y; v0.z += te0.z; v0.w += te0.w;
          v1.x += te1.x; v1.y += te1.y; v1.z += te1.z; v1.w += te1.w;
        }
      }
      if (MODE != 1) {
        bf16* o = reinterpret_cast<bf16*>(a.out_act) + row * a.act_ld;
        store_act4<bf16>(o + c0, v0);
        store_act4<bf16>(o + c1, v1);
      } else {
        v0.x += r0[k].x; v0.y += r0[k].y; v0.z += r0[k].z; v0.w += r0[k].w;
        v1.x += r1[k].x; v1.y += r1[k].y; v1.z += r1[k].z; v1.w += r1[k].w;
        float* of = a.out_f32 + row * a.f32_ld;
        *reinterpret_cast<float4*>(of + c0) = v0;
        *reinterpret_cast<float4*>(of + c1) = v1;
        // fused pre-LN of the transformer block that follows (transformer.py:262), eps 1e-5
        const float mean = warp_sum((v0.x + v0.y) + (v0.z + v0.w) + (v1.x + v1.y) + (v1.z + v1.w)) * (1.0f / C);
        const float d0 = v0.x - mean, d1 = v0.y - mean, d2 = v0.z - mean, d3 = v0.w - mean;
        const float d4 = v1.x - mean, d5 = v1.y - mean, d6 = v1.z - mean, d7 = v1.w - mean;
        const float var = warp_sum((d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3) + (d4 * d4 + d5 * d5) + (d6 * d6 + d7 * d7)) * (1.0f / C);
        const float rstd = 1.0f / sqrtf(var + 1e-5f);
        bf16* o = reinterpret_cast<bf16*>(a.out_ln) + row * a.ln_ld;
        store_act4<bf16>(o + c0, make_float4(d0 * rstd * lg0.x + lb0.x, d1 * rstd * lg0.y + lb0.y, d2 * rstd * lg0.z + lb0.z, d3 * rstd * lg0.w + lb0.w));
        store_act4<bf16>(o + c1, make_float4(d4 * rstd * lg1.x + lb1.x, d5 * rstd * lg1.y + lb1.y, d6 * rstd * lg1.z + lb1.z, d7 * rstd * lg1.w + lb1.w));
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------- vocoder tail
// LeakyReLU(0.01) -> conv_post (C -> 1, k = 7, padding 3) -> tanh -> clamp (hifigan/models.py:191-195).
// thread = input row: it holds the row's C values in registers and forms the SEVEN tap products w[j] . x[row] (7 C FMAs on
// register operands; the weights come as broadcast 16-byte shared loads); out[t] = bias + sum_j partial_j[t + j] then costs seven
// shared loads.  A block owns kPostOut = 250 outputs = 256 rows with the +-3 halo.  The first version read every x value from
// shared memory once per tap (448 LDS per output) and was bound by the shared-memory pipe at 2.0 TB/s; this one is an HBM stream.
constexpr int kPostOut = 250;
template <int C>
__global__ void __launch_bounds__(256) conv_post_kernel(const float* __restrict__ x, int L, const float* __restrict__ w,
                                                        const float* __restrict__ bias, float* __restrict__ wav,
                                                        const int* __restrict__ lens, int hop) {
  constexpr int C4 = C / 4, PITCH = C + 4;                     // row pitch in floats: 16-byte aligned, conflict-free for 16-byte accesses
  __shared__ __align__(16) float xs[256 * PITCH];
  __shared__ __align__(16) float ws[7 * C];
  __shared__ float ps[7][256 + 8];
  const int b = blockIdx.y, t0 = blockIdx.x * kPostOut;
  // ragged batch: samples beyond the utterance's own length were never computed upstream -> the waveform is zero there
  const long long valid = lens ? min((long long)L, (long long)max(lens[b], 0) * hop) : (long long)L;
  if (t0 >= valid) {
    if ((int)threadIdx.x < kPostOut && t0 + (int)threadIdx.x < L) wav[(long long)b * L + t0 + threadIdx.x] = 0.0f;
    return;
  }
  for (int i = threadIdx.x; i < 7 * C; i += 256) ws[i] = w[i];
  const float* xb = x + (long long)b * L * C;
  // coalesced 16-byte loads of the 256 x C window (rows t0 - 3 .. t0 + 252), LeakyReLU applied on the way in
#pragma unroll
  for (int it = 0; it < C4; ++it) {
    const int i = threadIdx.x + it * 256, r = i / C4, c = (i - r * C4) * 4, t = t0 + r - 3;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t >= 0 && t < L) v = __ldcs(reinterpret_cast<const float4*>(xb + (long long)t * C + c));
    v.x = v.x > 0.0f ? v.x : v.x * 0.01f; v.y = v.y > 0.0f ? v.y : v.y * 0.01f;
    v.z = v.z > 0.0f ? v.z : v.z * 0.01f; v.w = v.w > 0.0f ? v.w : v.w * 0.01f;
    *reinterpret_cast<float4*>(xs + r * PITCH + c) = v;
  }
  __syncthreads();
  float xr[C];
#pragma unroll
  for (int c4 = 0; c4 < C4; ++c4) {
    const float4 v = *reinterpret_cast<const float4*>(xs + threadIdx.x * PITCH + 4 * c4);
    xr[4 * c4] = v.x; xr[4 * c4 + 1] = v.y; xr[4 * c4 + 2] = v.z; xr[4 * c4 + 3] = v.w;
  }
#pragma unroll
  for (int j = 0; j < 7; ++j) {
    float acc = 0.0f;
#pragma unroll
    for (int c4 = 0; c4 < C4; ++c4) {
      const float4 wv = *reinterpret_cast<const float4*>(ws + j * C + 4 * c4);
      acc = fmaf(wv.x, xr[4 * c4], acc); acc = fmaf(wv.y, xr[4 * c4 + 1], acc);
      acc = fmaf(wv.z, xr[4 * c4 + 2], acc); acc = fmaf(wv.w, xr[4 * c4 + 3], acc);
    }
    ps[j][threadIdx.x] = acc;                                  // tap j of output (row - j): row = tid, output = tid - j
  }
  __syncthreads();
  const int t = t0 + threadIdx.x;
  if ((int)threadIdx.x >= kPostOut || t >= L) return;
  float acc = bias[0];
#pragma unroll
  for (int j = 0; j < 7; ++j) acc += ps[j][threadIdx.x + j];    // output tid reads rows tid .. tid + 6 (= samples t - 3 .. t + 3)
  float y = tanhf(acc);
  y = fminf(fmaxf(y, -1.0f), 1.0f);
  wav[(long long)b * L + t] = t < valid ? y : 0.0f;
}

}  // namespace

// ================================================================================================ launchers
template <typename OutT>
cudaError_t cf_to_cl(const float* in, int B, int C, int T, OutT* out, long long out_ld, long long out_bs, float scale,
                     RowMask mask, cudaStream_t s) {
  dim3 grid(ceil_div(T, 32), ceil_div(C, 32), B), block(32, 8);
  cf_to_cl_kernel<OutT><<<grid, block, 0, s>>>(in, C, T, out, out_ld, out_bs, scale, mask);
  return cudaGetLastError();
}
template cudaError_t cf_to_cl<float>(const float*, int, int, int, float*, long long, long long, float, RowMask, cudaStream_t);
template cudaError_t cf_to_cl<bf16>(const float*, int, int, int, bf16*, long long, long long, float, RowMask, cudaStream_t);

cudaError_t cl_to_cf(const float* in, long long in_ld, long long in_bs, int B, int C, int T, float* out, float mul,
                     float add, cudaStream_t s) {
  dim3 grid(ceil_div(T, 32), ceil_div(C, 32), B), block(32, 8);
  cl_to_cf_kernel<<<grid, block, 0, s>>>(in, in_ld, in_bs, C, T, out, mul, add);
  return cudaGetLastError();
}

cudaError_t i64_to_i32(const long long* in, int* out, int n, cudaStream_t s) {
  i64_to_i32_kernel<<<ceil_div(n, 256), 256, 0, s>>>(in, out, n);
  return cudaGetLastError();
}

cudaError_t upload_floats(float* dst, const float* vals_host, int n, cudaStream_t s) {
  for (int off = 0; off < n; off += 32) {
    Vals32 v;
    const int m = n - off < 32 ? n - off : 32;
    for (int i = 0; i < 32; ++i) v.v[i] = i < m ? vals_host[off + i] : 0.0f;
    upload_kernel<<<1, 32, 0, s>>>(dst + off, v, m);
  }
  return cudaGetLastError();
}

cudaError_t upload_words(void* dst, const void* words_host, int n, cudaStream_t s) {
  const uint32_t* src = reinterpret_cast<const uint32_t*>(words_host);
  for (int off = 0; off < n; off += kUploadWords) {
    Words v;
    const int m = n - off < kUploadWords ? n - off : kUploadWords;
    for (int i = 0; i < kUploadWords; ++i) v.w[i] = i < m ? src[off + i] : 0u;
    upload_words_kernel<<<1, 256, 0, s>>>(reinterpret_cast<uint32_t*>(dst) + off, v, m);
  }
  return cudaGetLastError();
}

cudaError_t embed_tokens(const long long* ids, const float* emb, int B, int Tx, int C, int n_vocab, float scale,
                         RowMask mask, float* out, long long out_ld, long long* flags, cudaStream_t s) {
  embed_tokens_kernel<<<B * Tx, 64, 0, s>>>(ids, emb, Tx, C, n_vocab, scale, mask, out, out_ld, flags);
  return cudaGetLastError();
}
cudaError_t embed_speakers(const long long* ids, const float* table, int B, int dim, int n_spks, float* out, long long* flags, cudaStream_t s) {
  embed_speakers_kernel<<<B, 64, 0, s>>>(ids, table, dim, n_spks, out, flags);
  return cudaGetLastError();
}
cudaError_t fill_speaker_channels(const float* spk, int B, int T, int dim, RowMask mask, float* buf, long long ld, int c0,
                                  cudaStream_t s) {
  fill_speaker_kernel<<<B * T, 64, 0, s>>>(spk, T, dim, mask, buf, ld, c0);
  return cudaGetLastError();
}

template <typename ActT>
cudaError_t layer_norm_rows(const LnArgs& a, cudaStream_t s) {
  const int rows = a.B * a.T;
  const int blocks = ceil_div(rows, 8);
  const int vpl = ceil_div(a.C, 32);
  if (vpl <= 6) return launch_pdl(layer_norm_kernel<ActT, 6>, dim3(blocks), dim3(256), 0, s, a);
  if (vpl <= 8) return launch_pdl(layer_norm_kernel<ActT, 8>, dim3(blocks), dim3(256), 0, s, a);
  if (vpl <= 32) return launch_pdl(layer_norm_kernel<ActT, 32>, dim3(blocks), dim3(256), 0, s, a);
  return cudaErrorInvalidValue;
}
template cudaError_t layer_norm_rows<float>(const LnArgs&, cudaStream_t);
template cudaError_t layer_norm_rows<bf16>(const LnArgs&, cudaStream_t);

cudaError_t time_sinusoid(const float* t_steps, int n, int dim, float* out, cudaStream_t s) {
  time_sinusoid_kernel<<<n, 128, 0, s>>>(t_steps, n, dim, out);
  return cudaGetLastError();
}

template <typename ActT>
cudaError_t decoder_pack_input(const float* z_cf, const float* mu_cf, const float* spk, int B, int F, int S, int T,
                               float temperature, const float* temperatures, RowMask mask, float* x_state, ActT* xin,
                               long long xin_ld, cudaStream_t s) {
  dim3 grid(ceil_div(T, 32), B);
  const size_t sh = (size_t)2 * F * 33 * sizeof(float);
  decoder_pack_kernel<ActT><<<grid, 256, sh, s>>>(z_cf, mu_cf, spk, F, S, T, temperature, temperatures, mask, x_state, xin, xin_ld);
  return cudaGetLastError();
}
template cudaError_t decoder_pack_input<float>(const float*, const float*, const float*, int, int, int, int, float, const float*, RowMask, float*,
                                               float*, long long, cudaStream_t);
template cudaError_t decoder_pack_input<bf16>(const float*, const float*, const float*, int, int, int, int, float, const float*, RowMask, float*,
                                              bf16*, long long, cudaStream_t);

cudaError_t group_norm_stats(const float* x, int B, int T, int C, int groups, double* partial, int* n_chunks_out,
                             cudaStream_t s) {
  const int cpg = C / groups;
  if (C > 1024 || C % groups || cpg > 32 || (cpg & (cpg - 1)) || (C % 32)) return cudaErrorInvalidValue;
  const int chunks = ceil_div(T, GN_ROWS);
  *n_chunks_out = chunks;
  gn_stats_kernel<<<dim3(chunks, B), C, 0, s>>>(x, T, C, cpg, partial);
  return cudaGetLastError();
}

template <typename ActT>
cudaError_t group_norm_apply(const GnApplyArgs& a, cudaStream_t s) {
  const int cpg = a.C / a.groups;
  if ((a.C & 3) || (cpg & 3) || (a.res_ld & 3) || (a.f32_ld & 3) || (a.act_ld & 3) || (a.ln_ld & 3)) return cudaErrorInvalidValue;
  const int v4 = ceil_div(a.C, 128);
  dim3 grid(ceil_div(a.T, 8 * GN_APPLY_ROWS), a.B);
  if constexpr (std::is_same<ActT, bf16>::value) {
    static const bool fast = []() { const char* v = getenv("EV_GN_FAST"); return !(v && atoi(v) == 0); }();   // EV_GN_FAST=0: generic kernel
    auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    if (fast && a.C == 256 && a.groups == 8 && al16(a.x) && al16(a.gamma) && al16(a.beta)) {
      const bool m0 = a.temb && !a.res && !a.out_f32 && !a.out_ln && a.out_act && al16(a.temb) && al16(a.out_act);
      const bool m1 = !a.temb && a.res && a.out_f32 && a.out_ln && !a.out_act && al16(a.res) && al16(a.out_f32) && al16(a.out_ln) &&
                      al16(a.ln_gamma) && al16(a.ln_beta);
      const bool m2 = !a.temb && !a.res && !a.out_f32 && !a.out_ln && a.out_act && al16(a.out_act);
      if (m0) return launch_pdl(gn_apply256_kernel<0>, grid, dim3(256), 0, s, a);
      if (m1) return launch_pdl(gn_apply256_kernel<1>, grid, dim3(256), 0, s, a);
      if (m2) return launch_pdl(gn_apply256_kernel<2>, grid, dim3(256), 0, s, a);
    }
  }
  const size_t sh = (size_t)a.groups * 2 * sizeof(float);
  if (v4 <= 2) return launch_pdl(gn_apply_kernel<ActT, 2>, grid, dim3(256), sh, s, a);
  if (v4 <= 8) return launch_pdl(gn_apply_kernel<ActT, 8>, grid, dim3(256), sh, s, a);
  return cudaErrorInvalidValue;
}
template cudaError_t group_norm_apply<float>(const GnApplyArgs&, cudaStream_t);
template cudaError_t group_norm_apply<bf16>(const GnApplyArgs&, cudaStream_t);

cudaError_t conv_post_tanh(const float* x, int B, int L, int C, const float* w, const float* bias, float* wav, const int* lens,
                           int hop, cudaStream_t s) {
  dim3 grid(ceil_div(L, kPostOut), B);
  if (C == 32) conv_post_kernel<32><<<grid, 256, 0, s>>>(x, L, w, bias, wav, lens, hop);
  else if (C == 16) conv_post_kernel<16><<<grid, 256, 0, s>>>(x, L, w, bias, wav, lens, hop);
  else return cudaErrorInvalidValue;
  return cudaGetLastError();
}

}  // namespace ev
