// fp32 CUDA-core flash attention over channel-last q/k/v (online softmax, keys tiled through shared memory).
// Two reference semantics:
//   mode 0  text encoder MultiHeadAttention (text_encoder.py:223-246): RoPE on the first rope_dim features of q and k
//           (rotate-half pairing, :147-169), scores/sqrt(d), masked_fill(mask==0, -1e4) where query OR key is padded.
//   mode 1  diffusers Attention as the decoder calls it (transformer.py:266-271): the 0/1 frame mask is a FLOAT
//           attn_mask, i.e. +1 is ADDED to the logits of valid keys and padded keys stay in the softmax (SURVEY H1).
#include "kernels.cuh"

namespace ev {
namespace {

constexpr int QPW = 4, NW = 8, BQ = QPW * NW, BKT = 32;

// text_encoder.py:147-169 (rotate-half pairing): out[d] = x[d]*cos + partner*sin, partner = -x[d + half] for d < half, x[d - half] above
__device__ __forceinline__ float rope_mix(float x, float partner, float c, float s) { return x * c + partner * s; }

// Stage `rows` rows (starting at t0) of D features into shared memory (row pitch `pitch` floats), RoPE applied to the first
// rope_dim features.  Work items are float4 groups: for d < rope_dim/2 one item loads the group at d AND its partner group at
// d + rope_dim/2 and writes both rotated outputs; features >= rope_dim are plain copies.  All loads of a thread are issued
// before the first use (the loops are fully unrolled).
template <int D>
__device__ __forceinline__ void load_tile_rope(const float* base, int t0, int rows, int pitch, float* dst, const AttnArgs& a) {
  const int half = a.rope_dim >> 1;
  const int pair_items = half >> 2, plain_items = (D - a.rope_dim) >> 2, per_row = pair_items + plain_items;
  const int total = rows * per_row;
  constexpr int MAX_IT = (BQ * (D / 4) + NW * 32 - 1) / (NW * 32);
  float4 x[MAX_IT], y[MAX_IT];
#pragma unroll
  for (int it = 0; it < MAX_IT; ++it) {
    const int idx = threadIdx.x + it * NW * 32;
    x[it] = y[it] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (idx < total) {
      const int r = idx / per_row, i = idx - r * per_row, t = t0 + r;
      if (t < a.T) {
        const float* row = base + (long long)t * a.ld;
        if (i < pair_items) { x[it] = *reinterpret_cast<const float4*>(row + 4 * i); y[it] = *reinterpret_cast<const float4*>(row + half + 4 * i); }
        else x[it] = *reinterpret_cast<const float4*>(row + a.rope_dim + 4 * (i - pair_items));
      }
    }
  }
#pragma unroll
  for (int it = 0; it < MAX_IT; ++it) {
    const int idx = threadIdx.x + it * NW * 32;
    if (idx >= total) continue;
    const int r = idx / per_row, i = idx - r * per_row, t = t0 + r;
    float* o = dst + r * pitch;
    if (i < pair_items) {
      float4 c4 = make_float4(1.f, 1.f, 1.f, 1.f), s4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (t < a.T) { c4 = *reinterpret_cast<const float4*>(a.rope_cos + t * half + 4 * i); s4 = *reinterpret_cast<const float4*>(a.rope_sin + t * half + 4 * i); }
      const int d = 4 * i;
      o[d] = rope_mix(x[it].x, -y[it].x, c4.x, s4.x); o[d + 1] = rope_mix(x[it].y, -y[it].y, c4.y, s4.y);
      o[d + 2] = rope_mix(x[it].z, -y[it].z, c4.z, s4.z); o[d + 3] = rope_mix(x[it].w, -y[it].w, c4.w, s4.w);
      o[d + half] = rope_mix(y[it].x, x[it].x, c4.x, s4.x); o[d + half + 1] = rope_mix(y[it].y, x[it].y, c4.y, s4.y);
      o[d + half + 2] = rope_mix(y[it].z, x[it].z, c4.z, s4.z); o[d + half + 3] = rope_mix(y[it].w, x[it].w, c4.w, s4.w);
    } else {
      const int d = a.rope_dim + 4 * (i - pair_items);
      o[d] = x[it].x; o[d + 1] = x[it].y; o[d + 2] = x[it].z; o[d + 3] = x[it].w;
    }
  }
}

template <typename ActT, int D>
__global__ void __launch_bounds__(NW * 32) attn_kernel(AttnArgs a) {
  extern __shared__ float sh[];
  float* Qs = sh;                      // [BQ][D]
  float* Ks = Qs + BQ * D;             // [BKT][D+1]
  float* Vs = Ks + BKT * (D + 1);      // [BKT][D]
  float* Ps = Vs + BKT * D;            // [NW][QPW][BKT]
  constexpr int DPL = D / 32;
  const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * BQ;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int len = a.lens ? a.lens[b] : (a.T << a.len_shift);
  const float* qb = a.q + b * a.bs + h * D;
  const float* kb = a.k + b * a.bs + h * D;
  const float* vb = a.v + b * a.bs + h * D;

  // q, k, v tiles are staged float4 by float4 with every load of a thread in flight at once (the element-wise version
  // spent most of the kernel in serial, latency-bound global loads); RoPE pairs (d, d + rope_dim/2) are rotated together
  load_tile_rope<D>(qb, q0, BQ, D, Qs, a);
  float m_run[QPW], l_run[QPW], o[QPW][DPL];
  bool qvalid[QPW];
#pragma unroll
  for (int qq = 0; qq < QPW; ++qq) {
    m_run[qq] = -INFINITY;
    l_run[qq] = 0.0f;
    const int t = q0 + warp * QPW + qq;
    qvalid[qq] = (t << a.len_shift) < len;
#pragma unroll
    for (int i = 0; i < DPL; ++i) o[qq][i] = 0.0f;
  }

  for (int k0 = 0; k0 < a.T; k0 += BKT) {
    __syncthreads();
    load_tile_rope<D>(kb, k0, BKT, D + 1, Ks, a);
#pragma unroll
    for (int it = 0; it < (BKT * D / 4) / (NW * 32); ++it) {
      const int idx = threadIdx.x + it * NW * 32, kj = idx / (D / 4), d = (idx - kj * (D / 4)) * 4, t = k0 + kj;
      float4 vv = make_float4(0.f, 0.f, 0.f, 0.f);
      if (t < a.T) vv = *reinterpret_cast<const float4*>(vb + (long long)t * a.ld + d);
      *reinterpret_cast<float4*>(Vs + kj * D + d) = vv;
    }
    __syncthreads();
    const int tk = k0 + lane;
    const bool k_in = tk < a.T;
    const bool kvalid = (tk << a.len_shift) < len;
    float s[QPW];
#pragma unroll
    for (int qq = 0; qq < QPW; ++qq) s[qq] = 0.0f;
    const float* krow = Ks + lane * (D + 1);
#pragma unroll 4
    for (int d = 0; d < D; d += 4) {
      const float k0v = krow[d], k1v = krow[d + 1], k2v = krow[d + 2], k3v = krow[d + 3];
#pragma unroll
      for (int qq = 0; qq < QPW; ++qq) {
        const float4 q4 = *reinterpret_cast<const float4*>(Qs + (warp * QPW + qq) * D + d);
        s[qq] = fmaf(q4.x, k0v, s[qq]);
        s[qq] = fmaf(q4.y, k1v, s[qq]);
        s[qq] = fmaf(q4.z, k2v, s[qq]);
        s[qq] = fmaf(q4.w, k3v, s[qq]);
      }
    }
#pragma unroll
    for (int qq = 0; qq < QPW; ++qq) {
      float sc = s[qq] * a.scale;
      if (a.mode == 0) sc = (qvalid[qq] && kvalid) ? sc : -1e4f;
      else sc += kvalid ? 1.0f : 0.0f;
      if (!k_in) sc = -INFINITY;
      const float m_new = fmaxf(m_run[qq], warp_max(sc));
      const float p = k_in ? expf(sc - m_new) : 0.0f;
      const float corr = expf(m_run[qq] - m_new);
      l_run[qq] = l_run[qq] * corr + warp_sum(p);
      m_run[qq] = m_new;
      Ps[(warp * QPW + qq) * BKT + lane] = p;
#pragma unroll
      for (int i = 0; i < DPL; ++i) o[qq][i] *= corr;
    }
    __syncwarp();
#pragma unroll 4
    for (int j = 0; j < BKT; ++j) {
      float vv[DPL];
#pragma unroll
      for (int i = 0; i < DPL; ++i) vv[i] = Vs[j * D + lane + 32 * i];
#pragma unroll
      for (int qq = 0; qq < QPW; ++qq) {
        const float pj = Ps[(warp * QPW + qq) * BKT + j];
#pragma unroll
        for (int i = 0; i < DPL; ++i) o[qq][i] = fmaf(pj, vv[i], o[qq][i]);
      }
    }
  }
  ActT* ob = reinterpret_cast<ActT*>(a.out) + b * a.out_bs + h * D;
#pragma unroll
  for (int qq = 0; qq < QPW; ++qq) {
    const int t = q0 + warp * QPW + qq;
    if (t >= a.T) continue;
    const float inv = 1.0f / l_run[qq];
#pragma unroll
    for (int i = 0; i < DPL; ++i) ob[(long long)t * a.out_ld + lane + 32 * i] = from_float<ActT>(o[qq][i] * inv);
  }
}

__global__ void rope_tables_kernel(float* cos_t, float* sin_t, int T, int rope_dim, float base) {
  const int half = rope_dim / 2;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= T * half) return;
  const int t = idx / half, i = idx - t * half;
  // text_encoder.py:131-141: theta_i = 1/(base^(2i/d)), angle = t*theta_i, all float32
  const float e = __fdiv_rn((float)(2 * i), (float)rope_dim);
  const float pw = (float)pow((double)base, (double)e);
  const float theta = __fdiv_rn(1.0f, pw);
  const float ang = __fmul_rn((float)t, theta);
  cos_t[idx] = (float)cos((double)ang);
  sin_t[idx] = (float)sin((double)ang);
}

template <typename ActT, int D>
cudaError_t launch_attn(const AttnArgs& a, cudaStream_t s) {
  const size_t sh = (size_t)(BQ * D + BKT * (D + 1) + BKT * D + NW * QPW * BKT) * sizeof(float);
  static DeviceOnce once;
  cudaError_t ce = once.run([&]() { return cudaFuncSetAttribute(attn_kernel<ActT, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sh); });
  if (ce != cudaSuccess) return ce;
  if ((a.rope_dim & 7) || ((D - a.rope_dim) & 3) || (a.ld & 3) || (a.bs & 3)) return cudaErrorInvalidValue;   // float4 staging
  dim3 grid(ceil_div(a.T, BQ), a.H, a.B);
  attn_kernel<ActT, D><<<grid, NW * 32, sh, s>>>(a);
  return cudaGetLastError();
}

}  // namespace

template <typename ActT>
cudaError_t attention_rows(const AttnArgs& a, cudaStream_t s) {
  if (a.D == 64) return launch_attn<ActT, 64>(a, s);
  if (a.D == 96) return launch_attn<ActT, 96>(a, s);
  if (a.D == 128) return launch_attn<ActT, 128>(a, s);
  return cudaErrorInvalidValue;
}
template cudaError_t attention_rows<float>(const AttnArgs&, cudaStream_t);
template cudaError_t attention_rows<bf16>(const AttnArgs&, cudaStream_t);

cudaError_t rope_tables(float* cos_t, float* sin_t, int T, int rope_dim, float base, cudaStream_t s) {
  const int n = T * (rope_dim / 2);
  rope_tables_kernel<<<ceil_div(n, 256), 256, 0, s>>>(cos_t, sin_t, T, rope_dim, base);
  return cudaGetLastError();
}

}  // namespace ev
