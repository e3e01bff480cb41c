// fp32 CUDA-core implicit-GEMM conv1d (channel-last), fixed summation order: taps outer, channels inner.
// Used for the text encoder / duration predictor (fp32 protects ceil(exp(logw)), SURVEY.md H2a) and as the
// EV_PREC_FP32 parity mode of the decoder and vocoder.
#include "conv.cuh"

namespace ev {

namespace {
constexpr int BM = 64, BK = 16, THREADS = 256;

// 64 x (16*TN) output tile, 4 x TN accumulators per thread, shared-memory double buffering with the next K-chunk's
// global loads in flight during the FMAs.  TN = 8 halves the shared-memory bytes read per FMA (the binding resource of
// a 4x4 register tile); TN = 4 serves narrow layers.  The per-output summation order is unchanged: taps outer,
// channels ascending, one fmaf chain.
template <int TN, bool ITEM>
__global__ void __launch_bounds__(THREADS)
conv_simt_kernel(ConvGeom g, const float* __restrict__ x, long long x_ld, long long x_bs,
                 const float* __restrict__ w, int N_pad, Epilogue e) {
  constexpr int BN = 16 * TN, NB4 = TN / 4;
  __shared__ __align__(16) float As[2][BK][BM + 4];
  __shared__ __align__(16) float Bs[2][BK][BN];
  const int b = blockIdx.z, m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int a_row = tid >> 2, a_c = (tid & 3) << 2;
  const int b_k = tid >> 4, b_n = (tid & 15) << 2;
  float acc[4][TN];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.0f;

  const float* xb = x + (long long)b * x_bs;
  const int kchunks = (g.C_in + BK - 1) / BK, n_it = g.taps * kchunks;
  float4 av, bv[NB4];
  auto fetch = [&](int it) {
    const int tap = it / kchunks, c0 = (it - tap * kchunks) * BK;
    const int t_in = (m0 + a_row) * g.conv_stride + g.tap_off[tap];
    const bool row_ok = (m0 + a_row < g.M) && t_in >= 0 && t_in < g.T_in;
    av = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row_ok && c0 + a_c < g.C_in) av = *reinterpret_cast<const float4*>(xb + (long long)t_in * x_ld + c0 + a_c);
    const float* wt = w + ((size_t)tap * g.C_in + c0 + b_k) * N_pad + n0 + b_n;
#pragma unroll
    for (int h = 0; h < NB4; ++h) {
      bv[h] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c0 + b_k < g.C_in && n0 + b_n + 64 * h < N_pad) bv[h] = __ldg(reinterpret_cast<const float4*>(wt + 64 * h));
    }
  };
  auto stash = [&](int buf) {
    As[buf][a_c + 0][a_row] = av.x; As[buf][a_c + 1][a_row] = av.y; As[buf][a_c + 2][a_row] = av.z; As[buf][a_c + 3][a_row] = av.w;
#pragma unroll
    for (int h = 0; h < NB4; ++h) *reinterpret_cast<float4*>(&Bs[buf][b_k][b_n + 64 * h]) = bv[h];
  };
  fetch(0);
  stash(0);
  __syncthreads();
  for (int it = 0; it < n_it; ++it) {
    const int cur = it & 1;
    if (it + 1 < n_it) fetch(it + 1);          // global loads fly during the FMAs below
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[cur][k][ty * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
      for (int h = 0; h < NB4; ++h) {
        const float4 b4 = *reinterpret_cast<const float4*>(&Bs[cur][k][tx * 4 + 64 * h]);
        const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][4 * h + j] = fmaf(a[i], bb[j], acc[i][4 * h + j]);
      }
    }
    if (it + 1 < n_it) stash(cur ^ 1);         // the other buffer was last read one iteration ago (barrier below)
    __syncthreads();
  }

  float* out_act = reinterpret_cast<float*>(e.out_act);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = m0 + ty * 4 + i;
    if (r >= g.M) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int n = n0 + tx * 4 + (j & 3) + 64 * (j >> 2);
      if (n >= g.N) continue;
      int t, co;
      if (!ep_coord(e, r, n, t, co)) continue;
      const float mv = e.mask.at(b, t);
      const float v = ep_value<ITEM>(e, b, t, co, acc[i][j], mv);
      if (e.out_f32) e.out_f32[b * e.f32_bs + (long long)t * e.f32_ld + co] = v;
      if (out_act) out_act[b * e.act_bs + (long long)t * e.act_ld + co] = ep_act(e, co, v, mv);
    }
  }
}
}  // namespace

cudaError_t conv_simt_launch(const ConvGeom& g, const float* x, long long x_ld, long long x_bs, const ConvWeights& w,
                             const Epilogue& e, cudaStream_t stream) {
  if ((g.C_in & 3) || (x_ld & 3) || (w.N_pad & 3)) return cudaErrorInvalidValue;
  const bool item = e.item_dt != nullptr;
  if (item && (!e.item_n || !e.res || e.res2 || e.div != 1.0f)) return cudaErrorInvalidValue;
  // the wide tile only pays when it still fills the machine a few times over (the text encoder's GEMMs are small)
  if (g.N > 64 && (long long)ceil_div(g.M, BM) * ceil_div(g.N, 128) * g.B >= 6 * 148) {
    dim3 grid(ceil_div(g.M, BM), ceil_div(g.N, 128), g.B);
    if (item) conv_simt_kernel<8, true><<<grid, THREADS, 0, stream>>>(g, x, x_ld, x_bs, w.w_f32, w.N_pad, e);
    else conv_simt_kernel<8, false><<<grid, THREADS, 0, stream>>>(g, x, x_ld, x_bs, w.w_f32, w.N_pad, e);
  } else {
    dim3 grid(ceil_div(g.M, BM), ceil_div(g.N, 64), g.B);
    if (item) conv_simt_kernel<4, true><<<grid, THREADS, 0, stream>>>(g, x, x_ld, x_bs, w.w_f32, w.N_pad, e);
    else conv_simt_kernel<4, false><<<grid, THREADS, 0, stream>>>(g, x, x_ld, x_bs, w.w_f32, w.N_pad, e);
  }
  return cudaGetLastError();
}

}  // namespace ev
