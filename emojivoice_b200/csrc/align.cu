// Duration -> length -> monotonic alignment path -> frame gather.  Integer-valued results, bit-exact against the
// CPU reference (matcha_tts.py:122-135, utils/model.py:7-41); see SURVEY.md H2 for the float traps reproduced here.
#include "aten_sum.h"
#include "kernels.cuh"

namespace ev {
namespace {

// one thread per utterance: the row is short (Tx tokens) and the summation ORDER is the contract.  length_scales (device, B)
// or nullptr = length_scale for every row: a row's arithmetic is the same either way.
__global__ void durations_kernel(const float* __restrict__ logw, const int* __restrict__ x_lens, int B, int Tx,
                                 float length_scale, const float* __restrict__ length_scales, float* __restrict__ w_ceil,
                                 long long* __restrict__ y_lengths, long long* __restrict__ y_max) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  if (length_scales) length_scale = length_scales[b];
  const float* lw = logw + (long long)b * Tx;
  float* wc = w_ceil + (long long)b * Tx;
  const int len = x_lens[b];
  for (int i = 0; i < Tx; ++i) {
    const float m = i < len ? 1.0f : 0.0f;
    const float w = __fmul_rn(expf(lw[i]), m);                 // w = exp(logw) * x_mask
    wc[i] = __fmul_rn(ceilf(w), length_scale);                 // w_ceil = ceil(w) * length_scale
  }
  const float s = evsum::sum_f32(wc, Tx);                      // torch.sum(w_ceil, [1, 2]) in ATen's CPU order
  const long long y = (long long)fmaxf(s, 1.0f);               // clamp_min(.., 1).long() truncates
  y_lengths[b] = y;
  if (y_max) atomicMax(y_max, y);                              // y_lengths.max(): the host's one read-back (utils/model.py:18)
}

__global__ void row_sum_kernel(const float* x, int B, int Tx, float* out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B) out[b] = evsum::sum_f32(x + (long long)b * Tx, Tx);
}

constexpr int PATH_ROWS = 8;  // token rows per block
// grid (ceil(Tx/PATH_ROWS), B).  torch.cumsum(float32) on CPU == running sum in float64 rounded to float32 at each
// prefix (SURVEY.md H2c); path[i][j] = (j < cum_i) - (j < cum_{i-1}) with j compared as float32, times the mask.
__global__ void generate_path_kernel(const float* __restrict__ w_ceil, const int* __restrict__ x_lens,
                                     const int* __restrict__ y_lens, int Tx, int T_pad, float* __restrict__ attn,
                                     int* __restrict__ frame_token) {
  __shared__ float cum[PATH_ROWS + 1];
  const int b = blockIdx.y, i0 = blockIdx.x * PATH_ROWS;
  if (threadIdx.x == 0) {
    const float* wc = w_ceil + (long long)b * Tx;
    double run = 0.0;
    for (int i = 0; i < i0; ++i) run += (double)wc[i];
    cum[0] = i0 == 0 ? 0.0f : (float)run;   // F.pad prepends a zero row, i.e. (j < cum_{-1}) == false
    for (int r = 0; r < PATH_ROWS; ++r) {
      const int i = i0 + r;
      if (i < Tx) run += (double)wc[i];
      cum[r + 1] = (float)run;
    }
  }
  __syncthreads();
  const int xl = x_lens[b], yl = y_lens[b];
  for (int idx = threadIdx.x; idx < PATH_ROWS * T_pad; idx += blockDim.x) {
    const int r = idx / T_pad, j = idx - r * T_pad, i = i0 + r;
    if (i >= Tx) break;
    const float fj = (float)j;
    const float lo = (i == 0) ? 0.0f : ((fj < cum[r]) ? 1.0f : 0.0f);
    const float hi = (fj < cum[r + 1]) ? 1.0f : 0.0f;
    const float m = (i < xl && j < yl) ? 1.0f : 0.0f;
    const float v = (hi - lo) * m;
    attn[((long long)b * Tx + i) * T_pad + j] = v;
    if (v == 1.0f) frame_token[(long long)b * T_pad + j] = i;
  }
}

// mu_y = attn^T mu_x is a gather (every frame column of attn holds at most one 1)
__global__ void gather_mu_kernel(const float* __restrict__ mu_x, const int* __restrict__ frame_token,
                                 const int* __restrict__ y_lens, int C, int Tx, int T_pad, float* __restrict__ mu_y,
                                 float* __restrict__ y_mask) {
  const int b = blockIdx.z, c = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= T_pad) return;
  const int tok = frame_token[(long long)b * T_pad + j];
  mu_y[((long long)b * C + c) * T_pad + j] = tok >= 0 ? mu_x[((long long)b * C + c) * Tx + tok] : 0.0f;
  if (c == 0) y_mask[(long long)b * T_pad + j] = j < y_lens[b] ? 1.0f : 0.0f;
}

}  // namespace

cudaError_t durations(const float* logw, const int* x_lens, int B, int Tx, float length_scale, const float* length_scales,
                      float* w_ceil, long long* y_lengths, long long* y_max, cudaStream_t s) {
  durations_kernel<<<ceil_div(B, 32), 32, 0, s>>>(logw, x_lens, B, Tx, length_scale, length_scales, w_ceil, y_lengths, y_max);
  return cudaGetLastError();
}
cudaError_t row_sum_aten(const float* x, int B, int Tx, float* out, cudaStream_t s) {
  row_sum_kernel<<<ceil_div(B, 32), 32, 0, s>>>(x, B, Tx, out);
  return cudaGetLastError();
}
cudaError_t generate_path(const float* w_ceil, const int* x_lens, const int* y_lens, int B, int Tx, int T_pad,
                          float* attn, int* frame_token, cudaStream_t s) {
  cudaError_t ce = cudaMemsetAsync(frame_token, 0xFF, (size_t)B * T_pad * sizeof(int), s);
  if (ce != cudaSuccess) return ce;
  generate_path_kernel<<<dim3(ceil_div(Tx, PATH_ROWS), B), 256, 0, s>>>(w_ceil, x_lens, y_lens, Tx, T_pad, attn, frame_token);
  return cudaGetLastError();
}
cudaError_t gather_mu(const float* mu_x_cf, const int* frame_token, const int* y_lens, int B, int C, int Tx, int T_pad,
                      float* mu_y_cf, float* y_mask, cudaStream_t s) {
  gather_mu_kernel<<<dim3(ceil_div(T_pad, 128), C, B), 128, 0, s>>>(mu_x_cf, frame_token, y_lens, C, Tx, T_pad, mu_y_cf, y_mask);
  return cudaGetLastError();
}

}  // namespace ev
