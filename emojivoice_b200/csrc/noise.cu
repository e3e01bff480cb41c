// Seeded prior noise of the flow-matching decoder (ev_prior_noise): z[b, f, t] is a function of (seeds[b], f, t) only.
// Philox4x32-10 (Random123's round function and constants) keyed by the utterance's 64-bit seed and countered by
// (t >> 2, f, 0, 0) gives four 32-bit words per group of four frames; two Box-Muller pairs in float64 turn them into four
// N(0, 1) samples, each rounded once to fp32.  oracle/prior_noise.py is the same definition in numpy.
#include "ctx.cuh"

namespace ev {
namespace {

constexpr uint32_t kPhiloxM0 = 0xD2511F53u, kPhiloxM1 = 0xCD9E8D57u;
constexpr uint32_t kPhiloxW0 = 0x9E3779B9u, kPhiloxW1 = 0xBB67AE85u;

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t lo0 = kPhiloxM0 * c.x, hi0 = __umulhi(kPhiloxM0, c.x);
    const uint32_t lo1 = kPhiloxM1 * c.z, hi1 = __umulhi(kPhiloxM1, c.z);
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += kPhiloxW0;
    k1 += kPhiloxW1;
  }
  return c;
}

// u = (a + 0.5) 2^-32 in (0, 1), v = b 2^-32 in [0, 1): both exact in double.  u >= 2^-33 bounds |z| by sqrt(66 ln 2) = 6.77.
__device__ __forceinline__ float2 box_muller(uint32_t a, uint32_t b) {
  const double u = ((double)a + 0.5) * 0x1p-32, v = (double)b * 0x1p-32;
  const double r = sqrt(-2.0 * log(u));
  double s, c;
  sincospi(2.0 * v, &s, &c);
  return make_float2((float)(r * c), (float)(r * s));
}

// One thread per (b, f, q): frames 4q .. 4q + 3 of row (b, f), a float4 store when the whole group lies in a 16-byte aligned
// row segment, scalar stores otherwise (a partial last group, or T % 4 != 0).
__global__ void __launch_bounds__(256) prior_noise_kernel(const unsigned long long* __restrict__ seeds, int F, int T, long long Q,
                                                          long long total, float* __restrict__ z) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const long long row = idx / Q;                   // b * F + f
  const long long q = idx - row * Q;
  const int b = (int)(row / F), f = (int)(row - (long long)b * F);
  const unsigned long long seed = seeds[b];
  const uint4 w = philox4x32_10(make_uint4((uint32_t)q, (uint32_t)f, 0u, 0u), (uint32_t)seed, (uint32_t)(seed >> 32));
  const float2 z01 = box_muller(w.x, w.y), z23 = box_muller(w.z, w.w);
  const long long t0 = 4 * q;
  float* p = z + row * T + t0;
  if (t0 + 4 <= T && (reinterpret_cast<uintptr_t>(p) & 15) == 0) {
    *reinterpret_cast<float4*>(p) = make_float4(z01.x, z01.y, z23.x, z23.y);
  } else {
    const float v[4] = {z01.x, z01.y, z23.x, z23.y};
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (t0 + i < T) p[i] = v[i];
  }
}

}  // namespace
}  // namespace ev

using namespace ev;

extern "C" int ev_prior_noise(ev_ctx* ctx, const int64_t* seeds, int B, int n_feats, int T, float* z, void* stream) {
  if (!ctx) return EV_ERR_INVALID;
  if (!seeds || !z || B <= 0 || n_feats <= 0 || T <= 0) return fail(ctx, EV_ERR_INVALID, "ev_prior_noise: null argument or empty shape");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  const long long Q = ((long long)T + 3) / 4, total = (long long)B * n_feats * Q;
  const long long blocks = (total + 255) / 256;
  if (blocks > 0x7fffffffLL) return fail(ctx, EV_ERR_INVALID, "ev_prior_noise: shape too large");
  EV_LAUNCH(ctx, s, "prior_noise", 0, 4.0 * B * (double)n_feats * T + 8.0 * B,
            (prior_noise_kernel<<<(unsigned)blocks, 256, 0, s>>>(reinterpret_cast<const unsigned long long*>(seeds), n_feats, T, Q,
                                                                 total, z),
             cudaGetLastError()));
  return EV_OK;
}
