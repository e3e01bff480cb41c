// Bias denoiser (hifigan/denoiser.py:7-64): centred hann STFT(n_fft 1024, hop 256) -> magnitude minus
// strength*bias_spec, clamped at 0 -> inverse STFT with the original phase.
//
// Round 1 ran both transforms as dense fp32 GEMMs against windowed Fourier bases (2 x 45 GFLOP per config-2 batch on the
// CUDA cores: 2.96 ms, 8 % of a step).  Now ONE kernel per PAIR of frames does the whole spectral path in shared memory:
//     z[n] = hann[n] * (x_f[n] + i x_{f+1}[n])  ->  1024-point complex FFT (radix-4 Stockham, 5 passes)
//     X_f[k] = (Z[k] + conj Z[N-k]) / 2,  X_{f+1}[k] = (Z[k] - conj Z[N-k]) / 2i          (two real spectra from one FFT)
//     X'[k] = X[k] * max(|X[k]| - strength * bias[k], 0) / |X[k]|                          (denoiser.py:61-62, phase kept)
//     Z'[k] = X'_f[k] + i X'_{f+1}[k] (Hermitian extension)  ->  inverse FFT  ->  y_f = Re z' hann, y_{f+1} = Im z' hann
// followed by the overlap-add / window-envelope normalisation of torch.istft.  2.2 GFLOP instead of 90, fp32 throughout
// (twiddles from a table computed in double precision); the reflect padding of torch.stft(center=True) is folded into the loads.
// The GEMM path stays available as EV_DN_FFT=0 (cross-check).
#include "ctx.cuh"

using namespace ev;

namespace {
cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

constexpr int NFFT = 1024, HOP = 256, NBIN = NFFT / 2 + 1, NSPEC = 2 * NBIN, SPEC_LD = 1028;


__device__ __forceinline__ double hann(int j) { return 0.5 - 0.5 * cospi(2.0 * j / (double)NFFT); }  // periodic hann

// forward basis  W[tap][ci][n]:  j = tap*256+ci ; n<513: win[j]*cos(2 pi n j/N) ; n>=513: -win[j]*sin(2 pi (n-513) j/N)
__global__ void fwd_basis_kernel(float* w, int N_pad) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= NFFT * NSPEC) return;
  const int j = idx / NSPEC, n = idx - j * NSPEC;
  const int k = n < NBIN ? n : n - NBIN;
  const int ph = (int)(((long long)k * j) % NFFT);
  const double a = 2.0 * ph / (double)NFFT;
  const double v = n < NBIN ? cospi(a) : -sinpi(a);
  w[(long long)j * N_pad + n] = (float)(hann(j) * v);
}
// inverse basis W[0][c][n] (c over re|im|2 pad, n over 1024 samples): irfft weights c_k/N, times the synthesis window
__global__ void inv_basis_kernel(float* w, float* win_sq) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < NFFT) { const double h = hann(idx); win_sq[idx] = (float)(h * h); }
  if (idx >= SPEC_LD * NFFT) return;
  const int c = idx / NFFT, n = idx - c * NFFT;
  double v = 0.0;
  if (c < NSPEC) {
    const int k = c < NBIN ? c : c - NBIN;
    const double ck = (k == 0 || k == NFFT / 2) ? 1.0 : 2.0;
    const int ph = (int)(((long long)k * n) % NFFT);
    const double a = 2.0 * ph / (double)NFFT;
    if (c < NBIN) v = ck * cospi(a) / NFFT;
    else v = (k == 0 || k == NFFT / 2) ? 0.0 : -ck * sinpi(a) / NFFT;   // c2r ignores the imaginary part of DC / Nyquist
  }
  w[(long long)c * NFFT + n] = (float)(v * hann(n));
}

__global__ void reflect_pad_kernel(const float* __restrict__ audio, int L, float* __restrict__ padded, long long ld_b) {
  const int b = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ld_b) return;
  float v = 0.0f;
  if (i < L + NFFT) {
    int j = i - NFFT / 2;
    if (j < 0) j = -j;
    if (j >= L) j = 2 * (L - 1) - j;
    v = (j >= 0 && j < L) ? audio[(long long)b * L + j] : 0.0f;
  }
  padded[b * ld_b + i] = v;
}

// in place on spec (B, frames, SPEC_LD): re|im -> denoised re|im ; optionally emits the magnitude of frame 0
__global__ void spectral_subtract_kernel(float* __restrict__ spec, int frames, const float* __restrict__ bias, float strength,
                                         float* __restrict__ mag0_out) {
  const long long row = blockIdx.x;  // b*frames + f
  float* s = spec + row * SPEC_LD;
  for (int k = threadIdx.x; k < NBIN; k += blockDim.x) {
    const float re = s[k], im = s[NBIN + k];
    const float mag = sqrtf(re * re + im * im);           // denoiser.py:33
    const float ang = atan2f(im, re);
    if (mag0_out && (row % frames) == 0) mag0_out[(row / frames) * NBIN + k] = mag;
    if (bias) {
      const float m2 = fmaxf(mag - bias[k] * strength, 0.0f);   // denoiser.py:61-62
      s[k] = m2 * cosf(ang);                                    // denoiser.py:43
      s[NBIN + k] = m2 * sinf(ang);
    }
  }
}

// torch.istft at output sample t of item b: overlap-add of the windowed frames divided by the overlap-added squared window,
// centre padding trimmed
__device__ __forceinline__ float overlap_add_at(const float* __restrict__ y, int frames, const float* __restrict__ win_sq, int b, int t) {
  const int tt = t + NFFT / 2;
  int f_lo = (tt - (NFFT - 1) + HOP - 1) / HOP;
  if (f_lo < 0) f_lo = 0;
  int f_hi = tt / HOP;
  if (f_hi > frames - 1) f_hi = frames - 1;
  float acc = 0.0f, env = 0.0f;
  for (int f = f_lo; f <= f_hi; ++f) {
    const int n = tt - f * HOP;
    acc += y[((long long)b * frames + f) * NFFT + n];
    env += win_sq[n];
  }
  return acc / env;
}

// lens (ragged batch, or nullptr): item b is written on [0, lens[b] * HOP) and zero beyond, where its frames were not computed
__global__ void overlap_add_kernel(const float* __restrict__ y, int frames, const float* __restrict__ win_sq, int L_out,
                                   const int* __restrict__ lens, float* __restrict__ out) {
  const int b = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= L_out) return;
  if (lens && t >= __ldg(lens + b) * HOP) { out[(long long)b * L_out + t] = 0.0f; return; }
  out[(long long)b * L_out + t] = overlap_add_at(y, frames, win_sq, b, t);
}

// overlap_add_kernel of a batch with a strength per item: an item with on[b] == 0 (on != nullptr) was not transformed and gets
// its input audio (B, L_in) unchanged, on [0, lens[b] * HOP) and zero beyond when lens != nullptr
__global__ void overlap_add_items_kernel(const float* __restrict__ y, int frames, const float* __restrict__ win_sq, int L_out,
                                         const int* __restrict__ lens, const float* __restrict__ audio, int L_in,
                                         const unsigned char* __restrict__ on, float* __restrict__ out) {
  const int b = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= L_out) return;
  float v = 0.0f;
  if (!lens || t < __ldg(lens + b) * HOP)
    v = (on && !__ldg(on + b)) ? audio[(long long)b * L_in + t] : overlap_add_at(y, frames, win_sq, b, t);
  out[(long long)b * L_out + t] = v;
}

// ---------------------------------------------------------------------------------------------- FFT path
// tw[i] = exp(-2 pi i * idx / 1024) as (cos, -sin): forward twiddles; the inverse uses the conjugate
__global__ void twiddle_kernel(float2* tw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < NFFT) { const double a = 2.0 * i / (double)NFFT; tw[i] = make_float2((float)cospi(a), (float)-sinpi(a)); }
}

__device__ __forceinline__ float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }

// one radix-4 Stockham pass over 1024 points, thread j = butterfly j (256 threads); INV: conjugate twiddles, +i rotation
template <bool INV>
__device__ __forceinline__ void fft_pass(const float2* __restrict__ in, float2* __restrict__ out, const float2* __restrict__ tw, int j, int Ns) {
  const int k = j & (Ns - 1);
  float2 v0 = in[j], v1 = in[j + 256], v2 = in[j + 512], v3 = in[j + 768];
  if (Ns > 1) {
    const int step = k * (256 / Ns);                      // angle unit: 2 pi k / (4 Ns) = 2 pi (k * 256 / Ns) / 1024
    float2 w1 = __ldg(tw + step), w2 = __ldg(tw + 2 * step), w3 = __ldg(tw + 3 * step);
    if (INV) { w1.y = -w1.y; w2.y = -w2.y; w3.y = -w3.y; }
    v1 = cmul(v1, w1); v2 = cmul(v2, w2); v3 = cmul(v3, w3);
  }
  const float2 a0 = make_float2(v0.x + v2.x, v0.y + v2.y), a1 = make_float2(v0.x - v2.x, v0.y - v2.y);
  const float2 a2 = make_float2(v1.x + v3.x, v1.y + v3.y);
  const float2 d = make_float2(v1.x - v3.x, v1.y - v3.y);
  const float2 a3 = INV ? make_float2(-d.y, d.x) : make_float2(d.y, -d.x);     // * (+i) or * (-i)
  const int j0 = ((j - k) << 2) + k;
  out[j0] = make_float2(a0.x + a2.x, a0.y + a2.y);
  out[j0 + Ns] = make_float2(a1.x + a3.x, a1.y + a3.y);
  out[j0 + 2 * Ns] = make_float2(a0.x - a2.x, a0.y - a2.y);
  out[j0 + 3 * Ns] = make_float2(a1.x - a3.x, a1.y - a3.y);
}

template <bool INV>
__device__ __forceinline__ float2* fft1024(float2* a, float2* b, const float2* tw, int j) {   // -> buffer holding the result
  fft_pass<INV>(a, b, tw, j, 1); __syncthreads();
  fft_pass<INV>(b, a, tw, j, 4); __syncthreads();
  fft_pass<INV>(a, b, tw, j, 16); __syncthreads();
  fft_pass<INV>(b, a, tw, j, 64); __syncthreads();
  fft_pass<INV>(a, b, tw, j, 256); __syncthreads();
  return b;
}

// A strength per item (ev_denoise_items, ev_to_waveform_items): item b is denoised with s[b], or not at all when on != nullptr
// and on[b] == 0.  The kernels take either this or one float for the batch; both give an item the same bits.
struct ItemStrengths { const float* s; const unsigned char* on; };
__device__ __forceinline__ float strength_of(float s, int) { return s; }
__device__ __forceinline__ float strength_of(const ItemStrengths& s, int b) { return __ldg(s.s + b); }
__device__ __forceinline__ bool denoised(float, int) { return true; }
__device__ __forceinline__ bool denoised(const ItemStrengths& s, int b) { return !s.on || __ldg(s.on + b); }

// One block per pair of frames (f0, f0 + 1), f0 even, 256 threads.  audio (B, L); y (B, frames, 1024) windowed inverse frames
// (bias != nullptr); mag0_out (B, 513): magnitude of frame 0 (the bias spectrum of ev_denoiser_init).
//   RAGGED = false: grid (ceil(frames / 2), B), every pair of every denoised item.
//   RAGGED = true: grid B * ceil(frames / 2), block i computes entry i of the compact (item, pair) list of ragged_build_table
//   (pairs[0] = its length, pairs[1 + i] = b << 16 | pair index) and blocks past its end exit.
// Both variants run the same per-pair code, so a pair's result does not depend on which of them computed it.
// S = float (one strength for the batch) or ItemStrengths; the scalar instantiations are the kernels of a single strength.
template <bool RAGGED, typename S = float>
__global__ void __launch_bounds__(256, RAGGED ? 3 : 0) denoise_fft_kernel(const float* __restrict__ audio, int L, int frames, const float2* __restrict__ tw,
                                                          const float* __restrict__ bias, S strength, float* __restrict__ y,
                                                          float* __restrict__ mag0_out, const int* __restrict__ pairs) {
  __shared__ float2 buf0[NFFT], buf1[NFFT];
  int b = blockIdx.y, f0 = blockIdx.x * 2;
  if (RAGGED) {
    if ((int)blockIdx.x >= __ldg(pairs)) return;
    const int e = __ldg(pairs + 1 + blockIdx.x);
    b = e >> 16; f0 = (e & 0xffff) * 2;
  } else if (!denoised(strength, b)) {
    return;                                                 // (the ragged list holds denoised items only)
  }
  const int f1 = f0 + 1, j = threadIdx.x;
  const float* xb = audio + (long long)b * L;
  const bool has1 = f1 < frames;
  float win[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int n = j + r * 256;
    win[r] = 0.5f - 0.5f * __ldg(tw + n).x;                // periodic hann: 0.5 - 0.5 cos(2 pi n / N)
    int i0 = f0 * HOP + n - NFFT / 2, i1 = i0 + HOP;       // torch.stft(center=True, pad_mode="reflect")
    if (i0 < 0) i0 = -i0;
    if (i0 >= L) i0 = 2 * (L - 1) - i0;
    if (i1 < 0) i1 = -i1;
    if (i1 >= L) i1 = 2 * (L - 1) - i1;
    const float x0 = (i0 >= 0 && i0 < L) ? xb[i0] : 0.0f;
    const float x1 = (has1 && i1 >= 0 && i1 < L) ? xb[i1] : 0.0f;
    buf0[n] = make_float2(win[r] * x0, win[r] * x1);
  }
  __syncthreads();
  float2* Z = fft1024<false>(buf0, buf1, tw, j);            // result in buf1
  float2* O = Z == buf1 ? buf0 : buf1;
  // two real spectra -> subtract -> Hermitian re-pack, bins k and N - k handled by one thread
  for (int k = j; k <= NFFT / 2; k += 256) {
    const float2 zk = Z[k], zn = Z[(NFFT - k) & (NFFT - 1)];
    float2 xa = make_float2(0.5f * (zk.x + zn.x), 0.5f * (zk.y - zn.y));          // frame f0
    float2 xc = make_float2(0.5f * (zk.y + zn.y), 0.5f * (zn.x - zk.x));          // frame f1: -i/2 (zk - conj zn)
    const float ma = sqrtf(xa.x * xa.x + xa.y * xa.y), mc = sqrtf(xc.x * xc.x + xc.y * xc.y);   // denoiser.py:33
    if (mag0_out && f0 == 0) mag0_out[(long long)b * NBIN + k] = ma;
    if (bias) {
      // m - bias * strength in one rounding (a fused multiply-add), spelled out: the compiler contracts it so in the scalar
      // kernels, and an instantiation that loads the strength must round the same way to give an item the same bits
      const float nb = -__ldg(bias + k), st = strength_of(strength, b);
      const float sa = ma > 0.0f ? fmaxf(__fmaf_rn(nb, st, ma), 0.0f) / ma : 0.0f, sc = mc > 0.0f ? fmaxf(__fmaf_rn(nb, st, mc), 0.0f) / mc : 0.0f;
      xa.x *= sa; xa.y *= sa; xc.x *= sc; xc.y *= sc;
      if (k == 0 || k == NFFT / 2) { xa.y = 0.0f; xc.y = 0.0f; }                  // c2r ignores the imaginary part of DC / Nyquist
      O[k] = make_float2(xa.x - xc.y, xa.y + xc.x);                               // xa + i xc
      if (k != 0 && k != NFFT / 2) O[NFFT - k] = make_float2(xa.x + xc.y, xc.x - xa.y);   // conj(xa) + i conj(xc)
    }
  }
  if (!bias) return;
  __syncthreads();
  float2* other = O == buf0 ? buf1 : buf0;
  const float2* R = fft1024<true>(O, other, tw, j);
  const float inv_n = 1.0f / NFFT;
  float* y0 = y + ((long long)b * frames + f0) * NFFT;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int n = j + r * 256;
    const float2 v = R[n];
    y0[n] = v.x * inv_n * win[r];
    if (has1) y0[NFFT + n] = v.y * inv_n * win[r];
  }
}

// lens32[b] = clamp(lengths[b], 0, max_len); wide (optional) = min(lens32[b] + extra, max_len) as int64
__global__ void ragged_lengths_kernel(const long long* __restrict__ lengths, int B, int max_len, int extra, int* __restrict__ lens32,
                                      long long* __restrict__ wide) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int n = (int)min(max(lengths[b], 0LL), (long long)max_len);
  lens32[b] = n;
  if (wide) wide[b] = min(n + extra, max_len);
}

// Mel frames past len_b that the denoised samples [0, len_b * HOP) depend on (DESIGN.md §4, ragged batches): sample t < len*HOP
// is an overlap-add of frames f <= len + 1; frame f shares its FFT with its pair partner, so pairs (f0, f0 + 1), f0 <= len + 1,
// are computed, and their windows read audio below (len + 2) * HOP + NFFT / 2 = (len + 4) * HOP.
constexpr int kDenoiseReach = 4;

// ragged_lengths_kernel of a batch with a strength per item.  lens32[b] = clamp(lengths[b], 0, max_len); table[b] = the STFT
// frames whose pairs are listed: lens32[b] + 2 for a denoised item, 0 (no pairs) for one that is not; wide (optional) = the
// frames the vocoder must get right: min(lens32[b] + kDenoiseReach, max_len) for a denoised item, lens32[b] for one that is not
__global__ void item_lengths_kernel(const long long* __restrict__ lengths, const unsigned char* __restrict__ on, int B, int max_len,
                                    int* __restrict__ lens32, int* __restrict__ table, long long* __restrict__ wide) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int n = (int)min(max(lengths[b], 0LL), (long long)max_len);
  const bool dn = !on || on[b];
  lens32[b] = n;
  table[b] = dn ? n + kDenoiseReach - 2 : 0;
  if (wide) wide[b] = dn ? min(n + kDenoiseReach, max_len) : n;
}

int ensure_basis(ev_ctx* ctx, cudaStream_t s) {
  DenoiseBasis& d = ctx->hifigan.dn;
  if (d.ready) return 0;
  void* p;
  ConvWeights f;
  f.taps = 4; f.C_in = HOP; f.N = NSPEC; f.N_pad = SPEC_LD; f.C_out = NSPEC; f.ksize = 4; f.pad = 0; f.dilation = 1; f.conv_stride = 1;
  EV_TRY(device_alloc(ctx, (size_t)NFFT * SPEC_LD * sizeof(float), &p, true, s));
  f.w_f32 = reinterpret_cast<float*>(p);
  fwd_basis_kernel<<<ceil_div(NFFT * NSPEC, 256), 256, 0, s>>>(f.w_f32, SPEC_LD);
  ConvWeights v;
  v.taps = 1; v.C_in = SPEC_LD; v.N = NFFT; v.N_pad = NFFT; v.C_out = NFFT; v.ksize = 1;
  EV_TRY(device_alloc(ctx, (size_t)SPEC_LD * NFFT * sizeof(float), &p, true, s));
  v.w_f32 = reinterpret_cast<float*>(p);
  EV_TRY(device_alloc(ctx, (size_t)NFFT * sizeof(float), &p, false, s));
  d.win_sq = reinterpret_cast<float*>(p);
  inv_basis_kernel<<<ceil_div(SPEC_LD * NFFT, 256), 256, 0, s>>>(v.w_f32, d.win_sq);
  EV_CUDA(ctx, cudaGetLastError());
  EV_TRY(device_alloc(ctx, (size_t)NFFT * sizeof(float2), &p, false, s));
  d.twiddle = p;
  twiddle_kernel<<<NFFT / 256, 256, 0, s>>>(reinterpret_cast<float2*>(p));
  EV_CUDA(ctx, cudaGetLastError());
  d.fwd = f; d.inv = v; d.ready = true;
  return 0;
}

// table (batches with a strength per item only): the frames item_lengths_kernel lists pairs for
struct DnBuffers { float* padded; float* spec; float* frames_t; int* lens32; int* table; int* pairs; long long pad_ld; int frames; };

void plan(int B, int L, Workspace& w, DnBuffers* d, bool items = false) {
  d->frames = L / HOP + 1;
  d->pad_ld = (long long)(d->frames + 3) * HOP;                 // rows of 256 samples, 3 extra rows for the 4 taps
  d->padded = w.take<float>((size_t)B * d->pad_ld);
  d->spec = w.take<float>((size_t)B * d->frames * SPEC_LD);
  d->frames_t = w.take<float>((size_t)B * d->frames * NFFT);
  d->lens32 = w.take<int>((size_t)B);                           // ragged batch: lengths and the compact pair list
  d->pairs = w.take<int>((size_t)B * ceil_div(d->frames, 2) + 1);
  d->table = items ? w.take<int>((size_t)B) : nullptr;
}

bool use_fft() {
  static const bool v = []() { const char* e = getenv("EV_DN_FFT"); return !(e && atoi(e) == 0); }();
  return v;
}

constexpr double kPairFlops = 2.0 * 5.0 * NFFT * 10.0;

// The length of the compact pair list (instrumented eager runs only, where a host copy is fine): the algorithmic work
int listed_pairs(ev_ctx* ctx, const int* pairs, double* n_pairs, cudaStream_t s) {
  if (!ctx->profiling) return 0;
  int n = 0;
  EV_CUDA(ctx, cudaMemcpyAsync(&n, pairs, sizeof(int), cudaMemcpyDeviceToHost, s));
  EV_CUDA(ctx, cudaStreamSynchronize(s));
  *n_pairs = n;
  return 0;
}

// STFT of `audio` (B, L) into d.spec (re|im); when bias != nullptr also denoise + ISTFT into out (B, HOP*(L/HOP)).
// lens32 (ragged batch, bias != nullptr, or nullptr): only the pairs that item b's samples [0, lens32[b] * HOP) read are
// computed, and out is zero beyond; what is written equals the dense result bit for bit.
int stft_pipeline(ev_ctx* ctx, const float* audio, int B, int L, const float* bias, float strength, float* mag0, float* out,
                  const int* lens32, DnBuffers& d, cudaStream_t s) {
  DenoiseBasis& bs = ctx->hifigan.dn;
  const int frames = d.frames;
  const double pair_flops = kPairFlops;
  if (use_fft() && lens32 && bias) {
    // frames [0, lens32[b] + 2) in pairs: ceil((len + 2) / 2) = floor((len + 1) / 2) + 1 pairs, all of them when len = frames - 1
    EV_LAUNCH(ctx, s, "ragged_table", 0, 8.0 * B, ragged_build_table(lens32, B, kDenoiseReach - 2, 1, 0, 2, frames, d.pairs, s));
    double n_pairs = (double)B * ceil_div(frames, 2);
    EV_TRY(listed_pairs(ctx, d.pairs, &n_pairs, s));
    EV_LAUNCH(ctx, s, "denoise_fft_ragged", pair_flops * n_pairs, 4.0 * n_pairs * 2.0 * (HOP + NFFT),
              (denoise_fft_kernel<true><<<B * ceil_div(frames, 2), 256, 0, s>>>(audio, L, frames, reinterpret_cast<const float2*>(bs.twiddle), bias,
                                                                                strength, d.frames_t, nullptr, d.pairs), cudaGetLastError()));
  } else if (use_fft()) {
    const double fft_flops = pair_flops * ceil_div(frames, 2) * B;
    EV_LAUNCH(ctx, s, "denoise_fft", fft_flops, 4.0 * B * ((double)L + (bias ? (double)frames * NFFT : NBIN)),
              (denoise_fft_kernel<false><<<dim3(ceil_div(frames, 2), B), 256, 0, s>>>(audio, L, frames, reinterpret_cast<const float2*>(bs.twiddle), bias,
                                                                                     strength, d.frames_t, mag0, nullptr), cudaGetLastError()));
  }
  if (use_fft()) {
    if (!bias) return 0;
    const int L_out = HOP * (frames - 1);
    EV_LAUNCH(ctx, s, "overlap_add", 0, 4.0 * B * (4.0 * L_out + L_out),
              (overlap_add_kernel<<<dim3(ceil_div(L_out, 256), B), 256, 0, s>>>(d.frames_t, frames, bs.win_sq, L_out, lens32, out), cudaGetLastError()));
    return 0;
  }
  EV_LAUNCH(ctx, s, "reflect_pad", 0, 8.0 * B * d.pad_ld,
            (reflect_pad_kernel<<<dim3(ceil_div((int)d.pad_ld, 256), B), 256, 0, s>>>(audio, L, d.padded, d.pad_ld), cudaGetLastError()));
  EV_CUDA(ctx, cudaMemsetAsync(d.spec, 0, (size_t)B * frames * SPEC_LD * sizeof(float), s));
  Epilogue e;
  e.out_f32 = d.spec; e.f32_ld = SPEC_LD; e.f32_bs = (long long)frames * SPEC_LD;
  // rows of 256 samples: frame f = rows f..f+3
  ConvGeom g;
  g.B = B; g.M = frames; g.N = NSPEC; g.C_in = HOP; g.taps = 4; g.conv_stride = 1; g.T_in = frames + 3;
  for (int j = 0; j < 4; ++j) g.tap_off[j] = j;
  e.T_out = frames; e.phase_cout = NSPEC;
  { LaunchScope ls(ctx, s, "stft_gemm_f32", 2.0 * B * frames * NFFT * NSPEC, 4.0 * B * frames * (HOP + NSPEC));
    cudaError_t ce = conv_simt_launch(g, d.padded, HOP, d.pad_ld, bs.fwd, e, s);
    if (ce != cudaSuccess) return cuda_fail(ctx, ce, "stft gemm"); }
  EV_LAUNCH(ctx, s, "spectral_subtract", 0, 8.0 * B * frames * NSPEC,
            (spectral_subtract_kernel<<<B * frames, 256, 0, s>>>(d.spec, frames, bias, strength, mag0), cudaGetLastError()));
  if (!bias) return 0;
  Epilogue ei;
  ei.out_f32 = d.frames_t; ei.f32_ld = NFFT; ei.f32_bs = (long long)frames * NFFT; ei.T_out = frames; ei.phase_cout = NFFT;
  ConvGeom gi;
  gi.B = B; gi.M = frames; gi.N = NFFT; gi.C_in = SPEC_LD; gi.taps = 1; gi.conv_stride = 1; gi.T_in = frames; gi.tap_off[0] = 0;
  { LaunchScope ls(ctx, s, "istft_gemm_f32", 2.0 * B * frames * NFFT * NSPEC, 4.0 * B * frames * (NFFT + NSPEC));
    cudaError_t ce = conv_simt_launch(gi, d.spec, SPEC_LD, (long long)frames * SPEC_LD, bs.inv, ei, s);
    if (ce != cudaSuccess) return cuda_fail(ctx, ce, "istft gemm"); }
  const int L_out = HOP * (frames - 1);
  EV_LAUNCH(ctx, s, "overlap_add", 0, 4.0 * B * (4.0 * L_out + L_out),
            (overlap_add_kernel<<<dim3(ceil_div(L_out, 256), B), 256, 0, s>>>(d.frames_t, frames, bs.win_sq, L_out, lens32, out), cudaGetLastError()));
  return 0;
}

// The FFT denoiser with a strength per item: `audio` (B, L) -> out (B, HOP*(L/HOP)).  lens32 (ragged batch, with d.table from
// item_lengths_kernel, or nullptr): as stft_pipeline's, the listed pairs are those of the denoised items only.  An item that is
// not denoised gets its audio (see overlap_add_items_kernel).  A denoised item's bits are those of stft_pipeline at its strength.
int denoise_items(ev_ctx* ctx, const float* audio, int B, int L, ItemStrengths st, const int* lens32, const DnBuffers& d, float* out,
                  cudaStream_t s) {
  const DenoiseBasis& bs = ctx->hifigan.dn;
  const float* bias = ctx->hifigan.denoise_bias;
  const float2* tw = reinterpret_cast<const float2*>(bs.twiddle);
  const int frames = d.frames, L_out = HOP * (frames - 1);
  if (lens32) {
    EV_LAUNCH(ctx, s, "ragged_table", 0, 8.0 * B, ragged_build_table(d.table, B, 0, 1, 0, 2, frames, d.pairs, s));
    double n_pairs = (double)B * ceil_div(frames, 2);
    EV_TRY(listed_pairs(ctx, d.pairs, &n_pairs, s));
    EV_LAUNCH(ctx, s, "denoise_fft_ragged", kPairFlops * n_pairs, 4.0 * n_pairs * 2.0 * (HOP + NFFT),
              (denoise_fft_kernel<true, ItemStrengths><<<B * ceil_div(frames, 2), 256, 0, s>>>(audio, L, frames, tw, bias, st, d.frames_t, nullptr,
                                                                                               d.pairs), cudaGetLastError()));
  } else {
    EV_LAUNCH(ctx, s, "denoise_fft", kPairFlops * ceil_div(frames, 2) * B, 4.0 * B * ((double)L + (double)frames * NFFT),
              (denoise_fft_kernel<false, ItemStrengths><<<dim3(ceil_div(frames, 2), B), 256, 0, s>>>(audio, L, frames, tw, bias, st, d.frames_t,
                                                                                                     nullptr, nullptr), cudaGetLastError()));
  }
  EV_LAUNCH(ctx, s, "overlap_add", 0, 4.0 * B * (4.0 * L_out + L_out),
            (overlap_add_items_kernel<<<dim3(ceil_div(L_out, 256), B), 256, 0, s>>>(d.frames_t, frames, bs.win_sq, L_out, lens32, audio, L, st.on, out),
             cudaGetLastError()));
  return 0;
}

// ev_to_waveform_ragged's workspace: widened lengths, the vocoded batch, the denoiser's buffers, the vocoder's workspace
struct WavBuffers { long long* wide; float* audio; DnBuffers d; char* voc_ws; size_t voc_bytes; };

void plan_to_waveform(const ev_ctx* ctx, int B, int T, Workspace& w, WavBuffers* t, bool items = false) {
  t->wide = w.take<long long>((size_t)B);
  t->audio = w.take<float>((size_t)B * T * HOP);
  plan(B, T * HOP, w, &t->d, items);
  t->voc_bytes = ev_vocode_workspace_bytes(ctx, B, T);
  t->voc_ws = w.take<char>(t->voc_bytes);
}

bool ragged_lists_fit(int B, int frames) { return B <= kRaggedMaxB && ceil_div(frames, 2) < 65536; }

// The argument checks of ev_denoise_ragged / ev_denoise_items (`name` prefixes the message)
int check_denoise_args(ev_ctx* ctx, const char* name, const float* audio, const int64_t* lengths, int B, int L, const float* out) {
  if (!ctx->hifigan.denoise_bias) return fail(ctx, EV_ERR_STATE, "ev_denoise: call ev_denoiser_init first");
  if (!audio || !out || B <= 0 || L < NFFT / 2 + 1) return fail(ctx, EV_ERR_INVALID, "ev_denoise: null argument or audio shorter than the reflect padding");
  if (lengths && !ragged_lists_fit(B, L / HOP + 1)) return fail(ctx, EV_ERR_INVALID, std::string(name) + ": batch or audio too long for the ragged pair list");
  return 0;
}

// The argument checks of ev_to_waveform_ragged / ev_to_waveform_items
int check_to_waveform_args(ev_ctx* ctx, const char* name, const float* mel, const int64_t* mel_lengths, int B, int T, int precision,
                           const float* wav) {
  const HifiganW& h = ctx->hifigan;
  const std::string n(name);
  if (!h.loaded) return fail(ctx, EV_ERR_STATE, n + ": hifigan weights not loaded");
  if (!h.denoise_bias) return fail(ctx, EV_ERR_STATE, n + ": call ev_denoiser_init first");
  if (!mel || !mel_lengths || !wav || B <= 0 || T <= 0) return fail(ctx, EV_ERR_INVALID, n + ": null argument or empty shape");
  if (h.total_up != HOP) return fail(ctx, EV_ERR_INVALID, n + ": the generator's hop must equal the denoiser's (256)");
  if (T * HOP < NFFT / 2 + 1) return fail(ctx, EV_ERR_INVALID, n + ": T < 3 frames is shorter than the reflect padding");
  if (!ragged_lists_fit(B, T + 1)) return fail(ctx, EV_ERR_INVALID, n + ": batch or T too large for the ragged pair list");
  if (precision != EV_PREC_FP32 && precision != EV_PREC_BF16) return fail(ctx, EV_ERR_INVALID, n + ": unknown precision");
  return 0;
}

// Per-item strengths are an input of the FFT kernel only; the GEMM cross-check path (EV_DN_FFT=0) takes one strength per call
int check_items_path(ev_ctx* ctx, const char* name, const float* strengths) {
  if (!strengths) return fail(ctx, EV_ERR_INVALID, std::string(name) + ": null strengths");
  if (!use_fft()) return fail(ctx, EV_ERR_INVALID, std::string(name) + ": per-item strengths need the FFT denoiser (EV_DN_FFT=0 selects the GEMM path, which takes one strength per call)");
  return 0;
}
}  // namespace

extern "C" size_t ev_denoise_workspace_bytes(const ev_ctx* ctx, int B, int L) {
  if (!ctx || B <= 0 || L <= 0) return 0;
  Workspace w(nullptr, 0);
  DnBuffers d;
  plan(B, L, w, &d);
  return w.off + 256;
}

extern "C" int ev_denoiser_init(ev_ctx* ctx, float* bias_spec_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!ctx) return EV_ERR_INVALID;
  if (!ctx->hifigan.loaded) return fail(ctx, EV_ERR_STATE, "ev_denoiser_init: hifigan weights not loaded");
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  EV_TRY(ensure_basis(ctx, s));
  HifiganW& h = ctx->hifigan;
  const int T = 88, L = T * h.total_up;                      // denoiser.py:20 mel_input = zeros(1, 80, 88)
  Workspace w(workspace, workspace_bytes);
  float* mel = w.take<float>((size_t)h.cfg.num_mels * T);
  float* wav = w.take<float>(L);
  DnBuffers d;
  plan(1, L, w, &d);
  const size_t voc_bytes = ev_vocode_workspace_bytes(ctx, 1, T);
  char* voc_ws = w.take<char>(voc_bytes);
  if (w.overflow || !workspace) return fail(ctx, EV_ERR_STATE, "ev_denoiser_init: workspace too small");
  if (!h.denoise_bias) {
    void* p;
    EV_TRY(device_alloc(ctx, NBIN * sizeof(float), &p, false, s));
    h.denoise_bias = reinterpret_cast<float*>(p);
  }
  EV_CUDA(ctx, cudaMemsetAsync(mel, 0, (size_t)h.cfg.num_mels * T * sizeof(float), s));
  EV_TRY(ev_vocode(ctx, mel, 1, T, EV_PREC_FP32, wav, voc_ws, voc_bytes, stream));
  EV_TRY(stft_pipeline(ctx, wav, 1, L, nullptr, 0.0f, h.denoise_bias, nullptr, nullptr, d, s));   // bias_spec[:, :, 0]
  if (bias_spec_out) EV_CUDA(ctx, cudaMemcpyAsync(bias_spec_out, h.denoise_bias, NBIN * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return 0;
}

extern "C" int ev_denoise_ragged(ev_ctx* ctx, const float* audio, const int64_t* lengths, int B, int L, float strength, float* out,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  if (!ctx) return EV_ERR_INVALID;
  EV_TRY(check_denoise_args(ctx, "ev_denoise_ragged", audio, lengths, B, L, out));
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  EV_TRY(ensure_basis(ctx, s));
  Workspace w(workspace, workspace_bytes);
  DnBuffers d;
  plan(B, L, w, &d);
  if (w.overflow || !workspace) return fail(ctx, EV_ERR_STATE, "ev_denoise: workspace too small");
  if (lengths)
    EV_LAUNCH(ctx, s, "ragged_lengths", 0, 12.0 * B,
              (ragged_lengths_kernel<<<ceil_div(B, 256), 256, 0, s>>>(reinterpret_cast<const long long*>(lengths), B, L / HOP, 0, d.lens32, nullptr),
               cudaGetLastError()));
  return stft_pipeline(ctx, audio, B, L, ctx->hifigan.denoise_bias, strength, nullptr, out, lengths ? d.lens32 : nullptr, d, s);
}

extern "C" int ev_denoise(ev_ctx* ctx, const float* audio, int B, int L, float strength, float* out, void* workspace,
                          size_t workspace_bytes, void* stream) {
  return ev_denoise_ragged(ctx, audio, nullptr, B, L, strength, out, workspace, workspace_bytes, stream);
}

extern "C" size_t ev_denoise_items_workspace_bytes(const ev_ctx* ctx, int B, int L) {
  if (!ctx || B <= 0 || L <= 0) return 0;
  Workspace w(nullptr, 0);
  DnBuffers d;
  plan(B, L, w, &d, true);
  return w.off + 256;
}

extern "C" int ev_denoise_items(ev_ctx* ctx, const float* audio, const int64_t* lengths, int B, int L, const float* strengths,
                                const uint8_t* denoise, float* out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!ctx) return EV_ERR_INVALID;
  EV_TRY(check_denoise_args(ctx, "ev_denoise_items", audio, lengths, B, L, out));
  EV_TRY(check_items_path(ctx, "ev_denoise_items", strengths));
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  EV_TRY(ensure_basis(ctx, s));
  Workspace w(workspace, workspace_bytes);
  DnBuffers d;
  plan(B, L, w, &d, true);
  if (w.overflow || !workspace) return fail(ctx, EV_ERR_STATE, "ev_denoise_items: workspace too small");
  if (lengths)
    EV_LAUNCH(ctx, s, "ragged_lengths", 0, 13.0 * B,
              (item_lengths_kernel<<<ceil_div(B, 256), 256, 0, s>>>(reinterpret_cast<const long long*>(lengths), denoise, B, L / HOP, d.lens32,
                                                                   d.table, nullptr), cudaGetLastError()));
  return denoise_items(ctx, audio, B, L, ItemStrengths{strengths, denoise}, lengths ? d.lens32 : nullptr, d, out, s);
}

extern "C" size_t ev_to_waveform_ragged_workspace_bytes(const ev_ctx* ctx, int B, int T) {
  if (!ctx || !ctx->hifigan.loaded || B <= 0 || T <= 0) return 0;
  Workspace w(nullptr, 0);
  WavBuffers t;
  plan_to_waveform(ctx, B, T, w, &t);
  return w.off + 256;
}

extern "C" int ev_to_waveform_ragged(ev_ctx* ctx, const float* mel, const int64_t* mel_lengths, int B, int T, int precision, float strength,
                                     float* wav, void* workspace, size_t workspace_bytes, void* stream) {
  if (!ctx) return EV_ERR_INVALID;
  EV_TRY(check_to_waveform_args(ctx, "ev_to_waveform_ragged", mel, mel_lengths, B, T, precision, wav));
  const HifiganW& h = ctx->hifigan;
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  EV_TRY(ensure_basis(ctx, s));
  Workspace w(workspace, workspace_bytes);
  WavBuffers t;
  plan_to_waveform(ctx, B, T, w, &t);
  if (w.overflow || !workspace) return fail(ctx, EV_ERR_STATE, "ev_to_waveform_ragged: workspace too small");
  // the vocoder is exact on [0, min(len + reach, T) * HOP), which holds every sample the denoised [0, len * HOP) reads
  EV_LAUNCH(ctx, s, "ragged_lengths", 0, 20.0 * B,
            (ragged_lengths_kernel<<<ceil_div(B, 256), 256, 0, s>>>(reinterpret_cast<const long long*>(mel_lengths), B, T, kDenoiseReach,
                                                                     t.d.lens32, t.wide), cudaGetLastError()));
  EV_TRY(ev_vocode_ragged(ctx, mel, reinterpret_cast<const int64_t*>(t.wide), B, T, precision, t.audio, t.voc_ws, t.voc_bytes, stream));
  return stft_pipeline(ctx, t.audio, B, T * HOP, h.denoise_bias, strength, nullptr, wav, t.d.lens32, t.d, s);
}

extern "C" size_t ev_to_waveform_items_workspace_bytes(const ev_ctx* ctx, int B, int T) {
  if (!ctx || !ctx->hifigan.loaded || B <= 0 || T <= 0) return 0;
  Workspace w(nullptr, 0);
  WavBuffers t;
  plan_to_waveform(ctx, B, T, w, &t, true);
  return w.off + 256;
}

extern "C" int ev_to_waveform_items(ev_ctx* ctx, const float* mel, const int64_t* mel_lengths, int B, int T, int precision,
                                    const float* strengths, const uint8_t* denoise, float* wav, void* workspace, size_t workspace_bytes,
                                    void* stream) {
  if (!ctx) return EV_ERR_INVALID;
  EV_TRY(check_to_waveform_args(ctx, "ev_to_waveform_items", mel, mel_lengths, B, T, precision, wav));
  EV_TRY(check_items_path(ctx, "ev_to_waveform_items", strengths));
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  EV_TRY(ensure_basis(ctx, s));
  Workspace w(workspace, workspace_bytes);
  WavBuffers t;
  plan_to_waveform(ctx, B, T, w, &t, true);
  if (w.overflow || !workspace) return fail(ctx, EV_ERR_STATE, "ev_to_waveform_items: workspace too small");
  // a denoised item needs the vocoder exact on min(len + reach, T) frames, one that is not only on its own len
  EV_LAUNCH(ctx, s, "ragged_lengths", 0, 25.0 * B,
            (item_lengths_kernel<<<ceil_div(B, 256), 256, 0, s>>>(reinterpret_cast<const long long*>(mel_lengths), denoise, B, T, t.d.lens32,
                                                                 t.d.table, t.wide), cudaGetLastError()));
  EV_TRY(ev_vocode_ragged(ctx, mel, reinterpret_cast<const int64_t*>(t.wide), B, T, precision, t.audio, t.voc_ws, t.voc_bytes, stream));
  return denoise_items(ctx, t.audio, B, T * HOP, ItemStrengths{strengths, denoise}, t.d.lens32, t.d, wav, s);
}
