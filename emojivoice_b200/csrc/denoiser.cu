// Bias denoiser (hifigan/denoiser.py:7-64): centred hann STFT(n_fft 1024, hop 256) -> magnitude minus
// strength*bias_spec, clamped at 0 -> inverse STFT with the original phase.
//
// ONE kernel per PAIR of frames does the whole spectral path in shared memory:
//     z[n] = hann[n] * (x_f[n] + i x_{f+1}[n])  ->  1024-point complex FFT (radix-4 Stockham, 5 passes)
//     X_f[k] = (Z[k] + conj Z[N-k]) / 2,  X_{f+1}[k] = (Z[k] - conj Z[N-k]) / 2i          (two real spectra from one FFT)
//     X'[k] = X[k] * max(|X[k]| - strength * bias[k], 0) / |X[k]|                          (denoiser.py:61-62, phase kept)
//     Z'[k] = X'_f[k] + i X'_{f+1}[k] (Hermitian extension)  ->  inverse FFT  ->  y_f = Re z' hann, y_{f+1} = Im z' hann
// followed by the overlap-add / window-envelope normalisation of torch.istft.  2.2 GFLOP per config-2 batch, fp32 throughout
// (twiddles and window from tables computed in double precision); the reflect padding of torch.stft(center=True) is folded
// into the loads.  The strength is one number for the batch or one per item, and an item may be left undenoised; a ragged
// batch transforms only the frame pairs each item's valid samples read.  Every entry point runs the same pipeline.
#include "ctx.cuh"

using namespace ev;

namespace {
cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

constexpr int NFFT = 1024, HOP = 256, NBIN = NFFT / 2 + 1;


__device__ __forceinline__ double hann(int j) { return 0.5 - 0.5 * cospi(2.0 * j / (double)NFFT); }  // periodic hann

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

// lens (ragged batch, or nullptr): item b is written on [0, lens[b] * HOP) and zero beyond, where its frames were not computed.
// on (or nullptr: every item is denoised): an item with on[b] == 0 was not transformed and gets its input audio (B, L_in)
__global__ void overlap_add_kernel(const float* __restrict__ y, int frames, const float* __restrict__ win_sq, int L_out,
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

// tw[i] = exp(-2 pi i * idx / 1024) as (cos, -sin): forward twiddles; the inverse uses the conjugate.  win_sq[i] = hann[i]^2,
// the window envelope of the overlap-add.
__global__ void twiddle_kernel(float2* tw, float* win_sq) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= NFFT) return;
  const double a = 2.0 * i / (double)NFFT, h = hann(i);
  tw[i] = make_float2((float)cospi(a), (float)-sinpi(a));
  win_sq[i] = (float)(h * h);
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

// The denoiser's strength: s for every item (items == nullptr) or items[b] (ev_denoise_items, ev_to_waveform_items, device
// memory); with items, item b is denoised at all unless on != nullptr and on[b] == 0.
struct Strength { float s; const float* items; const unsigned char* on; };

// The FFT kernel takes S = float (one strength for the batch, every item denoised) or S = Strength with items != nullptr.  As
// a kernel parameter the strength is an operand of the spectral cut; reading it per item instead measured 0.6 % more time in
// the dense kernel (B200, 1000 W, 32 x 668), so the scalar calls keep their own instantiations.
__device__ __forceinline__ float strength_of(float s, int) { return s; }
__device__ __forceinline__ float strength_of(const Strength& s, int b) { return __ldg(s.items + b); }
__device__ __forceinline__ bool denoised(float, int) { return true; }
__device__ __forceinline__ bool denoised(const Strength& s, int b) { return !s.on || __ldg(s.on + b); }

// One block per pair of frames (f0, f0 + 1), f0 even, 256 threads.  audio (B, L); y (B, frames, 1024) windowed inverse frames
// (bias != nullptr); mag0_out (B, 513): magnitude of frame 0 (the bias spectrum of ev_denoiser_init).
//   RAGGED = false: grid (ceil(frames / 2), B), every pair of every denoised item.
//   RAGGED = true: grid B * ceil(frames / 2), block i computes entry i of the compact (item, pair) list of ragged_build_table
//   (pairs[0] = its length, pairs[1 + i] = b << 16 | pair index) and blocks past its end exit.
// Both variants run the same per-pair code, so a pair's result does not depend on which of them computed it.
template <bool RAGGED, typename S>
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
      // m - bias * strength in one rounding (a fused multiply-add), spelled out: the compiler contracts it for a strength that is
      // a kernel parameter but not necessarily for one loaded from memory, and both must give an item the same bits
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

// Mel frames past len_b that the denoised samples [0, len_b * HOP) depend on (DESIGN.md §4, ragged batches): sample t < len*HOP
// is an overlap-add of frames f <= len + 1; frame f shares its FFT with its pair partner, so pairs (f0, f0 + 1), f0 <= len + 1,
// are computed, and their windows read audio below (len + 2) * HOP + NFFT / 2 = (len + 4) * HOP.
constexpr int kDenoiseReach = 4;

// The lengths of a ragged batch.  lens32[b] = clamp(lengths[b], 0, max_len); table[b] = the STFT frames whose pairs are listed:
// lens32[b] + 2 for a denoised item, 0 (no pairs) for one that is not (on != nullptr and on[b] == 0); wide (optional) = the
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

int ensure_tables(ev_ctx* ctx, cudaStream_t s) {
  DenoiseTables& d = ctx->hifigan.dn;
  if (d.ready) return 0;
  void* p;
  EV_TRY(device_alloc(ctx, (size_t)NFFT * sizeof(float), &p, false, s));
  d.win_sq = reinterpret_cast<float*>(p);
  EV_TRY(device_alloc(ctx, (size_t)NFFT * sizeof(float2), &p, false, s));
  d.twiddle = reinterpret_cast<float2*>(p);
  twiddle_kernel<<<NFFT / 256, 256, 0, s>>>(d.twiddle, d.win_sq);
  EV_CUDA(ctx, cudaGetLastError());
  d.ready = true;
  return 0;
}

// frames_t: the windowed inverse frames; lens32, table, pairs: a ragged batch's lengths, the frames item_lengths_kernel lists
// pairs for, and the compact pair list
struct DnBuffers { float* frames_t; int* lens32; int* table; int* pairs; int frames; };

void plan(int B, int L, Workspace& w, DnBuffers* d) {
  d->frames = L / HOP + 1;
  d->frames_t = w.take<float>((size_t)B * d->frames * NFFT);
  d->lens32 = w.take<int>((size_t)B);
  d->pairs = w.take<int>((size_t)B * ceil_div(d->frames, 2) + 1);
  d->table = w.take<int>((size_t)B);
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

// item_lengths_kernel of a ragged batch into d.lens32 / d.table (and wide); bytes: lengths and flags read, the rest written
int item_lengths(ev_ctx* ctx, const int64_t* lengths, const unsigned char* on, int B, int max_len, DnBuffers& d, long long* wide,
                 cudaStream_t s) {
  EV_LAUNCH(ctx, s, "ragged_lengths", 0, B * (8.0 + (on ? 1.0 : 0.0) + 4.0 + 4.0 + (wide ? 8.0 : 0.0)),
            (item_lengths_kernel<<<ceil_div(B, 256), 256, 0, s>>>(reinterpret_cast<const long long*>(lengths), on, B, max_len, d.lens32,
                                                                 d.table, wide), cudaGetLastError()));
  return 0;
}

// denoise_fft_kernel<RAGGED, S> for the strength st: S = float when it is one number for the batch
template <bool RAGGED>
cudaError_t launch_denoise_fft(dim3 grid, cudaStream_t s, const float* audio, int L, int frames, const float2* tw, const float* bias,
                               Strength st, float* y, float* mag0_out, const int* pairs) {
  if (st.items) denoise_fft_kernel<RAGGED, Strength><<<grid, 256, 0, s>>>(audio, L, frames, tw, bias, st, y, mag0_out, pairs);
  else denoise_fft_kernel<RAGGED, float><<<grid, 256, 0, s>>>(audio, L, frames, tw, bias, st.s, y, mag0_out, pairs);
  return cudaGetLastError();
}

// The denoiser: `audio` (B, L) -> out (B, HOP*(L/HOP)).  lens32 (ragged batch, with d.table from item_lengths_kernel, or
// nullptr): only the pairs that a denoised item b's samples [0, lens32[b] * HOP) read are computed, and out is zero beyond;
// what is written equals the dense result bit for bit.  An item that is not denoised gets its audio (see overlap_add_kernel).
int run_denoiser(ev_ctx* ctx, const float* audio, int B, int L, Strength st, const int* lens32, const DnBuffers& d, float* out,
                 cudaStream_t s) {
  const DenoiseTables& tb = ctx->hifigan.dn;
  const float* bias = ctx->hifigan.denoise_bias;
  const int frames = d.frames, L_out = HOP * (frames - 1);
  if (lens32) {
    // frames [0, table[b]) in pairs: ceil((len + 2) / 2) = floor((len + 1) / 2) + 1 pairs, all of them when len = frames - 1
    EV_LAUNCH(ctx, s, "ragged_table", 0, 8.0 * B, ragged_build_table(d.table, B, 0, 1, 0, 2, frames, d.pairs, s));
    double n_pairs = (double)B * ceil_div(frames, 2);
    EV_TRY(listed_pairs(ctx, d.pairs, &n_pairs, s));
    EV_LAUNCH(ctx, s, "denoise_fft_ragged", kPairFlops * n_pairs, 4.0 * n_pairs * 2.0 * (HOP + NFFT),
              launch_denoise_fft<true>(B * ceil_div(frames, 2), s, audio, L, frames, tb.twiddle, bias, st, d.frames_t, nullptr, d.pairs));
  } else {
    EV_LAUNCH(ctx, s, "denoise_fft", kPairFlops * ceil_div(frames, 2) * B, 4.0 * B * ((double)L + (double)frames * NFFT),
              launch_denoise_fft<false>(dim3(ceil_div(frames, 2), B), s, audio, L, frames, tb.twiddle, bias, st, d.frames_t, nullptr, nullptr));
  }
  EV_LAUNCH(ctx, s, "overlap_add", 0, 4.0 * B * (4.0 * L_out + L_out),
            (overlap_add_kernel<<<dim3(ceil_div(L_out, 256), B), 256, 0, s>>>(d.frames_t, frames, tb.win_sq, L_out, lens32, audio, L, st.on, out),
             cudaGetLastError()));
  return 0;
}

// ev_to_waveform_*'s workspace: widened lengths, the vocoded batch, the denoiser's buffers, the vocoder's workspace
struct WavBuffers { long long* wide; float* audio; DnBuffers d; char* voc_ws; size_t voc_bytes; };

void plan_to_waveform(const ev_ctx* ctx, int B, int T, Workspace& w, WavBuffers* t) {
  t->wide = w.take<long long>((size_t)B);
  t->audio = w.take<float>((size_t)B * T * HOP);
  plan(B, T * HOP, w, &t->d);
  t->voc_bytes = ev_vocode_workspace_bytes(ctx, B, T);
  t->voc_ws = w.take<char>(t->voc_bytes);
}

bool ragged_lists_fit(int B, int frames) { return B <= kRaggedMaxB && ceil_div(frames, 2) < 65536; }

// The argument checks of ev_denoise / ev_denoise_ragged / ev_denoise_items (`name` prefixes the message)
int check_denoise_args(ev_ctx* ctx, const char* name, const float* audio, const int64_t* lengths, int B, int L, const float* out) {
  const std::string n(name);
  if (!ctx->hifigan.denoise_bias) return fail(ctx, EV_ERR_STATE, n + ": call ev_denoiser_init first");
  if (!audio || !out || B <= 0 || L < NFFT / 2 + 1) return fail(ctx, EV_ERR_INVALID, n + ": null argument or audio shorter than the reflect padding");
  if (lengths && !ragged_lists_fit(B, L / HOP + 1)) return fail(ctx, EV_ERR_INVALID, n + ": batch or audio too long for the ragged pair list");
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

// The per-item entry points take their strengths from device memory
int check_strengths(ev_ctx* ctx, const char* name, const float* strengths) {
  if (!strengths) return fail(ctx, EV_ERR_INVALID, std::string(name) + ": null strengths");
  return 0;
}

// ev_denoise, ev_denoise_ragged (lengths) and ev_denoise_items (per_item)
int denoise_call(ev_ctx* ctx, const char* name, const float* audio, const int64_t* lengths, int B, int L, Strength st, bool per_item,
                 float* out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!ctx) return EV_ERR_INVALID;
  EV_TRY(check_denoise_args(ctx, name, audio, lengths, B, L, out));
  if (per_item) EV_TRY(check_strengths(ctx, name, st.items));
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  EV_TRY(ensure_tables(ctx, s));
  Workspace w(workspace, workspace_bytes);
  DnBuffers d;
  plan(B, L, w, &d);
  if (w.overflow || !workspace) return fail(ctx, EV_ERR_STATE, std::string(name) + ": workspace too small");
  if (lengths) EV_TRY(item_lengths(ctx, lengths, st.on, B, L / HOP, d, nullptr, s));
  return run_denoiser(ctx, audio, B, L, st, lengths ? d.lens32 : nullptr, d, out, s);
}

// ev_to_waveform_ragged and ev_to_waveform_items (per_item)
int to_waveform_call(ev_ctx* ctx, const char* name, const float* mel, const int64_t* mel_lengths, int B, int T, int precision, Strength st,
                     bool per_item, float* wav, void* workspace, size_t workspace_bytes, void* stream) {
  if (!ctx) return EV_ERR_INVALID;
  EV_TRY(check_to_waveform_args(ctx, name, mel, mel_lengths, B, T, precision, wav));
  if (per_item) EV_TRY(check_strengths(ctx, name, st.items));
  cudaStream_t s = as_stream(stream);
  EV_CUDA(ctx, cudaSetDevice(ctx->device));
  EV_TRY(ensure_tables(ctx, s));
  Workspace w(workspace, workspace_bytes);
  WavBuffers t;
  plan_to_waveform(ctx, B, T, w, &t);
  if (w.overflow || !workspace) return fail(ctx, EV_ERR_STATE, std::string(name) + ": workspace too small");
  // a denoised item needs the vocoder exact on min(len + reach, T) frames, which hold every sample its denoised [0, len * HOP)
  // reads; one that is not only on its own len
  EV_TRY(item_lengths(ctx, mel_lengths, st.on, B, T, t.d, t.wide, s));
  EV_TRY(ev_vocode_ragged(ctx, mel, reinterpret_cast<const int64_t*>(t.wide), B, T, precision, t.audio, t.voc_ws, t.voc_bytes, stream));
  return run_denoiser(ctx, t.audio, B, T * HOP, st, t.d.lens32, t.d, wav, s);
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
  EV_TRY(ensure_tables(ctx, s));
  HifiganW& h = ctx->hifigan;
  const int T = 88, L = T * h.total_up, frames = L / HOP + 1;   // denoiser.py:20 mel_input = zeros(1, 80, 88)
  Workspace w(workspace, workspace_bytes);
  float* mel = w.take<float>((size_t)h.cfg.num_mels * T);
  float* wav = w.take<float>(L);
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
  // bias_spec[:, :, 0]: the magnitude of frame 0, which the forward half of the denoiser writes when it has no bias to subtract
  EV_LAUNCH(ctx, s, "denoise_fft", kPairFlops * ceil_div(frames, 2), 4.0 * ((double)L + NBIN),
            (denoise_fft_kernel<false, float><<<dim3(ceil_div(frames, 2), 1), 256, 0, s>>>(wav, L, frames, h.dn.twiddle, nullptr, 0.0f, nullptr,
                                                                                          h.denoise_bias, nullptr), cudaGetLastError()));
  if (bias_spec_out) EV_CUDA(ctx, cudaMemcpyAsync(bias_spec_out, h.denoise_bias, NBIN * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return 0;
}

extern "C" int ev_denoise_ragged(ev_ctx* ctx, const float* audio, const int64_t* lengths, int B, int L, float strength, float* out,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  return denoise_call(ctx, "ev_denoise_ragged", audio, lengths, B, L, Strength{strength, nullptr, nullptr}, false, out, workspace,
                      workspace_bytes, stream);
}

extern "C" int ev_denoise(ev_ctx* ctx, const float* audio, int B, int L, float strength, float* out, void* workspace,
                          size_t workspace_bytes, void* stream) {
  return denoise_call(ctx, "ev_denoise", audio, nullptr, B, L, Strength{strength, nullptr, nullptr}, false, out, workspace,
                      workspace_bytes, stream);
}

extern "C" size_t ev_denoise_items_workspace_bytes(const ev_ctx* ctx, int B, int L) { return ev_denoise_workspace_bytes(ctx, B, L); }

extern "C" int ev_denoise_items(ev_ctx* ctx, const float* audio, const int64_t* lengths, int B, int L, const float* strengths,
                                const uint8_t* denoise, float* out, void* workspace, size_t workspace_bytes, void* stream) {
  return denoise_call(ctx, "ev_denoise_items", audio, lengths, B, L, Strength{0.0f, strengths, denoise}, true, out, workspace,
                      workspace_bytes, stream);
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
  return to_waveform_call(ctx, "ev_to_waveform_ragged", mel, mel_lengths, B, T, precision, Strength{strength, nullptr, nullptr}, false,
                          wav, workspace, workspace_bytes, stream);
}

extern "C" size_t ev_to_waveform_items_workspace_bytes(const ev_ctx* ctx, int B, int T) {
  return ev_to_waveform_ragged_workspace_bytes(ctx, B, T);
}

extern "C" int ev_to_waveform_items(ev_ctx* ctx, const float* mel, const int64_t* mel_lengths, int B, int T, int precision,
                                    const float* strengths, const uint8_t* denoise, float* wav, void* workspace, size_t workspace_bytes,
                                    void* stream) {
  return to_waveform_call(ctx, "ev_to_waveform_items", mel, mel_lengths, B, T, precision, Strength{0.0f, strengths, denoise}, true, wav,
                          workspace, workspace_bytes, stream);
}
