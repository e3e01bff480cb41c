// Implicit-GEMM 1-D convolution: geometry, fused epilogue and weight layouts shared by the two back ends
//   conv_simt.cu : fp32 CUDA-core kernel, fixed summation order (text encoder always; parity mode elsewhere)
//   conv_tc.cu   : bf16 tcgen05/TMEM kernel fed by TMA (decoder + vocoder in EV_PREC_BF16)
//
// All activations are CHANNEL-LAST: element (b, t, c) of a tensor lives at  base + b*bs + t*ld + c.
// One GEMM row = one output time step, K = taps x C_in, N = C_out.  Every reference op on the path maps onto it:
//   nn.Conv1d(k, dilation d, "same")      taps=k,  t_in = t + j*d - pad
//   nn.Conv1d(3, stride 2, pad 1)         taps=3,  t_in = 2t + j - 1                       (decoder.py:67)
//   nn.ConvTranspose1d(k=2s, stride s, p) polyphase: GEMM row r holds outputs t = s*r + phase - p,
//                                         N = s*C_out, taps=2 (t_in = r, r-1)               (decoder.py:144, hifigan/models.py:160)
//   nn.Linear / 1x1 conv                  taps=1
#pragma once
#include "common.cuh"

struct CUtensorMap_st;

namespace ev {

constexpr int kMaxTaps = 16;

struct ConvGeom {
  int B;            // batch items
  int M;            // GEMM rows per batch item
  int N;            // GEMM columns (C_out, or s*C_out for the polyphase transposed conv)
  int C_in;         // channels reduced per tap
  int taps;
  int conv_stride;  // input rows advanced per GEMM row
  int T_in;         // valid input rows per batch item (outside -> zero padding)
  int tap_off[kMaxTaps];  // t_in = row*conv_stride + tap_off[j]
};

// out value  v = ((acc + bias) [*mask] * alpha + res + res2) / div
// out_f32 <- v ;  out_act <- act(v) [*mask]
struct Epilogue {
  const float* bias = nullptr;      // [C_out]
  const float* res = nullptr;       long long res_ld = 0, res_bs = 0;
  const float* res2 = nullptr;      long long res2_ld = 0, res2_bs = 0;
  float* out_f32 = nullptr;         long long f32_ld = 0, f32_bs = 0;
  void* out_act = nullptr;          long long act_ld = 0, act_bs = 0;   // float (SIMT) or bf16 (TC)
  RowMask mask = {nullptr, 0};
  int mask_pre = 0, mask_act = 0;
  float alpha = 1.0f, div = 1.0f;
  int f32_is_act = 0;  // tensor-core path: out_f32 receives the activated, masked value instead of the pre-activation one
  int act = ACT_NONE;
  float slope = 0.0f;
  const float* snake_a = nullptr;     // exp(alpha)            [C_out]
  const float* snake_invb = nullptr;  // 1/(exp(beta)+1e-9)    [C_out]
  int phase_cout = 0;  // C_out per phase (== N for ordinary convs)
  int up_s = 1, up_p = 0;
  int T_out = 0;       // valid output rows per batch item
  // optional fused GroupNorm statistics of the fp32 output (tensor-core path, 32 channels per group): per (b, group)
  // sum and sum of squares over ALL rows are accumulated into gn_sum[(b*G + g)*2 + {0,1}] (zeroed by the caller)
  double* gn_sum = nullptr;
  int gn_groups = 0;
};

// (GEMM row r, GEMM column n) -> (output time t, output channel co); returns false when the slot is outside the output.
__device__ __forceinline__ bool ep_coord(const Epilogue& e, int r, int n, int& t, int& co) {
  int phase = n / e.phase_cout;
  co = n - phase * e.phase_cout;
  t = e.up_s * r + phase - e.up_p;
  return t >= 0 && t < e.T_out;
}

__device__ __forceinline__ float ep_value(const Epilogue& e, int b, int t, int co, float acc, float maskv) {
  float v = acc + (e.bias ? __ldg(e.bias + co) : 0.0f);
  if (e.mask_pre && maskv == 0.0f) v = 0.0f;   // select: a padded row may hold a non-finite value
  v *= e.alpha;
  if (e.res) v += e.res[b * e.res_bs + (long long)t * e.res_ld + co];
  if (e.res2) v += e.res2[b * e.res2_bs + (long long)t * e.res2_ld + co];
  if (e.div != 1.0f) v = v / e.div;
  return v;
}

__device__ __forceinline__ float ep_act(const Epilogue& e, int co, float v, float maskv) {
  float sa = 0.0f, sb = 0.0f;
  if (e.act == ACT_SNAKE) { sa = __ldg(e.snake_a + co); sb = __ldg(e.snake_invb + co); }
  float w = apply_act(v, e.act, e.slope, sa, sb);
  if (e.mask_act && maskv == 0.0f) w = 0.0f;
  return w;
}

// Packed weights of one convolution / linear layer, both layouts (owned by the context).
struct ConvWeights {
  float* w_f32 = nullptr;   // [taps][C_in][N_pad]      (N contiguous; SIMT B-operand)
  bf16* w_bf16 = nullptr;   // [taps][N_pad128][K_pad]  (C_in contiguous, K-major; TMA/UMMA B-operand)
  float* w_tf32 = nullptr;  // [taps][N_pad128][3*K32]  split fp32 for the 3xTF32 path: [hi | lo | hi], K32 = C_in padded to 32
  // 3xFP16 split (the faster fp32-accurate path): w * 2^e as [hi | lo | hi] halves, [taps][N_pad128][3*C_in] (C_in % 64 == 0);
  // e is chosen per layer so that max |w| 2^e lies in [2^13, 2^14): both halves of every weight of ordinary size are normal fp16
  // numbers.  f16_scale[0] = 2^e, f16_scale[1] = 2^-e / kF16ActScale (what the epilogue multiplies the accumulator with).
  void* w_f16x3 = nullptr; float* f16_scale = nullptr;
  int K32 = 0;
  float* bias = nullptr;    // [C_out] or nullptr
  int taps = 0, C_in = 0, N = 0, N_pad = 0, N_pad_tc = 0, K_pad = 0;
  // geometry template
  int conv_stride = 1, dilation = 1, pad = 0, transposed = 0, up_s = 1, up_p = 0, C_out = 0, ksize = 1;
};

// ---- ragged batches (ragged.cu) ---------------------------------------------------------------------------------
// The vocoder is purely convolutional, so the samples of utterance b up to len_b*hop depend only on mel frames up to
// len_b + (receptive field); tiles that start beyond (len_b + margin) * rows_per_frame are never computed.  The tile
// kernels walk a COMPACT list of (item, m-tile) pairs instead of the dense B x m_tiles grid:
//     table[0] = number of pairs,  table[1 + i] = (b << 16) | m_tile      (built on the device from the lengths, so a
// captured CUDA graph follows the lengths of each replay).  Tables are cached per (rows_per_frame, len_shift, tile_rows, M, margin).
struct RaggedPlanner {
  const int* lens = nullptr;      // device [B], valid frames per item; nullptr = dense batch
  int B = 0, margin = 0;          // margin in frames (>= the generator's receptive field, see hifigan.cu)
  int rows_per_frame = 1;         // GEMM rows per frame of the launches that follow (set by the caller per stage)
  int len_shift = 0;              // frames valid at this level = ceil(lens[b] / 2^len_shift) (decoder half-rate levels)
  int* arena = nullptr;           // table storage (caller's workspace)
  size_t arena_ints = 0, arena_off = 0;
  struct Entry { int rpf, shift, tile_rows, M, margin; const int* table; };
  Entry cache[32];
  int n_cache = 0;
  long long* launch_counter = nullptr;   // bumped once per table kernel (the context's launch statistics)
  // optional side branch: table kernels only depend on the lengths, so they are issued on `side` (which the caller has made
  // wait for the lengths) and the consumer's stream waits for `ready` -- in a captured graph every table is then built at the
  // very beginning, next to the first layers, instead of sitting in front of its first consumer
  cudaStream_t side = nullptr;
  cudaEvent_t ready = nullptr;
  bool active() const { return lens != nullptr; }
  // compact tile list for tiles of `tile_rows` GEMM rows over M rows per item; nullptr -> run dense (always correct)
  const int* table(int tile_rows, int M, cudaStream_t s);
};
constexpr int kRaggedMaxB = 2048;
// one table, built directly: item b needs rows [0, min(M, (ceil(lens[b] / 2^len_shift) + margin) * rows_per_frame)); `table`
// holds B * ceil(M / tile_rows) + 1 ints
cudaError_t ragged_build_table(const int* lens, int B, int margin, int rows_per_frame, int len_shift, int tile_rows, int M, int* table,
                               cudaStream_t s);

// conv_simt.cu
cudaError_t conv_simt_launch(const ConvGeom& g, const float* x, long long x_ld, long long x_bs, const ConvWeights& w,
                             const Epilogue& e, cudaStream_t stream);
// conv_tc.cu
// Per-call schedule: -1 keeps what the EV_TC_* switch chooses (EV_TC_LEAN, EV_TC_MB, EV_TC_CTA2, EV_TC_WIDE, EV_TC_RESIDENT,
// EV_TC_BK32, EV_TC_HALO, EV_TF32_SHARE); lean / resident / bk32 / halo / share 0 or 1, mb 1 or 2, ctas_per_sm 1 or 2, epi_warps 8 or
// 16 force that choice.  A forced choice the launch cannot honour fails it (cudaErrorInvalidValue and a message in *err); it is
// never swapped for another variant.  Forcing only picks among plans that pass the launcher's shared-memory and TMEM guards.
struct TcSchedule { int lean = -1, mb = -1, ctas_per_sm = -1, epi_warps = -1, resident = -1, bk32 = -1, halo = -1, share = -1; };
// What a launch ran: tile width BN, m-blocks per tile, CTAs per SM, epilogue warps, MMA issuer warps, resident weights, activation /
// weight ring slots, K-chunk width, halo reuse (one activation tile serves several taps), TMA boxes per activation tile, lean
// activation-only epilogue, vector epilogue (else the scalar one), split mode (0 bf16, 1 3xTF32, 2 3xFP16), accumulation groups per
// tile (> 1: the two-level flush), 3xTF32 operand sharing, compact (ragged) tile list, grid, tiles of the dense batch.
struct TcLaunchInfo {
  int bn = 0, mb = 0, ctas_per_sm = 0, epi_warps = 0, issuers = 0, resident = 0, a_slots = 0, b_slots = 0, bk = 0, halo = 0, a_boxes = 0,
      act_only = 0, vec_ok = 0, split = 0, flush_groups = 0, tf32_share = 0, ragged = 0, grid = 0, total_tiles = 0;
};
// x: bf16 activations, or (tf32x3 != 0) the split fp32 pair [hi | lo] of width 2*C_in per row (x_ld, x_bs in elements)
// split: 0 = bf16 operands; 1 = 3xTF32 (x: the fp32 pair [hi | lo], 2*C_in floats per row); 2 = 3xFP16 (x: [hi | lo] halves, 2*C_in per row)
cudaError_t conv_tc_launch(const ConvGeom& g, const void* x, long long x_ld, long long x_bs, int tf32x3,
                           const ConvWeights& w, const Epilogue& e, cudaStream_t stream, std::string* err,
                           RaggedPlanner* ragged = nullptr, const TcSchedule* sched = nullptr, TcLaunchInfo* info = nullptr);
bool conv_tc_init(std::string* err);
// 3-D bf16 tensor map (dims d0 fastest; strides in bytes for d1, d2; box b0 x b1 x 1; swizzle 128 or 64 bytes)
bool tc_encode_bf16_map(::CUtensorMap_st* map, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t s1_bytes,
                        uint64_t s2_bytes, uint32_t b0, uint32_t b1, int swizzle_bytes, std::string* err);
int tc_sm_count();
cudaError_t conv_tc_read_trace(unsigned long long* host, int n);   // diagnostic: clock stamps of the last traced launch

// resblock_tc.cu: one fused HiFi-GAN ResBlock1 (six convs, residual stream resident in TMEM)
// Per-call schedule: -1 keeps the EV_RB_* switch (EV_RB_CLUSTER, EV_RB_OCC2, EV_RB_WAVE, EV_RB_RESIDENT, same values); any other value
// is forced, and a forced choice the kernel cannot honour for this block fails the launch instead of running another variant.
struct RbSchedule { int cluster = -1, occ2 = -1, wave = -1, resident = -1; };
// What a launch ran: CTAs per cluster, CTAs per SM, wavefront schedule, resident weights, weight ring slots, epilogue warps, grid,
// output rows per (cluster) window and windows of the dense batch.
struct RbLaunchInfo { int cl = 0, occ = 0, wave = 0, resident = 0, w_slots = 0, n_epi = 0, grid = 0, Wv = 0, total_tiles = 0; };
bool resblock_tc_supported(int C, int k, const int* dil);
cudaError_t resblock_tc_launch(int C, int k, const ConvWeights* const c1[3], const ConvWeights* const c2[3], const float* const bacc[3],
                               const float* x, float* sum, bf16* act_out, int B, int L, int mode, float inv_n, float slope_out,
                               int write_f32, cudaStream_t s, std::string* err, RaggedPlanner* ragged = nullptr,
                               const RbSchedule* sched = nullptr, RbLaunchInfo* info = nullptr);
int conv_tc_pick_bn(int N);

// ff_tc.cu: LayerNorm -> Linear(256 -> inner) -> SnakeBeta -> Linear(inner -> 256) -> + residual -> * mask, one kernel
struct FfTcArgs {
  const float* x = nullptr;             // fp32 residual stream (b, t, 256), dense
  // attention tail mode (instead of x): x = xr_cf + att Wo^T + bo is formed in the kernel
  const bf16* att = nullptr; long long att_ld = 0, att_bs = 0;   // attention output (b, t, 128) bf16
  const ConvWeights* oproj = nullptr;                            // Linear(128 -> 256) + bias
  const float* xr_cf = nullptr;                                  // fp32 residual stream, CHANNEL-FIRST (b, 256, t)
  const float* ln_g = nullptr; const float* ln_b = nullptr; float eps = 1e-5f;
  const ConvWeights* ff1 = nullptr; const ConvWeights* ff2 = nullptr;
  const float* snake_a = nullptr; const float* snake_invb = nullptr;
  bf16* out = nullptr; long long out_ld = 0, out_bs = 0;   // (b, t, 256) bf16 operand of the next conv, masked
  const int* lens = nullptr; int len_shift = 0;
  int B = 0, T = 0;
  // optional compact list of the 128-row tiles that hold at least one valid row (ragged_build_table, margin 0): the output
  // of a padded row is zero whatever its input, so tiles without a valid row are not computed, only zero-filled
  const int* tiles = nullptr;
};
bool ff_tc_supported(const ConvWeights& ff1, const ConvWeights& ff2);
bool ff_tc_oproj_supported(const ConvWeights& wo);
cudaError_t ff_tc_launch(const FfTcArgs& a, cudaStream_t s, std::string* err);
cudaError_t ff_tc_read_trace(unsigned long long* host, int n);   // diagnostic (EV_FF_DEBUG & 16)

// resnet_tc.cu: one whole ResnetBlock1D (+ the following pre-LayerNorm) per launch; conv2 == nullptr -> conv -> GN -> Mish -> mask only
struct ResnetTcArgs {
  const bf16* x = nullptr; long long x_ld = 0, x_bs = 0;   // masked bf16 block input (b, t, C_in)
  const ConvWeights* conv1 = nullptr; const ConvWeights* conv2 = nullptr; const ConvWeights* res = nullptr;
  const float *gn_g1 = nullptr, *gn_b1 = nullptr, *gn_g2 = nullptr, *gn_b2 = nullptr;
  const float* temb = nullptr;                              // [256] time embedding of this block and step
  long long temb_bs = 0;                                    // item stride of temb (0: shared by the batch)
  const float *ln_g = nullptr, *ln_b = nullptr;
  const int* lens = nullptr; int len_shift = 0;
  int B = 0, T = 0;
  bf16* a_buf = nullptr; long long a_ld = 0, a_bs = 0;      // the output when conv2 == nullptr; else an optional copy of conv2's operand (tests)
  float* xr = nullptr; bf16* n_out = nullptr;               // (b, t, 256) dense outputs of the full block
  float* xr_cf = nullptr;                                   // instead of xr: the fp32 stream channel-first (b, 256, t)
  // optional (with xr_cf): the attention's stacked q|k|v projection (Linear 256 -> 384, no bias) of n, in the same launch; n_out is
  // then not written (nobody else reads it)
  const ConvWeights* qkv = nullptr; bf16* qkv_out = nullptr;   // (b, t, 384) dense
};
bool resnet_tc_qkv_supported(const ConvWeights& qkv);
int resnet_tc_plan(int B, int T);
bool resnet_tc_supported(const ConvWeights& conv1, const ConvWeights* conv2, const ConvWeights* res, int B, int T);
cudaError_t resnet_tc_launch(const ResnetTcArgs& a, cudaStream_t s, std::string* err);
cudaError_t resnet_tc_read_trace(unsigned long long* host, int n);

}  // namespace ev
