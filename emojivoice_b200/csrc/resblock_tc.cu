// Fused HiFi-GAN ResBlock1 (hifigan/models.py:59-97) on tcgen05: all six convolutions of one block
//     for l in 0..2:  x = x + conv2_l( lrelu( conv1_l( lrelu(x) ; dilation d_l ) ) )
// run inside one kernel per time tile.  Only x (fp32, once) is read from and y (once) written to HBM -- the
// layer-by-layer path moves 16 B per element per conv pair, i.e. ~6x more, and is HBM-bound for C <= 128.
//
// Per CTA (persistent, one per SM) and per window of W = MB*128 time steps (halo H = 6(k-1) recomputed per tile):
//   * the fp32 RESIDUAL STREAM lives in TMEM (acc_x, MB x C columns) for the whole block: it is loaded once with
//     tcgen05.st and every conv2 simply accumulates onto it (accumulate = 1), so the residual add costs nothing;
//     conv2 biases are tracked as a per-channel offset that is added whenever acc_x is read.
//   * conv1 accumulates into a second TMEM region (acc_mid).
//   * ONE shared-memory operand buffer (bf16, K-major, hardware swizzle layout written by hand) holds lrelu(x) for
//     conv1, is overwritten by lrelu(conv1 + b) for conv2, then by lrelu(x_new) for the next pair.  Taps are row
//     offsets into it; zero margins / rows outside [0, L) implement each conv's own zero padding.
//   * weight tiles [C x C] per (conv, tap, K-chunk) stream from L2 through a TMA ring.
// CL = 2: two CTAs of a thread-block cluster share one window of 2 W rows: each owns W rows and, after every operand
// phase, pushes its 32 edge rows into the neighbour's margin through distributed shared memory (st.shared::cluster +
// a remote mbarrier arrive), so the halo is recomputed per PAIR of windows: at C = 128, k = 11 a window yields
// (512 - 120) / 2 = 196 output rows per CTA instead of 136.  (Clusters of 2 pack all 148 SMs; clusters of 4 strand 16.)
// Warps: 0 = TMA producer (weights), 1-2 = MMA issuers (half of the m-blocks each; warp 1 owns the TMEM allocation),
// 3.. = 16 (or 8) "epilogue" warps that load x, convert
// accumulators into the next operand, and write y.  Phases alternate strictly MMA -> epilogue (two mbarriers); the
// epilogue phases are short next to the MMA phases (<= 30 % even at k = 3).
#include <cuda.h>
#include <cudaTypedefs.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <mutex>

#include "conv.cuh"
#include "tc_ptx.cuh"

namespace ev {
using namespace tc;
namespace {

constexpr int RB_MAX_EPI_WARPS = 16;          // 16 epilogue warps (576 threads), or 8 when shared memory is needed for resident weights
constexpr int RB_MARG = 32;            // zero rows on both sides of the operand buffer (>= largest tap reach, 25)
constexpr int RB_STAGE_LD = 36;
constexpr int RB_MAX_SLOTS = 16;

struct RbMaps { CUtensorMap m[6]; };   // weights of conv1_0, conv2_0, conv1_1, conv2_1, conv1_2, conv2_2

struct RbParams {
  const float* x; long long x_bs;      // (b, t, c) fp32, dense rows of C
  float* sum; long long sum_bs;        // fp32 (b, t, c): MRF accumulator / output
  bf16* act_out; long long act_bs;     // optional bf16 (b, t, c): lrelu of the MRF mean (next stage's operand)
  const float* bias1[3];               // conv1_l bias [C]
  const float* bacc[3];                // sum_{i<=l} conv2_i bias [C]
  const float* bias2[3];               // conv2_l bias [C] (bias-by-MMA path)
  int L, k, dil[3];
  int mode;                            // 0: sum = y   1: sum += y   2: v = (sum + y) * inv_n -> sum (if write_f32) / act_out
  float inv_n, slope_out;
  int write_f32;
  int tiles_per_item, total_tiles, Wv, H;
  int w_slots;
  int resident;                        // all 6*k weight tiles stay in shared memory (C = 32): no per-tap barrier traffic
  int debug;                           // EV_RB_DEBUG (timing experiments, wrong results): 1 = no waits on the neighbour, 2 = no edge pushes
  const int* rag;                      // ragged batch: compact (item, window) list (RaggedPlanner, conv.cuh) or nullptr = dense
};

template <int C> struct RbCfg {
  static constexpr int MB = C == 128 ? 2 : 4;
  static constexpr int W = MB * 128;
  static constexpr int KC = C == 128 ? 2 : 1;            // K-chunks = planes of the operand buffer
  static constexpr int RB = C == 32 ? 64 : 128;          // bytes per operand row per plane (= swizzle width)
  static constexpr int KS = RB / 32;                     // UMMA K-steps (16 bf16) per chunk
  static constexpr int A_ROWS = W + 2 * RB_MARG;
  static constexpr int A_PLANE = A_ROWS * RB;
  static constexpr int W_TILE = C * RB;                  // one weight tile: C output rows x RB bytes
  static constexpr int NCB = C / 32;                     // 32-column blocks per accumulator
  static constexpr uint32_t TMEM_COLS = 2 * MB * C <= 256 ? 256 : 512;
  static constexpr uint32_t LAYOUT = RB == 128 ? 2u : 4u;
  static constexpr int STAGE_WARP = 32 * RB_STAGE_LD * 4;
  // Biases by MMA (C <= 64, where the kernel is bound by the epilogue warps' instruction issue): every conv gets one
  // extra K = 16 MMA per m-block, A = a constant tile whose rows are [1, 1, 0, ...], B = [bias_hi, bias_lo, 0, ...] per
  // output channel (bf16 hi + lo split: the bias stays accurate to 2^-17), both in the un-swizzled K-major core-matrix
  // layout (8 rows x 16 B core matrices, LBO = 128 B between the two K halves, SBO = 256 B between 8-row groups).  That
  // removes 32 FADDs and 8 bias loads per thread and block from every epilogue phase and keeps the residual stream in
  // TMEM bias-complete.
  static constexpr bool BIAS_MMA = C <= 64;
  static constexpr int ONES_BYTES = BIAS_MMA ? 128 * 32 : 0;
  static constexpr int BIAS_TILE = BIAS_MMA ? C * 32 : 0;
  static constexpr int EXTRA = ONES_BYTES + 6 * BIAS_TILE;
};

__device__ __forceinline__ uint32_t rb_cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t rb_map_to_cta(uint32_t local_saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_saddr), "r"(rank));
  return r;
}
// 16 bytes into the shared memory of a peer CTA; completes 16 bytes of transaction count on THAT CTA's mbarrier once the data
// has landed (no fence, no release/acquire at cluster scope: those compile to MEMBAR.ALL.GPU / CCTL.IVALL, ~1.5 us per phase)
__device__ __forceinline__ void rb_st_async16(uint32_t raddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t rbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];"
               ::"r"(raddr), "r"(a), "r"(b), "r"(c), "r"(d), "r"(rbar) : "memory");
}
// tcgen05.commit that arrives on the barrier at the same offset in every CTA of `mask` (the peers learn that this CTA's MMAs --
// the readers of its margins -- are complete, without a hop through a thread of this CTA)
__device__ __forceinline__ void rb_commit_multicast(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ void rb_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// OCC = CTAs per SM: 2 (C = 32 only: 8 epilogue warps, 256 TMEM columns and <= 112 KB of shared memory per CTA) lets one
// CTA's epilogue phases run under the other's MMA phases -- the phases of one window are short (k*8 MMAs of 40 clk
// against ~1.5k clk of accumulator -> operand conversion) and strictly alternate, so a lone CTA leaves the tensor pipe
// idle more than half of the time.
//
// WAVE = m-block wavefront (resident weights only): instead of "all MMAs of a conv, then all of its epilogue", the issuer
// walks the m-blocks of the window one after the other and commits each on its own mbarrier; the epilogue warps of m-block
// j convert its accumulator as soon as the MMAs of m-block j+1 have completed (they still read j's last rows through
// their taps), and the next conv's MMAs on m-block j start once the operand rows of j-1, j, j+1 are in place.  The
// tensor pipe then only idles when one m-block's epilogue (~400 clk) outlasts the next m-block's MMAs (k*KS*40-48 clk).
//
// CL = CTAs per cluster (1 or 2; not combined with WAVE): see the header comment.  Protocol per operand phase: a CTA's edge warps
// wait until the neighbour has finished the MMAs that read its margins (`nbr_done`: the neighbour's issuers commit on it by
// multicast next to their own `mma_done`), then write their 32 edge rows locally and -- st.async, 16 bytes each completing 16
// bytes of the neighbour's `marg_full` -- into the neighbour's margin; the MMA issuers wait for `epi_done` (own rows) and
// `marg_full` (margin rows) before the next conv.  No cluster-scope fences or barriers inside the loop.
template <int C, int OCC, bool WAVE, int CL>
__global__ void __launch_bounds__(OCC == 2 ? 96 + 32 * 8 : 96 + 32 * RB_MAX_EPI_WARPS, OCC)
resblock_tc_kernel(const __grid_constant__ RbMaps maps, const __grid_constant__ RbParams p) {
  using G = RbCfg<C>;
  constexpr int MB = G::MB, W = G::W, KC = G::KC, RB = G::RB, KS = G::KS, NCB = G::NCB;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t w_full[RB_MAX_SLOTS], w_empty[RB_MAX_SLOTS], mma_done, epi_done;
  __shared__ __align__(8) uint64_t mma_done_mb[4], epi_done_mb[4];   // WAVE: one pair per m-block
  __shared__ __align__(8) uint64_t nbr_done, marg_full;              // CL > 1: written by the neighbour CTA(s) of the cluster
  static_assert(!(WAVE && CL > 1), "the wavefront schedule is not combined with clusters");
  const uint32_t crank = CL > 1 ? rb_cluster_rank() : 0u;
  const int n_nbr = CL > 1 ? (crank > 0 ? 1 : 0) + (crank + 1 < (uint32_t)CL ? 1 : 0) : 0;
  const uint16_t nbr_mask = CL > 1 ? (uint16_t)((crank > 0 ? 1u << (crank - 1) : 0u) | (crank + 1 < (uint32_t)CL ? 1u << (crank + 1) : 0u)) : (uint16_t)0;
  static_assert(CL <= 2, "one neighbour per CTA");
  // Every CTA walks the taps of a conv upwards, like the single-window kernel: the per-row accumulation order -- and with it every
  // output bit -- does not depend on the pairing.  Rank 0 (neighbour to the right) meets the taps that reach into the neighbour's
  // rows in the second half of a conv and waits for the margin there; rank 1 needs its left margin from the first tap on.
  // (Walking the taps downwards on rank 1 to hide that wait as well was measured: no gain, and the bits then depend on the rank.)
  constexpr bool tap_desc = false;
  const int margin_tap = (CL > 1 && crank == 0) ? (p.k - 1) / 2 + 1 : 0;     // first tap index that reads the neighbour's rows
  const int cid = CL > 1 ? (int)blockIdx.x / CL : (int)blockIdx.x, n_cl = CL > 1 ? (int)gridDim.x / CL : (int)gridDim.x;
  __shared__ uint32_t tmem_base_smem;
#ifdef EV_RB_TRACE
  __shared__ long long rb_tr[32];          // EV_RB_DEBUG & 64: clock stamps of CTA 0's second window (printed at the end of the launch)     // nvcc -DEV_RB_TRACE + EV_RB_DEBUG=64: the device printf below costs registers, so it is not in normal builds
#define RB_TR(i) do { if ((p.debug & 64) && blockIdx.x == 0 && lane == 0 && tr_it == 1) rb_tr[(i)] = clock64(); } while (0)
#else
#define RB_TR(i) do { (void)tr_it; } while (0)
#endif

  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base_gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t a_s = base, w_s = base + KC * G::A_PLANE;
  uint8_t* a_gen = base_gen;
  const int n_epi = (int)(blockDim.x >> 5) - 3, n_slots = n_epi >> 2;   // epilogue warps; warps per TMEM lane quadrant
  const int w_tiles = p.resident ? 6 * p.k : p.w_slots;
  float* stage = reinterpret_cast<float*>(base_gen + KC * G::A_PLANE + w_tiles * G::W_TILE);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t extra_off = (uint32_t)(KC * G::A_PLANE + w_tiles * G::W_TILE + n_epi * G::STAGE_WARP);
  const uint32_t ones_s = base + extra_off, bias_s = ones_s + (uint32_t)G::ONES_BYTES;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 6; ++i) asm volatile("prefetch.tensormap [%0];" ::"l"(&maps.m[i]) : "memory");
    // two MMA issuer warps (m-blocks split between them): both commit on the weight-slot and phase barriers
    for (int s = 0; s < RB_MAX_SLOTS; ++s) { mbar_init(&w_full[s], 1); mbar_init(&w_empty[s], 2); }
    mbar_init(&mma_done, 2);
    mbar_init(&epi_done, (blockDim.x >> 5) - 3);
    for (int m = 0; m < 4; ++m) { mbar_init(&mma_done_mb[m], 1); mbar_init(&epi_done_mb[m], 4 * NCB); }   // one arrival per (lane quadrant, 32-column block)
    mbar_init(&nbr_done, CL > 1 && n_nbr ? 2 * n_nbr : 1); // one multicast commit per neighbour, issuer warp and conv
    mbar_init(&marg_full, 1);                              // expect_tx by issuer warp 1; the neighbours' st.async complete the bytes
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "r"(G::TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // zero the operand buffer once: its margins are never written again
  for (int i = threadIdx.x; i < KC * G::A_PLANE / 16; i += blockDim.x) reinterpret_cast<uint4*>(a_gen)[i] = make_uint4(0, 0, 0, 0);
  if constexpr (G::BIAS_MMA) {
    uint8_t* ex = base_gen + extra_off;
    for (int i = threadIdx.x; i < G::EXTRA / 16; i += blockDim.x) reinterpret_cast<uint4*>(ex)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    for (int r = threadIdx.x; r < 128; r += blockDim.x)       // A: every row [1, 1, 0, ...]
      *reinterpret_cast<uint32_t*>(ex + (r >> 3) * 256 + (r & 7) * 16) = 0x3F803F80u;
    for (int i = threadIdx.x; i < 6 * C; i += blockDim.x) {    // B: row n of conv ci = [bias_hi, bias_lo, 0, ...] (weights: safe before pdl_wait)
      const int ci = i / C, n = i - ci * C;
      const float bv = __ldg(((ci & 1) ? p.bias2[ci >> 1] : p.bias1[ci >> 1]) + n);
      const __nv_bfloat16 bh = __float2bfloat16_rn(bv);
      const __nv_bfloat16 bl = __float2bfloat16_rn(bv - __bfloat162float(bh));
      const uint32_t pk = (uint32_t)__bfloat16_as_ushort(bh) | ((uint32_t)__bfloat16_as_ushort(bl) << 16);
      *reinterpret_cast<uint32_t*>(ex + G::ONES_BYTES + ci * G::BIAS_TILE + (n >> 3) * 256 + (n & 7) * 16) = pk;
    }
  }
  fence_proxy_async();
  tcgen05_fence_before();
  if constexpr (CL > 1) rb_cluster_sync();     // the peer's barriers exist and its margins are zeroed before anything is pushed at them
  else __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_base_smem;
  pdl_trigger();
  pdl_wait();        // prologue (barriers, TMEM, zeroed operand buffer) overlapped the previous kernel's tail
  const int total_tiles = p.rag ? __ldg(p.rag) : p.total_tiles;   // ragged batch: only windows that hold needed rows
  const uint32_t acc_x = tmem_base, acc_mid = tmem_base + (uint32_t)(MB * C);
  const int k = p.k, half_k = (p.k - 1) / 2;

  if (warp == 0) {
    if (lane == 0) {
      // ---------------- TMA producer: weight tiles in the exact order the MMA warp consumes them
      int sl = 0;
      uint32_t ph = 1;
      if (p.resident) {     // every (conv, tap) tile once, kept for the CTA's lifetime
        mbar_expect_tx(&w_full[0], (uint32_t)(6 * k * G::W_TILE));
        for (int ci = 0; ci < 6; ++ci)
          for (int j = 0; j < k; ++j)
            tma_load_3d(w_s + (uint32_t)((ci * k + j) * G::W_TILE), &maps.m[ci], &w_full[0], 0, 0, j);
      }
      for (int tile = cid; tile < total_tiles && !p.resident; tile += n_cl) {
        for (int ci = 0; ci < 6; ++ci)
          for (int jj = 0; jj < k; ++jj)
            for (int kc = 0; kc < KC; ++kc) {
              const int j = tap_desc ? k - 1 - jj : jj;
              mbar_wait(&w_empty[sl], ph);
              mbar_expect_tx(&w_full[sl], (uint32_t)G::W_TILE);
              tma_load_3d(w_s + (uint32_t)(sl * G::W_TILE), &maps.m[ci], &w_full[sl], kc * (RB / 2), 0, j);
              if (++sl == p.w_slots) { sl = 0; ph ^= 1u; }
            }
      }
    }
    __syncwarp();
  } else if (WAVE && warp < 3) {
    // ---------------- wavefront issuer: warp 1 alone (one thread with straight-line code saturates the pipe at N <= 64)
    if (warp == 1) {
      constexpr uint32_t idesc = make_idesc(128, C);
      const uint32_t hi = ((uint32_t)(8 * RB) >> 4) | (1u << 14) | (G::LAYOUT << 29);
      const uint32_t a_lo0 = ((a_s & 0x3FFFFu) >> 4) | (1u << 16), w_lo0 = ((w_s & 0x3FFFFu) >> 4) | (1u << 16);
      const uint32_t hi_ns = (256u >> 4) | (1u << 14);
      const uint64_t d_ones = ((uint64_t)hi_ns << 32) | (((ones_s & 0x3FFFFu) >> 4) | (8u << 16));
      const uint32_t bias_lo0 = ((bias_s & 0x3FFFFu) >> 4) | (8u << 16);
      mbar_wait(&w_full[0], 0);
      tcgen05_fence_after();
      uint32_t cn = 0;                      // convs issued so far: epi_done_mb[*] completion number to wait for
      for (int tile = cid; tile < total_tiles; tile += n_cl) {
#pragma unroll 1
        for (int ci = 0; ci < 6; ++ci, ++cn) {
          const int l = ci >> 1, second = ci & 1;
          const int d = second ? 1 : p.dil[l];
          const uint32_t d_base = second ? acc_x : acc_mid;
          const uint32_t par = cn & 1u;
          const uint64_t d_bias = ((uint64_t)hi_ns << 32) | (bias_lo0 + (uint32_t)((ci * G::BIAS_TILE) >> 4));
          const uint32_t a_step = (uint32_t)((d * RB) >> 4), b_step = (uint32_t)(G::W_TILE >> 4);
          const uint32_t b_first = w_lo0 + (uint32_t)((ci * k * G::W_TILE) >> 4);
          const uint32_t a_first = a_lo0 + (uint32_t)(((RB_MARG - half_k * d) * RB) >> 4);
#pragma unroll 1
          for (int mb = 0; mb < MB; ++mb) {
            // operand rows of m-blocks mb-1, mb, mb+1 must hold this conv's input
            if (mb == 0) { mbar_wait(&epi_done_mb[0], par); if (MB > 1) mbar_wait(&epi_done_mb[1], par); }
            else if (mb + 1 < MB) mbar_wait(&epi_done_mb[mb + 1], par);
            tcgen05_fence_after();
            if (elect_one()) {
              const uint32_t dt = d_base + (uint32_t)(mb * C);
              umma_bf16(dt, d_ones, d_bias, idesc, second ? 1u : 0u);      // bias row: initialises conv1's accumulator
              uint32_t a_lo = a_first + (uint32_t)((mb * 128 * RB) >> 4), b_lo = b_first;
              for (int j = 0; j < k; ++j) {
#pragma unroll
                for (int ks = 0; ks < KS; ++ks)
                  umma_bf16(dt, ((uint64_t)hi << 32) | (a_lo + 2u * ks), ((uint64_t)hi << 32) | (b_lo + 2u * ks), idesc, 1u);
                a_lo += a_step;
                b_lo += b_step;
              }
              umma_commit(&mma_done_mb[mb]);
            }
            __syncwarp();
          }
        }
      }
    }
  } else if (warp < 3) {
    // ---------------- two MMA issuers (warp-uniform control flow, one elected lane each): warp 1 issues the first
    // half of the m-blocks, warp 2 the second half, so one warp's barrier / bookkeeping work overlaps the other's MMAs
    constexpr int MBH = MB / 2;
    const int mb0 = (warp - 1) * MBH;
    constexpr uint32_t idesc = make_idesc(128, C);
    const uint32_t hi = ((uint32_t)(8 * RB) >> 4) | (1u << 14) | (G::LAYOUT << 29);
    const uint32_t a_lo0 = ((a_s & 0x3FFFFu) >> 4) | (1u << 16), w_lo0 = ((w_s & 0x3FFFFu) >> 4) | (1u << 16);
    int sl = 0;
    uint32_t wph = 0, eph = 0;
    const bool resident = p.resident != 0;
    // un-swizzled K-major descriptors of the constant-ones tile and the bias tiles (SBO = 256 B, LBO = 128 B)
    const uint32_t hi_ns = (256u >> 4) | (1u << 14);
    const uint64_t d_ones = ((uint64_t)hi_ns << 32) | (((ones_s & 0x3FFFFu) >> 4) | (8u << 16));
    const uint32_t bias_lo0 = ((bias_s & 0x3FFFFu) >> 4) | (8u << 16);
    if (resident) { mbar_wait(&w_full[0], 0); tcgen05_fence_after(); }
    // CL = 2: the warp that owns the m-block next to the neighbour (rank 0: the last one, warp 2; rank 1: the first one, warp 1)
    // waits for the neighbour's 32 edge rows right before the first tap that reads them
    const bool margin_warp = CL > 1 && n_nbr && warp == (crank == 0 ? 2 : 1);
    uint32_t gph = 0;
    auto margin_wait = [&]() {
      if (p.debug & 3) return;
      if (elect_one()) mbar_expect_tx(&marg_full, (uint32_t)(32 * C * 2));
      __syncwarp();
      mbar_wait(&marg_full, gph);
      gph ^= 1u;
      fence_proxy_async();
      tcgen05_fence_after();
    };
    int tr_it = 0;
    for (int tile = cid; tile < total_tiles; tile += n_cl, ++tr_it) {
      for (int ci = 0; ci < 6; ++ci) {
        const int l = ci >> 1, second = ci & 1;
        const int d = second ? 1 : p.dil[l];
        const uint32_t d_tmem = second ? acc_x : acc_mid;
        mbar_wait(&epi_done, eph);          // the operand buffer holds this conv's input
        if (warp == 1) RB_TR(16 + 2 * ci);
        eph ^= 1u;
        tcgen05_fence_after();
        uint32_t fresh = second ? 0u : 1u;  // conv2 accumulates onto the residual stream from its first MMA on
        if (resident) {                     // KC == 1: one straight run of MMAs per conv, no barrier traffic
          if constexpr (G::BIAS_MMA) {
            if (elect_one()) {
              const uint64_t d_bias = ((uint64_t)hi_ns << 32) | (bias_lo0 + (uint32_t)((ci * G::BIAS_TILE) >> 4));
#pragma unroll
              for (int m = 0; m < MBH; ++m) umma_bf16(d_tmem + (uint32_t)((mb0 + m) * C), d_ones, d_bias, idesc, fresh ? 0u : 1u);
            }
            __syncwarp();
            fresh = 0;
          }
          const uint32_t b_base = w_lo0 + (uint32_t)((ci * k * G::W_TILE) >> 4);
          for (int jj = 0; jj < k; ++jj) {
            const int j = tap_desc ? k - 1 - jj : jj;
            if constexpr (CL > 1) { if (margin_warp && jj == margin_tap) margin_wait(); }
            if (elect_one()) {
              const uint32_t a_lo = a_lo0 + (uint32_t)(((RB_MARG + (j - half_k) * d) * RB) >> 4);
              const uint32_t b_lo = b_base + (uint32_t)((j * G::W_TILE) >> 4);
#pragma unroll
              for (int m = 0; m < MBH; ++m) {
                const int mb = mb0 + m;
#pragma unroll
                for (int ks = 0; ks < KS; ++ks) {
                  const uint64_t da = ((uint64_t)hi << 32) | (a_lo + (uint32_t)((mb * 128 * RB) >> 4) + 2u * ks);
                  const uint64_t db = ((uint64_t)hi << 32) | (b_lo + 2u * ks);
                  umma_bf16(d_tmem + (uint32_t)(mb * C), da, db, idesc, (fresh && ks == 0) ? 0u : 1u);
                }
              }
            }
            __syncwarp();
            fresh = 0;
          }
          if (elect_one()) {
            umma_commit(&mma_done);
            if constexpr (CL > 1) { if (n_nbr && !(p.debug & 4)) rb_commit_multicast(&nbr_done, nbr_mask); }
          }
          __syncwarp();
          continue;
        }
        if constexpr (G::BIAS_MMA) {
          if (elect_one()) {
            const uint64_t d_bias = ((uint64_t)hi_ns << 32) | (bias_lo0 + (uint32_t)((ci * G::BIAS_TILE) >> 4));
#pragma unroll
            for (int m = 0; m < MBH; ++m) umma_bf16(d_tmem + (uint32_t)((mb0 + m) * C), d_ones, d_bias, idesc, fresh ? 0u : 1u);
          }
          __syncwarp();
          fresh = 0;
        }
        for (int jj = 0; jj < k; ++jj) {
          const int j = tap_desc ? k - 1 - jj : jj;
          if constexpr (CL > 1) { if (margin_warp && jj == margin_tap) margin_wait(); }
          for (int kc = 0; kc < KC; ++kc) {
            mbar_wait(&w_full[sl], wph);
            tcgen05_fence_after();
            const uint32_t b_lo = w_lo0 + (uint32_t)((sl * G::W_TILE) >> 4);
            const uint32_t a_lo = a_lo0 + (uint32_t)((kc * G::A_PLANE + (RB_MARG + (j - half_k) * d) * RB) >> 4);
            if (elect_one()) {
#pragma unroll
              for (int m = 0; m < MBH; ++m) {
                const int mb = mb0 + m;
#pragma unroll
                for (int ks = 0; ks < KS; ++ks) {
                  const uint64_t da = ((uint64_t)hi << 32) | (a_lo + (uint32_t)((mb * 128 * RB) >> 4) + 2u * ks);
                  const uint64_t db = ((uint64_t)hi << 32) | (b_lo + 2u * ks);
                  umma_bf16(d_tmem + (uint32_t)(mb * C), da, db, idesc, (fresh && ks == 0) ? 0u : 1u);
                }
              }
              umma_commit(&w_empty[sl]);
            }
            __syncwarp();
            fresh = 0;
            if (++sl == p.w_slots) { sl = 0; wph ^= 1u; }
          }
        }
        if (elect_one()) {
          umma_commit(&mma_done);
          if constexpr (CL > 1) { if (n_nbr && !(p.debug & 4)) rb_commit_multicast(&nbr_done, nbr_mask); }
        }
        __syncwarp();
        if (warp == 1) RB_TR(17 + 2 * ci);
      }
    }
  } else {
    // ---------------- 16 epilogue warps.  Warp (q, slot): TMEM lanes [32q, 32q+32), blocks slot, slot+4, ... of the
    // MB*NCB (m-block, 32-column block) pairs of that lane quadrant.
    const int ew = warp - 3, q = warp & 3, slot = ew >> 2;   // n_slots warps share a lane quadrant
    const int sub = lane >> 3, cl = (lane & 7) * 4;
    float* wstage = stage + ew * (32 * RB_STAGE_LD);
    const uint32_t lane_addr = ((uint32_t)(q * 32) << 16);
    const int L = p.L, H = p.H;
    uint32_t mph = 0;
    // CL > 1: which of this warp's blocks are edge rows of the CTA's window (first / last 32 rows) with a neighbour behind them
    bool edge_l = false, edge_r = false;
    if constexpr (CL > 1) {
      for (int blk = slot; blk < MB * NCB; blk += n_slots) {
        const int mb = blk / NCB;
        if (crank > 0 && q == 0 && mb == 0) edge_l = true;
        if (crank + 1 < (uint32_t)CL && q == 3 && mb == MB - 1) edge_r = true;
      }
    }
    const int n_blk = max(0, (MB * NCB - slot + n_slots - 1) / n_slots);   // this warp's (m-block, 32-column block) pairs
    // edge blocks LAST: the neighbour's "my MMAs are done" arrival (one DSMEM hop behind our own mma_done) is then awaited behind
    // this warp's other block instead of in front of the whole phase
    const bool rev = CL > 1 && edge_l;
    uint32_t sig = 0;                    // CL > 1: convs whose MMAs this CTA has reported to its neighbours
    const uint32_t marg_full_s = smem_u32(&marg_full);
    auto conv_done_signal = [&]() { if constexpr (CL > 1) ++sig; };   // (the issuers' multicast commits tell the neighbours)
    // before an operand phase pushes edge rows: every neighbour has finished the MMAs of all `sig` convs so far
    auto nbr_wait = [&]() {
      if constexpr (CL > 1) {
        if ((edge_l || edge_r) && sig && !(p.debug & 1)) mbar_wait(&nbr_done, (sig - 1u) & 1u);
      }
    };

    // write 32 activated channels of one row into the operand buffer (bf16, swizzled K-major layout)
    auto put_operand = [&](int wr, int cb, const float (&v)[32]) {
      const int row = RB_MARG + wr;
      const int plane = (cb * 32) / (RB / 2), c16 = ((cb * 32) % (RB / 2)) / 8;     // 16-byte chunk index inside the row
      uint8_t* rp = a_gen + plane * G::A_PLANE + row * RB;
      const int sw = RB == 128 ? (row & 7) : ((row >> 1) & 3);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        uint32_t w4[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          __nv_bfloat162 h2 = __floats2bfloat162_rn(v[8 * i + 2 * e], v[8 * i + 2 * e + 1]);
          w4[e] = *reinterpret_cast<uint32_t*>(&h2);
        }
        *reinterpret_cast<uint4*>(rp + (((c16 + i) ^ sw) << 4)) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
      }
    };
    // CL > 1: the same 32 channels of an edge row into the neighbour's margin (dir = -1: our first 32 rows -> the right margin
    // of the left neighbour, dir = +1: our last 32 rows -> the left margin of the right neighbour); every 16 bytes complete
    // 16 bytes of the neighbour's `marg_full` transaction count
    auto put_remote = [&](int wr, int cb, const float (&v)[32], int dir) {
      const int row = RB_MARG + wr - dir * W;
      const int plane = (cb * 32) / (RB / 2), c16 = ((cb * 32) % (RB / 2)) / 8;
      const int sw = RB == 128 ? (row & 7) : ((row >> 1) & 3);
      const uint32_t ra = rb_map_to_cta(a_s + (uint32_t)(plane * G::A_PLANE + row * RB), crank + (uint32_t)dir);
      const uint32_t rbar = rb_map_to_cta(marg_full_s, crank + (uint32_t)dir);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        uint32_t w4[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          __nv_bfloat162 h2 = __floats2bfloat162_rn(v[8 * i + 2 * e], v[8 * i + 2 * e + 1]);
          w4[e] = *reinterpret_cast<uint32_t*>(&h2);
        }
        rb_st_async16(ra + (uint32_t)(((c16 + i) ^ sw) << 4), w4[0], w4[1], w4[2], w4[3], rbar);
      }
    };
    auto put_edges = [&](int mb, int wr, int cb, const float (&v)[32]) {
      if constexpr (CL > 1) {
        if (p.debug & 2) return;
        if (edge_l && mb == 0) { nbr_wait(); put_remote(wr, cb, v, -1); }
        if (edge_r && mb == MB - 1) { nbr_wait(); put_remote(wr, cb, v, +1); }
      }
    };
    // MRF accumulator read-back (mode >= 1): the 32 x 32 block of `sum` that belongs to output block `blk` is copied global -> the
    // warp's transpose buffer with cp.async (no registers, no stall), row-major like the accumulator rows the threads will hold.
    // Issued for the warp's first block BEFORE the wait for the last conv's MMAs, so that DRAM latency hides behind them; the
    // row pass then adds it from shared memory.  (Read inside the row pass, every load sat behind the previous row's store to the
    // same array: eight DRAM latencies per block, traced as 14-25 k clk of a 60-120 k clk window.)
    auto stage_sum = [&](int b_, int w0_, int blk) {
      const int mb = blk / NCB, cb = blk - mb * NCB;
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int wr2 = mb * 128 + q * 32 + u * 4 + sub, t2 = w0_ + wr2, g2 = (int)crank * W + wr2;
        if (g2 < H || g2 >= CL * W - H || t2 < 0 || t2 >= L) continue;     // rows that are not stored: whatever the buffer holds
        const float* src = p.sum + b_ * p.sum_bs + (long long)t2 * C + cb * 32 + cl;
        const uint32_t dst = smem_u32(wstage + (u * 4 + sub) * RB_STAGE_LD + cl);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto phase_done = [&]() {
      if constexpr (WAVE) return;        // wavefront mode hands over block by block (block_done)
      tcgen05_fence_before();
      fence_proxy_async();               // operand buffer writes -> visible to the tensor core (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(&epi_done);
    };
    uint32_t cn = 0;                     // WAVE: convs consumed so far = mma_done_mb[*] completion number to wait for
    auto wave_wait = [&](int mb) {       // m-block mb may be converted once mb+1's MMAs (which read mb's last rows) are done
      if constexpr (WAVE) {
        mbar_wait(&mma_done_mb[mb + 1 < MB ? mb + 1 : MB - 1], cn & 1u);
        tcgen05_fence_after();
      }
    };
    auto block_done = [&](int mb) {
      if constexpr (WAVE) {
        tcgen05_fence_before();
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&epi_done_mb[mb]);
      }
    };

    // L2 prefetch of the NEXT window's rows of x (and of the MRF accumulator when it is read back): a lone CTA per SM otherwise sits
    // through two rounds of DRAM latency in phase 0 and again in the output phase of every window
    const int pf_tid = ew * 32 + lane, pf_n = n_epi * 32;
    auto prefetch_window = [&](int tile_n) {
      if (tile_n >= total_tiles || (p.debug & 32)) return;
      int bn, tn;
      if (p.rag) { const int pair = __ldg(p.rag + 1 + tile_n); bn = pair >> 16; tn = pair & 0xffff; }
      else { bn = tile_n / p.tiles_per_item; tn = tile_n - bn * p.tiles_per_item; }
      const int wn = tn * p.Wv - H + (int)crank * W;
      constexpr int LPR = C * 4 / 128 > 0 ? C * 4 / 128 : 1;          // 128-byte lines per row (C = 32: one line per row)
      const char* xn = reinterpret_cast<const char*>(p.x + bn * p.x_bs);
      const char* sn = reinterpret_cast<const char*>(p.sum + bn * p.sum_bs);
      for (int i = pf_tid; i < W * LPR; i += pf_n) {
        const int t = wn + i / LPR;
        if (t < 0 || t >= L) continue;
        const long long off = (long long)t * C * 4 + (i % LPR) * 128;
        asm volatile("prefetch.global.L2 [%0];" ::"l"(xn + off));
        if (p.mode >= 1) asm volatile("prefetch.global.L2 [%0];" ::"l"(sn + off));
      }
    };
    int tr_it = 0;
    for (int tile = cid; tile < total_tiles; tile += n_cl, ++tr_it) {
      int b, ti;
      if (p.rag) { const int pair = __ldg(p.rag + 1 + tile); b = pair >> 16; ti = pair & 0xffff; }
      else { b = tile / p.tiles_per_item; ti = tile - b * p.tiles_per_item; }
      if (ew == 0) RB_TR(0);
      const int w0 = ti * p.Wv - H + (int)crank * W;     // CL > 1: the cluster's window is CL * W rows, this CTA owns rows [crank * W, +W)
      const bool interior = w0 >= 0 && w0 + W <= L;    // no row of this window lies outside the sequence: no zero-padding fix-ups
      const float* xb = p.x + b * p.x_bs;
      // ---- phase 0: x -> acc_x (fp32, TMEM) and lrelu(x) -> operand buffer
#pragma unroll 1
      for (int bi = 0; bi < n_blk; ++bi) {
        const int blk = slot + (rev ? n_blk - 1 - bi : bi) * n_slots;
        const int mb = blk / NCB, cb = blk - mb * NCB;
#pragma unroll
        for (int u = 0; u < 8; ++u) {          // coalesced: 8 lanes x float4 per row, 4 rows per instruction
          const int wr = mb * 128 + q * 32 + u * 4 + sub, t = w0 + wr;
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (t >= 0 && t < L) v = *reinterpret_cast<const float4*>(xb + (long long)t * C + cb * 32 + cl);
          *reinterpret_cast<float4*>(wstage + (u * 4 + sub) * RB_STAGE_LD + cl) = v;
        }
        __syncwarp();
        uint32_t raw[32];
        float a[32];
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 v = *reinterpret_cast<const float4*>(wstage + lane * RB_STAGE_LD + j);
          raw[j] = __float_as_uint(v.x); raw[j + 1] = __float_as_uint(v.y); raw[j + 2] = __float_as_uint(v.z); raw[j + 3] = __float_as_uint(v.w);
          a[j] = fmaxf(v.x, 0.1f * v.x); a[j + 1] = fmaxf(v.y, 0.1f * v.y); a[j + 2] = fmaxf(v.z, 0.1f * v.z); a[j + 3] = fmaxf(v.w, 0.1f * v.w);
        }
        tmem_st32(acc_x + lane_addr + (uint32_t)(mb * C + cb * 32), raw);
        put_operand(mb * 128 + q * 32 + lane, cb, a);
        put_edges(mb, mb * 128 + q * 32 + lane, cb, a);
        __syncwarp();
        if constexpr (WAVE) { tmem_st_wait(); block_done(mb); }
      }
      tmem_st_wait();
      phase_done();
      if (ew == 0) RB_TR(1);
      // measured (ragged config-2 batch, vocoder total): no prefetch 13.58 ms, everywhere 13.49 ms (k3 at C = 128: 831 -> 761 us, C = 64:
      // 640 -> 580, C = 32: 497 -> 454); EV_RB_DEBUG=128 switches it off
      if (!(p.debug & 128)) prefetch_window(tile + n_cl);

#pragma unroll 1
      for (int l = 0; l < 3; ++l) {
        // ---- after conv1_l: operand <- lrelu(acc_mid + b1), zero outside the sequence (conv2's zero padding)
        if constexpr (!WAVE) {
          mbar_wait(&mma_done, mph);
          mph ^= 1u;
          tcgen05_fence_after();
          conv_done_signal();
          if (ew == 0) RB_TR(2 + 4 * l);
        }
#pragma unroll 1
        for (int bi = 0; bi < n_blk; ++bi) {
          const int blk = slot + (rev ? n_blk - 1 - bi : bi) * n_slots;
          const int mb = blk / NCB, cb = blk - mb * NCB;
          const int wr = mb * 128 + q * 32 + lane, t = w0 + wr;
          const float keep = (t >= 0 && t < L) ? 1.0f : 0.0f;
          wave_wait(mb);
          uint32_t raw[32];
          tmem_ld32(acc_mid + lane_addr + (uint32_t)(mb * C + cb * 32), raw);
          float a[32];
          if constexpr (G::BIAS_MMA) {
#pragma unroll
            for (int j = 0; j < 32; ++j) { const float v = __uint_as_float(raw[j]); a[j] = fmaxf(v, 0.1f * v); }
          } else {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias1[l] + cb * 32 + j));
              const float v0 = __uint_as_float(raw[j]) + bv.x, v1 = __uint_as_float(raw[j + 1]) + bv.y;
              const float v2 = __uint_as_float(raw[j + 2]) + bv.z, v3 = __uint_as_float(raw[j + 3]) + bv.w;
              a[j] = fmaxf(v0, 0.1f * v0); a[j + 1] = fmaxf(v1, 0.1f * v1);
              a[j + 2] = fmaxf(v2, 0.1f * v2); a[j + 3] = fmaxf(v3, 0.1f * v3);
            }
          }
          if (!interior) {
#pragma unroll
            for (int j = 0; j < 32; ++j) a[j] *= keep;
          }
          put_operand(wr, cb, a);
          put_edges(mb, wr, cb, a);
          block_done(mb);
        }
        ++cn;
        phase_done();
        if (ew == 0) RB_TR(3 + 4 * l);
        // ---- after conv2_l: acc_x now holds x_new - (accumulated conv2 biases)
        if (l == 2 && p.mode >= 1 && n_blk > 0) stage_sum(b, w0, slot + (rev ? n_blk - 1 : 0) * n_slots);
        if constexpr (!WAVE) {
          mbar_wait(&mma_done, mph);
          mph ^= 1u;
          tcgen05_fence_after();
          conv_done_signal();
          if (ew == 0) RB_TR(4 + 4 * l);
        }
#pragma unroll 1
        for (int bi = 0; bi < n_blk; ++bi) {
          const int blk = slot + (rev ? n_blk - 1 - bi : bi) * n_slots;
          const int mb = blk / NCB, cb = blk - mb * NCB;
          const int wr = mb * 128 + q * 32 + lane, t = w0 + wr;
          wave_wait(mb);
          uint32_t raw[32];
          tmem_ld32(acc_x + lane_addr + (uint32_t)(mb * C + cb * 32), raw);
          float a[32];
          if constexpr (G::BIAS_MMA) {
#pragma unroll
            for (int j = 0; j < 32; ++j) a[j] = __uint_as_float(raw[j]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bacc[l] + cb * 32 + j));
              a[j] = __uint_as_float(raw[j]) + bv.x; a[j + 1] = __uint_as_float(raw[j + 1]) + bv.y;
              a[j + 2] = __uint_as_float(raw[j + 2]) + bv.z; a[j + 3] = __uint_as_float(raw[j + 3]) + bv.w;
            }
          }
          if (l < 2) {
#pragma unroll
            for (int j = 0; j < 32; ++j) a[j] = fmaxf(a[j], 0.1f * a[j]);
            if (!interior) {
              const float keep = (t >= 0 && t < L) ? 1.0f : 0.0f;
#pragma unroll
              for (int j = 0; j < 32; ++j) a[j] *= keep;
            }
            put_operand(wr, cb, a);
            put_edges(mb, wr, cb, a);
            block_done(mb);
          } else {
            // ---- block output: (+ the staged MRF accumulator) -> transpose through the private buffer -> coalesced rows
            if (p.mode >= 1) {
              asm volatile("cp.async.wait_group 0;" ::: "memory");
              __syncwarp();                                            // every lane's copies have landed
#pragma unroll
              for (int j = 0; j < 32; j += 4) {
                const float4 s4 = *reinterpret_cast<const float4*>(wstage + lane * RB_STAGE_LD + j);
                a[j] += s4.x; a[j + 1] += s4.y; a[j + 2] += s4.z; a[j + 3] += s4.w;
              }
              __syncwarp();                                            // all rows read before the buffer is rewritten
            }
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              *reinterpret_cast<float4*>(wstage + lane * RB_STAGE_LD + j) = make_float4(a[j], a[j + 1], a[j + 2], a[j + 3]);
            __syncwarp();
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const int wr2 = mb * 128 + q * 32 + u * 4 + sub, t2 = w0 + wr2;
              const int g2 = (int)crank * W + wr2;                   // row inside the cluster's window: its outer H rows are halo
              if (g2 < H || g2 >= CL * W - H || t2 < 0 || t2 >= L) continue;
              float4 v = *reinterpret_cast<const float4*>(wstage + (u * 4 + sub) * RB_STAGE_LD + cl);
              const long long off = (long long)t2 * C + cb * 32 + cl;
              if (p.mode == 2) { v.x *= p.inv_n; v.y *= p.inv_n; v.z *= p.inv_n; v.w *= p.inv_n; }
              if (p.mode < 2 || p.write_f32) *reinterpret_cast<float4*>(p.sum + b * p.sum_bs + off) = v;
              if (p.mode == 2 && p.act_out) {
                const float s = p.slope_out;
                __nv_bfloat162 lo = __floats2bfloat162_rn(fmaxf(v.x, s * v.x), fmaxf(v.y, s * v.y));
                __nv_bfloat162 hi2 = __floats2bfloat162_rn(fmaxf(v.z, s * v.z), fmaxf(v.w, s * v.w));
                uint2 pk;
                pk.x = *reinterpret_cast<uint32_t*>(&lo);
                pk.y = *reinterpret_cast<uint32_t*>(&hi2);
                *reinterpret_cast<uint2*>(p.act_out + b * p.act_bs + off) = pk;
              }
            }
            __syncwarp();                                              // the row pass has read the buffer
            if (p.mode >= 1 && bi + 1 < n_blk) stage_sum(b, w0, slot + (rev ? n_blk - 2 - bi : bi + 1) * n_slots);
          }
        }
        ++cn;
        if (l < 2) phase_done();
        if (ew == 0) RB_TR(5 + 4 * l);
      }
      tcgen05_fence_before();   // acc_x is rewritten by the next tile's phase 0
    }
  }
  tcgen05_fence_before();
  if constexpr (CL > 1) rb_cluster_sync();     // no CTA exits while a peer may still push rows or arrivals at it
  else __syncthreads();
#ifdef EV_RB_TRACE
  if ((p.debug & 64) && blockIdx.x == 0 && threadIdx.x == 0) {
    const long long t0 = rb_tr[0];
    printf("RBTR C=%d k=%d cl=%d occ=%d | epi: ph0 %lld |", C, p.k, CL, OCC, rb_tr[1] - t0);
    for (int l = 0; l < 3; ++l) printf(" c1 mma_done %lld op %lld c2 mma_done %lld op %lld |", rb_tr[2 + 4 * l] - t0, rb_tr[3 + 4 * l] - t0, rb_tr[4 + 4 * l] - t0, rb_tr[5 + 4 * l] - t0);
    printf(" issuer (epi_done seen, issued):");
    for (int ci = 0; ci < 6; ++ci) printf(" %lld %lld", rb_tr[16 + 2 * ci] - t0, rb_tr[17 + 2 * ci] - t0);
    printf("\n");
  }
#endif
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(G::TMEM_COLS) : "memory");
  }
}

int g_rb_resident = 1;   // EV_RB_RESIDENT=0: stream weights through the ring even when they would fit

int g_rb_occ2 = 1;       // EV_RB_OCC2=0: one CTA per SM also at C = 32
int g_rb_cluster = 2;    // EV_RB_CLUSTER=1: single-CTA windows (every CTA recomputes its own halo)
int g_rb_wave = 0;       // EV_RB_WAVE=1: m-block wavefront schedule instead of phase alternation (measured equal: the kernel is
                         // bound by shared-memory bandwidth -- MMA operand fetch alone takes 32 + N/4 of every 40-48 clk)

// launch with programmatic stream serialization and (cl > 1) a thread-block cluster of `cl` CTAs along x
template <typename... KArgs, typename... Args>
cudaError_t launch_rb_kernel(void (*kernel)(KArgs...), int grid, int block, size_t smem, int cl, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  at[1].id = cudaLaunchAttributeClusterDimension;
  at[1].val.clusterDim.x = cl; at[1].val.clusterDim.y = 1; at[1].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = cl > 1 ? 2 : 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

template <int C>
cudaError_t launch_rb(const RbMaps& maps, RbParams& p, int B, cudaStream_t s, RaggedPlanner* ragged, const RbSchedule& sched,
                      RbLaunchInfo* info, std::string* err) {
  using G = RbCfg<C>;
  // the EV_RB_* switches, unless this call overrides them
  const int cluster = sched.cluster >= 0 ? sched.cluster : g_rb_cluster;
  const bool occ2_on = sched.occ2 >= 0 ? sched.occ2 != 0 : g_rb_occ2 != 0;
  const bool wave_on = sched.wave >= 0 ? sched.wave != 0 : g_rb_wave != 0;
  const bool resident_on = sched.resident >= 0 ? sched.resident != 0 : g_rb_resident != 0;
  // CTAs per cluster window: 2 halves the recomputed halo (the wavefront schedule keeps single CTAs)
  // Measured on B200 (profiles/r02_resblock_clusters.txt, us per ResBlock on the ragged config-2 batch, single / paired windows):
  //   C=128: k3 797/855  k7 1658/1546  k11 2849/2194     C=64: k3 633/662  k7 1189/1172  k11 1641/1509
  //   C=32 : k3 479/558  k7  975/1016  k11 1339/1291
  // Launching the SAME code as clusters of two costs 2-3 % by itself (CTA placement) and the paired kernel another ~5 %, so pairs pay
  // where the halo is a large part of a window: k >= 7 at C >= 64, k = 11 at C = 32.  EV_RB_CLUSTER=3 pairs everything, =1 nothing.
  const bool pair_pays = (p.k >= 7 && C >= 64) || p.k >= 11;
  const int cl = ((cluster >= 3 || (cluster == 2 && pair_pays)) && !wave_on) ? 2 : 1;
  { static const int dbg = []() { const char* v = getenv("EV_RB_DEBUG"); return v ? atoi(v) : 0; }(); p.debug = dbg; }
  p.H = 6 * (p.k - 1);                    // sum over the three pairs of (k-1)/2 * (d_l + 1), d = 1, 3, 5
  p.Wv = cl * G::W - 2 * p.H;             // output rows per (cluster) window
  p.tiles_per_item = ceil_div(p.L, p.Wv);
  p.total_tiles = p.tiles_per_item * B;
  // plan: CTAs per SM, all weights resident in shared memory or a ring of w_slots tiles, epilogue warps, shared memory per CTA
  int occ = 1, n_epi = 16, smem = 0;
  p.resident = 0;
  p.w_slots = 0;
  if constexpr (C == 32) {
    if (occ2_on) {
      const int per_cta = (228 * 1024) / 2 - 2048;
      const int fixed8 = 1024 + G::KC * G::A_PLANE + 8 * G::STAGE_WARP + G::EXTRA;
      const int res_bytes = 6 * p.k * G::W_TILE;
      if (resident_on && fixed8 + res_bytes <= per_cta) { p.resident = 1; p.w_slots = 1; smem = fixed8 + res_bytes; }
      else {
        p.resident = 0;
        p.w_slots = std::min((per_cta - fixed8) / G::W_TILE, RB_MAX_SLOTS);
        smem = fixed8 + p.w_slots * G::W_TILE;
      }
      if (p.w_slots >= 1 && (p.resident || p.w_slots >= 4)) { occ = 2; n_epi = 8; }
    }
  }
  const int limit = 224 * 1024;
  if (occ == 1) {
    const int fixed16 = 1024 + G::KC * G::A_PLANE + 16 * G::STAGE_WARP + G::EXTRA, fixed8 = 1024 + G::KC * G::A_PLANE + 8 * G::STAGE_WARP + G::EXTRA;
    const int res_bytes = 6 * p.k * G::W_TILE;
    p.resident = 0;
    if (G::KC == 1 && resident_on && fixed16 + res_bytes <= limit) { p.resident = 1; smem = fixed16 + res_bytes; }
    else if (G::KC == 1 && resident_on && fixed8 + res_bytes <= limit) { p.resident = 1; n_epi = 8; smem = fixed8 + res_bytes; }
    else {
      int slots = std::min((limit - fixed16) / G::W_TILE, RB_MAX_SLOTS);
      if (slots < 3) return cudaErrorInvalidConfiguration;
      p.w_slots = slots;
      smem = fixed16 + slots * G::W_TILE;
    }
    if (p.resident) p.w_slots = 1;
  }
  const bool wave = wave_on && p.resident && G::BIAS_MMA && G::KC == 1;   // the wavefront issuer needs every weight tile resident
  // a schedule the caller forces is launched as asked or not at all
  const char* refuse = nullptr;
  if (sched.wave == 1 && !wave) refuse = "the wavefront schedule needs resident weights (C = 32, one CTA per SM)";
  else if (sched.cluster >= 3 && cl != 2) refuse = "paired windows are not combined with the wavefront schedule";
  else if (sched.occ2 == 1 && occ != 2) refuse = "two CTAs per SM run at C = 32 only";
  else if (sched.resident == 1 && !p.resident) refuse = "the weights of this block do not fit in shared memory at this occupancy";
  if (refuse) {
    if (err) *err = std::string("resblock_tc: forced schedule cannot run: ") + refuse;
    return cudaErrorInvalidValue;
  }
  const int grid = cl * std::min(p.total_tiles, occ * tc_sm_count() / cl);
  if (info) {
    info->cl = cl; info->occ = occ; info->wave = wave ? 1 : 0; info->resident = p.resident; info->w_slots = p.w_slots;
    info->n_epi = n_epi; info->grid = grid; info->Wv = p.Wv; info->total_tiles = p.total_tiles;
  }
  p.rag = ragged ? ragged->table(p.Wv, p.L, s) : nullptr;
  if constexpr (C == 32) {
    if (occ == 2) {
      const int per_cta = (228 * 1024) / 2 - 2048;
      static DeviceOnce once2;
      cudaError_t ce2 = once2.run([&]() {
        cudaError_t ce = cudaFuncSetAttribute(resblock_tc_kernel<C, 2, false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, per_cta);
        if (ce == cudaSuccess) ce = cudaFuncSetAttribute(resblock_tc_kernel<C, 2, false, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, per_cta);
        if (ce == cudaSuccess) ce = cudaFuncSetAttribute(resblock_tc_kernel<C, 2, true, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, per_cta);
        return ce;
      });
      if (ce2 != cudaSuccess) return ce2;
      // at least a third of the SM's shared memory: a third CTA would not find TMEM columns (2 x 256 are taken)
      const size_t sm = (size_t)std::max(smem, 80 * 1024);
      if (wave) return launch_rb_kernel(resblock_tc_kernel<C, 2, true, 1>, grid, 96 + 32 * 8, sm, 1, s, maps, p);
      if (cl == 2) return launch_rb_kernel(resblock_tc_kernel<C, 2, false, 2>, grid, 96 + 32 * 8, sm, 2, s, maps, p);
      return launch_rb_kernel(resblock_tc_kernel<C, 2, false, 1>, grid, 96 + 32 * 8, sm, 1, s, maps, p);
    }
  }
  static DeviceOnce once;
  cudaError_t ce1 = once.run([&]() {
    cudaError_t ce = cudaFuncSetAttribute(resblock_tc_kernel<C, 1, false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, limit);
    if (ce == cudaSuccess) ce = cudaFuncSetAttribute(resblock_tc_kernel<C, 1, false, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, limit);
    if (ce == cudaSuccess && G::BIAS_MMA && G::KC == 1) ce = cudaFuncSetAttribute(resblock_tc_kernel<C, 1, G::BIAS_MMA && G::KC == 1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, limit);
    return ce;
  });
  if (ce1 != cudaSuccess) return ce1;
  if (p.debug & 8) {     // how many clusters the device holds at once
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(96 + 32 * n_epi); cfg.dynamicSmemBytes = (size_t)std::max(smem, 120 * 1024);
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cl; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int n = -1;
    cudaError_t ce = cl == 2 ? cudaOccupancyMaxActiveClusters(&n, resblock_tc_kernel<C, 1, false, 2>, &cfg) : cudaOccupancyMaxActiveClusters(&n, resblock_tc_kernel<C, 1, false, 1>, &cfg);
    fprintf(stderr, "resblock_tc C=%d k=%d cl=%d grid=%d tiles=%d smem=%d: max active clusters %d (%s)\n", C, p.k, cl, grid, p.total_tiles, smem, n, cudaGetErrorString(ce));
  }
  // shared memory above half an SM keeps a second CTA (and its TMEM allocation) off the SM
  const size_t sm = (size_t)std::max(smem, 120 * 1024);
  if (wave)
    return launch_rb_kernel(resblock_tc_kernel<C, 1, G::BIAS_MMA && G::KC == 1, 1>, grid, 96 + 32 * n_epi, sm, 1, s, maps, p);
  if (cl == 2) return launch_rb_kernel(resblock_tc_kernel<C, 1, false, 2>, grid, 96 + 32 * n_epi, sm, 2, s, maps, p);
  return launch_rb_kernel(resblock_tc_kernel<C, 1, false, 1>, (p.debug & 16) ? grid / 2 * 2 : grid, 96 + 32 * n_epi, sm, (p.debug & 16) ? 2 : 1, s, maps, p);
}

}  // namespace

int g_rb_policy = -1;    // EV_RB_FUSE: 0 = never, 1 = where measured faster (default), 2 = wherever the kernel can run

// EV_RB_* switches (read once)
static void rb_read_env() {
  static std::once_flag once;
  std::call_once(once, []() {
    const char* v = getenv("EV_RB_RESIDENT"); g_rb_resident = !(v && atoi(v) == 0);
    v = getenv("EV_RB_OCC2"); g_rb_occ2 = !(v && atoi(v) == 0);
    v = getenv("EV_RB_WAVE"); g_rb_wave = v && atoi(v) != 0;
    v = getenv("EV_RB_CLUSTER"); if (v) g_rb_cluster = atoi(v);
    v = getenv("EV_RB_FUSE"); g_rb_policy = v ? atoi(v) : 1;
  });
}

bool resblock_tc_supported(int C, int k, const int* dil) {
  rb_read_env();
  if (g_rb_policy == 0) return false;
  if (C != 32 && C != 64 && C != 128) return false;
  if (k != 3 && k != 7 && k != 11) return false;
  if (dil[0] != 1 || dil[1] != 3 || dil[2] != 5) return false;
  if (g_rb_policy >= 2) return true;
  // Measured on B200 (profiles/r01_resblocks_v17_biasmma_occ2.txt vs r01_layers_v15_two_issuers.txt, us per ResBlock at B=32 x 668
  // frames, fused / layer-by-layer):
  //   C=128: k3 1145/1686  k7 2408/2265  k11 4128/2844     C=64: k3  888/1764  k7 1668/2145  k11 2341/2682
  //   C=32 : k3  662/1644  k7 1356/1953  k11 1915/2649
  // The fused kernel wins wherever the layer-by-layer path is HBM/epilogue-bound (everything at C <= 64, k = 3 at C = 128); at
  // C = 128 with k >= 7 the separate convs are already MMA-bound (1.1-1.2 PFLOP/s) and the halo recompute (H = 6(k-1) rows
  // per window side, 256-row windows) costs more than the saved traffic.
  // With paired windows (launch_rb) the halo share drops from 88 % to 31 % of the output rows at k = 11 (39 % -> 16 % at k = 7) and the
  // fused kernel wins at C = 128 as well: k7 1546 us against 1999 layer by layer, k11 2194 against 2384 (ragged config-2 batch).
  if (C <= 64) return true;
  if (k == 3) return true;
  return g_rb_cluster >= 2 && !g_rb_wave;
}

// One fused ResBlock1.  c1[l] / c2[l]: packed conv weights (bf16 K-major, as conv_tc uses); bacc[l] = cumulative conv2
// biases (device, [C]).  x, sum: fp32 (B, L, C); act_out: bf16 (B, L, C) or nullptr.  A shape the kernel does not take is
// rejected (cudaErrorInvalidValue and a message in *err).
cudaError_t resblock_tc_launch(int C, int k, const ConvWeights* const c1[3], const ConvWeights* const c2[3], const float* const bacc[3],
                               const float* x, float* sum, bf16* act_out, int B, int L, int mode, float inv_n, float slope_out,
                               int write_f32, cudaStream_t s, std::string* err, RaggedPlanner* ragged, const RbSchedule* sched,
                               RbLaunchInfo* info) {
  rb_read_env();
  const char* bad = nullptr;
  if (C != 32 && C != 64 && C != 128) bad = "C must be 32, 64 or 128";
  else if (k != 3 && k != 7 && k != 11) bad = "k must be 3, 7 or 11";
  else if (c1[0]->dilation != 1 || c1[1]->dilation != 3 || c1[2]->dilation != 5) bad = "dilations must be (1, 3, 5)";
  else if (B <= 0 || L <= 0) bad = "empty batch";
  else if (mode < 0 || mode > 2) bad = "mode must be 0, 1 or 2";
  if (bad) {
    if (err) *err = std::string("resblock_tc: ") + bad;
    return cudaErrorInvalidValue;
  }
  RbMaps maps;
  RbParams p{};
  const int rb = C == 32 ? 64 : 128;
  for (int l = 0; l < 3; ++l) {
    const ConvWeights* cw[2] = {c1[l], c2[l]};
    for (int h = 0; h < 2; ++h) {
      const ConvWeights& w = *cw[h];
      if (!w.w_bf16 || w.C_in != C || w.N != C || w.taps != k || w.N_pad_tc != C || !w.bias) {
        if (err) *err = "resblock_tc: unexpected weight packing";
        return cudaErrorInvalidValue;
      }
      if (!tc_encode_bf16_map(&maps.m[2 * l + h], w.w_bf16, (uint64_t)w.K_pad, (uint64_t)w.N_pad_tc, (uint64_t)w.taps, (uint64_t)w.K_pad * 2,
                              (uint64_t)w.K_pad * w.N_pad_tc * 2, (uint32_t)(rb / 2), (uint32_t)C, rb, err))
        return cudaErrorInvalidValue;
    }
    p.bias1[l] = c1[l]->bias;
    p.bias2[l] = c2[l]->bias;
    p.bacc[l] = bacc[l];
    p.dil[l] = c1[l]->dilation;
  }
  p.x = x; p.x_bs = (long long)L * C;
  p.sum = sum; p.sum_bs = (long long)L * C;
  p.act_out = act_out; p.act_bs = (long long)L * C;
  p.L = L; p.k = k; p.mode = mode; p.inv_n = inv_n; p.slope_out = slope_out; p.write_f32 = write_f32;
  const RbSchedule sc = sched ? *sched : RbSchedule{};
  switch (C) {
    case 32: return launch_rb<32>(maps, p, B, s, ragged, sc, info, err);
    case 64: return launch_rb<64>(maps, p, B, s, ragged, sc, info, err);
    default: return launch_rb<128>(maps, p, B, s, ragged, sc, info, err);
  }
}

}  // namespace ev
