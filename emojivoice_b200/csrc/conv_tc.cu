// bf16 implicit-GEMM conv1d on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM), operands
// staged by TMA (cp.async.bulk.tensor, hardware swizzle) through mbarrier rings.  sm_100a only.
//
// Tile: MB x 128 output time steps (UMMA M = 128 = TMEM lanes, MB in {1,2} accumulators) x BN output channels
// (UMMA N = BN TMEM columns), reduced over K-chunks of BK channels x taps.
//   A (activations) : 3-D tensor map (channel, time, batch) over the channel-last bf16 tensor.  ONE haloed tile
//                     [BK ch x (MB*128 + (taps-1)*dilation) rows] is fetched per K-chunk at row m0 - pad (one or two TMA
//                     boxes); every tap's / m-block's MMA reads the same smem tile through a descriptor whose start
//                     address is advanced by whole rows (the swizzle is a function of absolute smem address bits, so
//                     no base-offset is needed -- verified on hardware).  Rows outside [0,T) are zero-filled by TMA,
//                     which IS the convolution's zero padding (no im2col, no halo copies in HBM).
//                     The stride-2 conv reads a (T/2, 2*ld) view of the same memory (tap_col selects even/odd rows).
//   B (weights)     : 3-D tensor map (c_in, n, tap) over [taps][N_pad][K_pad] bf16, box [BK x BN].  A weight tile is
//                     fetched ONCE per (K-chunk, tap) and used by all MB m-blocks (halves the L2->SM weight stream,
//                     which -- not the tensor pipe -- bounds 128x128 tiles); narrow layers keep all taps resident.
//   BK = 64 (128-byte swizzle) or, for layers with C_in <= 32, BK = 32 (64-byte swizzle: no zero-padded K).
// PERSISTENT CTAs walk the tile list; TMEM holds two accumulator sets so the epilogue of tile i overlaps the TMA/MMA
// main loop of tile i+1.  Narrow configurations run two CTAs per SM.
// Warp roles: warp 0 = TMA producer; warps 1-2 = MMA issuers, one per m-block (warp 1 also owns the TMEM allocation):
// the tensor core's instruction queue is shallow, so a single issuer's barrier waits and bookkeeping (~450 clk per
// weight tile) left the pipe idle about half of the time -- with all loads and stores disabled the MMA-bound layers
// ran no faster; two issuers on independent accumulators overlap one's bookkeeping with the other's MMAs;
// warps 3.. = 8 or 16 epilogue warps, per 32 x 32 block: residual loads issued -> tcgen05.ld -> private fp32 transpose
// buffer -> row-wise coalesced pass with the fused bias / mask / Euler-or-residual / MRF-mean / activation and stores
// (or the lean activation-only path, or the two-level-accumulation flush of the 3xTF32 mode).
#include <cuda.h>
#include <cudaTypedefs.h>

#include <algorithm>
#include <cstdlib>

#include "conv.cuh"
#include "tc_ptx.cuh"

namespace ev {
using namespace tc;
namespace {

constexpr int BM = 128;
constexpr int UMMA_K = 16;
constexpr int NUM_THREADS = 32 * (2 + 8);         // producer + 1 MMA issuer + 8 epilogue warps (two CTAs per SM: 96 regs x 640 threads)
constexpr int NUM_THREADS_WIDE = 32 * (3 + 16);   // producer + 2 MMA issuers (one per m-block) + 16 epilogue warps (one CTA per SM)
constexpr int MAX_A_SLOTS = 4, MAX_B_SLOTS = 8;
constexpr int MB_MAX = 2;
constexpr int kMaxGroups = kMaxTaps;
constexpr int SMEM_LIMIT = 224 * 1024;     // dynamic shared memory one CTA may ask for

struct TcParams {
  // ---- scalars first: everything the TMA producer / MMA issuers read before their first instruction of real work sits
  // in the first two constant-cache lines of the parameter block (a traced launch showed the lone producer thread
  // spending ~2400 clk between griddepcontrol.wait and its first TMA, mostly on cold constant loads and two IDIVs)
  int m_tiles, n_tiles, total_tiles;
  const int* rag;               // ragged batch: compact (item, m-tile) list (RaggedPlanner, conv.cuh) or nullptr = dense grid
  int mb;                       // m-blocks (128 rows) per tile
  int kchunks;
  int n_groups;                 // taps are processed in groups that share one activation tile (see grp_* below)
  int grp_taps;                 // taps per group (all groups alike: `taps` with halo reuse, else 1)
  int a_boxes, a_box_rows;      // the activation tile is a_boxes TMA boxes of a_box_rows rows each
  int a_slot_bytes;             // tile bytes rounded up to 1024
  int a_slots, b_slots;
  int bk, row_bytes, ksteps;    // K-chunk channels, bytes per smem row (= swizzle width), UMMA K-steps per chunk
  int b_tile_bytes;
  int resident;                 // all weight tiles stay in smem for the CTA's lifetime (narrow layers)
  int tf32;                     // split-operand path (3xTF32 or 3xFP16): K-chunks walk the sections [hi | hi | lo] of A
  int mma_tf32;                 // the MMAs are kind::tf32 (3xTF32); 0: kind::f16 (bf16 operands, or the fp16 halves of the 3xFP16 split)
  const float* descale;         // 3xFP16: descale[1] multiplies every partial sum when it is flushed (undoes the power-of-two pre-scaling)
  int kch1;                     // K-chunks per section (== kchunks unless tf32)
  int tf32_share;               // 3xTF32 with operand sharing: per 32-channel chunk c the steps (x_hi, w_lo) (x_hi, w_hi) (x_lo, w_hi)
                                // run back to back, the activation tile of step 0 is reused by step 1 and the weight tiles of
                                // step 1 by step 2: 2 + 2*taps tile loads per chunk instead of 3 + 3*taps (the path is L2->SM bound)
  int sec_off[3];               // column offset of each A section
  int idle_arrive;              // see `idle_issuer` in the kernel (EV_TC_IDLE_ARRIVE=0 switches it off)
  int debug_nob;                // EV_TC_DEBUG_NOB bit 0 / 1 / 2: skip weight loads / activation loads / lean-path stores.  Timing
                                // experiments only (results are wrong): they showed the MMA-bound layers are issue-bound, not memory-bound
  int trace;                    // EV_TC_TRACE=1: per-CTA clock64 stamps of the pipeline's milestones (scripts/conv_trace.py)
  unsigned long long div_n, div_m;   // ceil(2^44 / n_tiles), ceil(2^44 / m_tiles): tile -> (b, m-tile, n-tile) without IDIV
  int flush_kc;                 // K-chunks per accumulation group: the TMEM partial sum is flushed into an fp32 master
                                // accumulator (rounded adds) after every group; == kchunks means one group per tile
  int n_issuers;                // MMA issuer warps: 2 (one per m-block) in the wide configuration, else 1
  int act_only;                 // epilogue writes only the bf16 operand tensor (no residual / fp32 output): lean path
  int vec_ok;
  uint32_t desc_sbo, desc_layout;
  uint32_t tmem_cols;
  uint32_t idesc;               // instruction descriptor (kind::f16 bf16, or kind::tf32)
  uint32_t tap_first16;         // (byte offset of tap 0's first row inside a haloed tile) >> 4
  uint32_t tap_step16;          // (bytes from one tap's first row to the next one's) >> 4, two's complement when negative
  // with halo reuse all taps form one group whose tile covers rows [m0 + grp_row0, m0 + grp_row0 + a_rows); otherwise
  // every tap is its own group
  int grp_row0[kMaxGroups], grp_col0[kMaxGroups], grp_first[kMaxGroups], grp_count[kMaxGroups];
  int tap_byte_off[kMaxTaps];   // byte offset of tap j's first row inside its group's tile
  ConvGeom g;
  Epilogue e;
};

// tile index -> (batch item, m-tile, n-tile) with two multiplies (exact for tile < 2^22 and divisors < 2^20)
__device__ __forceinline__ void decode_tile(const TcParams& p, int tile, int& b, int& mt, int& nt) {
  const uint32_t rest = (uint32_t)(((unsigned long long)(uint32_t)tile * p.div_n) >> 44);
  nt = tile - (int)rest * p.n_tiles;
  if (p.rag) {      // ragged batch: the (item, m-tile) pairs that hold needed rows are listed explicitly
    const int pair = __ldg(p.rag + 1 + rest);
    b = pair >> 16;
    mt = pair & 0xffff;
    return;
  }
  b = (int)(((unsigned long long)rest * p.div_m) >> 44);
  mt = (int)rest - b * p.m_tiles;
}

// [CTA][16] clock stamps of the most recent traced launch (diagnostic; read back by ev_test_conv_trace)
__device__ unsigned long long g_trace[512 * 24];
#define EV_TR(i) do { if (p.trace && lane == 0 && blockIdx.x < 512) g_trace[blockIdx.x * 24 + (i)] = (unsigned long long)clock64(); } while (0)
// accumulated clocks a role spent inside mbarrier waits (slots 16..19), written once at the end of the role's loop
#define EV_TW_BEGIN() long long _tw0 = p.trace ? clock64() : 0
#define EV_TW_END(acc) do { if (p.trace) (acc) += clock64() - _tw0; } while (0)
#define EV_TW_STORE(i, acc) do { if (p.trace && lane == 0 && blockIdx.x < 512) g_trace[blockIdx.x * 24 + (i)] = (unsigned long long)(acc); } while (0)

// Upper / lower words of a shared-memory matrix descriptor (tc_ptx.cuh make_smem_desc_ex): the MMA warp advances the
// low word by plain adds instead of rebuilding descriptors.
__device__ __forceinline__ uint32_t desc_hi_word(uint32_t sbo, uint32_t layout) { return ((sbo >> 4) & 0x3FFFu) | (1u << 14) | (layout << 29); }
__device__ __forceinline__ uint32_t desc_lo_word(uint32_t saddr) { return ((saddr & 0x3FFFFu) >> 4) | (1u << 16); }
__device__ __forceinline__ uint64_t desc_join(uint32_t hi, uint32_t lo) { return ((uint64_t)hi << 32) | lo; }

// All MMAs of one (K-chunk, tap): VMB m-blocks x KS K-steps, issued by the elected lane.
template <int KS, bool TF32>
__device__ __forceinline__ void issue_tap(uint32_t d_tmem, uint32_t hi, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t acc) {
#pragma unroll
  for (int k = 0; k < KS; ++k) {
    if (TF32) umma_tf32(d_tmem, desc_join(hi, a_lo + 2u * k), desc_join(hi, b_lo + 2u * k), idesc, (acc | (uint32_t)k) ? 1u : 0u);
    else umma_bf16(d_tmem, desc_join(hi, a_lo + 2u * k), desc_join(hi, b_lo + 2u * k), idesc, (acc | (uint32_t)k) ? 1u : 0u);
  }
}

constexpr int STAGE_LD = 36;                                   // floats per staged row (32 + 4: conflict-free float4 access)
constexpr int STAGING_WARP_BYTES = 32 * STAGE_LD * 4;          // one private 32 x 32 transpose buffer per epilogue warp
constexpr int ACT_PITCH = 80;                                  // bytes per staged bf16 row (64 + 16: conflict-free 16-byte access)

// generic scalar epilogue of one staged 32 x 32 block (unaligned strides / channel counts that are not multiples of 4);
// kept out of line so the hot vector path stays compact in the instruction cache
__device__ __noinline__ void scalar_block(const TcParams& p, const float* wstage, int b, int r0, int c0, int lane) {
  const Epilogue& e = p.e;
  bf16* out_act = reinterpret_cast<bf16*>(e.out_act);
  for (int idx = lane; idx < 32 * 32; idx += 32) {
    const int rl = idx >> 5, nl = idx & 31;
    const int r = r0 + rl, nn = c0 + nl;
    if (r >= p.g.M || nn >= p.g.N) continue;
    int t, cc;
    if (!ep_coord(e, r, nn, t, cc)) continue;
    const float mv = e.mask.at(b, t);
    const float v = ep_value(e, b, t, cc, wstage[rl * STAGE_LD + nl], mv);
    if (e.out_f32) e.out_f32[b * e.f32_bs + (long long)t * e.f32_ld + cc] = e.f32_is_act ? ep_act(e, cc, v, mv) : v;
    if (out_act) out_act[b * e.act_bs + (long long)t * e.act_ld + cc] = __float2bfloat16_rn(ep_act(e, cc, v, mv));
  }
}

// ------------------------------------------------------------------------------------------------ the kernel
template <int BN>
__global__ void __launch_bounds__(NUM_THREADS_WIDE, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t a_full[MAX_A_SLOTS], a_empty[MAX_A_SLOTS], b_full[MAX_B_SLOTS], b_empty[MAX_B_SLOTS];
  __shared__ __align__(8) uint64_t acc_full[2], acc_empty[2];
  __shared__ uint32_t tmem_base_smem;

  const uint32_t tiles0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t a_base = tiles0, b_base = tiles0 + (uint32_t)(p.a_slots * p.a_slot_bytes);
  float* stage = reinterpret_cast<float*>(smem_raw + (tiles0 - smem_u32(smem_raw)) + p.a_slots * p.a_slot_bytes + p.b_slots * p.b_tile_bytes);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0) {
    EV_TR(0);
    if (p.trace && lane == 0 && blockIdx.x < 512) { unsigned long long gt; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt)); g_trace[blockIdx.x * 24 + 11] = gt; }
  }
  const int A_SLOTS = p.a_slots, B_SLOTS = p.b_slots;
  const int tile_rows = p.mb * BM;
  const int ROLE_WARPS = 1 + p.n_issuers;   // producer + issuers; the epilogue warps follow

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    // two MMA-issuer warps: each one commits on the slot / accumulator barriers
    for (int s = 0; s < MAX_A_SLOTS; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], p.n_issuers); }
    for (int s = 0; s < MAX_B_SLOTS; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], p.n_issuers); }
    for (int s = 0; s < 2; ++s) { mbar_init(&acc_full[s], p.n_issuers); mbar_init(&acc_empty[s], (blockDim.x >> 5) - ROLE_WARPS); }   // every epilogue warp releases
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "r"(p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // every role decodes its first tile (and pulls the parameter block through the constant cache) BEFORE the barrier and
  // the programmatic-dependency wait: this part overlaps the TMEM allocation and, under PDL, the previous kernel's tail
  int first_b = 0, first_mt = 0, first_nt = 0;
  if (!p.rag) decode_tile(p, (int)blockIdx.x, first_b, first_mt, first_nt);
  asm volatile("" ::"r"(first_b), "r"(first_mt), "r"(first_nt));
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_base_smem;
  if (warp == 0) EV_TR(1);
  pdl_trigger();     // the next kernel may start its prologue
  pdl_wait();        // everything above overlapped the previous kernel's tail; its results are visible from here on
  if (warp == 0) EV_TR(2);
  // ragged batch: the tile count and the tile list live in device memory (written by an earlier kernel of the stream)
  const int total_tiles = p.rag ? __ldg(p.rag) * p.n_tiles : p.total_tiles;
  if (p.rag && (int)blockIdx.x < total_tiles) decode_tile(p, (int)blockIdx.x, first_b, first_mt, first_nt);

  if (warp == 0) {
    if (lane == 0) {
      // ---------------- TMA producer: per tile, per K-chunk, per tap group: one (haloed) activation tile, then one
      // weight tile per tap.  Ring positions run on across tiles, so the next tile's loads start while this one computes.
      int sa = 0, sb = 0;
      long long tw_a = 0, tw_b = 0;
      uint32_t pa = 1, pb = 1;      // parity to wait for on the "empty" barriers (fresh barriers pass parity 1)
      const uint32_t a_bytes = (uint32_t)(p.a_boxes * p.a_box_rows * p.row_bytes), box_bytes = (uint32_t)(p.a_box_rows * p.row_bytes);
      const int kchunks = p.kchunks, n_groups = p.n_groups, grp_taps = p.grp_taps;
      const bool resident = p.resident != 0;
      if (resident) {   // narrow layers: every (K-chunk, tap) weight tile is fetched once and kept
        const int n_w = kchunks * p.g.taps;
        mbar_expect_tx(&b_full[0], (uint32_t)(n_w * p.b_tile_bytes));
        for (int kc = 0; kc < kchunks; ++kc)
          for (int j = 0; j < p.g.taps; ++j)
            tma_load_3d(b_base + (uint32_t)((kc * p.g.taps + j) * p.b_tile_bytes), &tmB, &b_full[0], kc * p.bk, 0, j);
      }
      EV_TR(12);
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        int nt = first_nt, mt = first_mt, b = first_b;
        if (tile != (int)blockIdx.x) decode_tile(p, tile, b, mt, nt);
        const int m0 = mt * tile_rows, n0 = nt * BN;
        if (tile == (int)blockIdx.x) EV_TR(13);
        for (int kc = 0; kc < kchunks; ++kc) {
          for (int g = 0; g < n_groups; ++g) {
            const int sh_c = kc / 3, sh_s = kc - 3 * sh_c;       // operand-sharing walk (tf32_share): chunk, step
            if (p.tf32_share) {
              if (sh_s != 1) {     // step 1 reuses step 0's activation tile
                { EV_TW_BEGIN(); mbar_wait(&a_empty[sa], pa); EV_TW_END(tw_a); }
                mbar_expect_tx(&a_full[sa], a_bytes);
                const uint32_t dst = a_base + (uint32_t)(sa * p.a_slot_bytes);
                const int col = p.grp_col0[0] + (sh_s == 2 ? p.sec_off[2] : 0) + sh_c * p.bk, row = m0 + p.grp_row0[0];
                tma_load_3d(dst, &tmA, &a_full[sa], col, row, b);
                if (p.a_boxes > 1) tma_load_3d(dst + box_bytes, &tmA, &a_full[sa], col, row + p.a_box_rows, b);
                if (++sa == A_SLOTS) { sa = 0; pa ^= 1u; }
              }
              if (sh_s != 2) {     // step 2 reuses step 1's weight tiles; sections of the packed weights are [hi | lo | hi]
                const int wcol = (sh_s == 0 ? p.kch1 * p.bk : 0) + sh_c * p.bk;
                for (int j = 0; j < grp_taps; ++j) {
                  { EV_TW_BEGIN(); mbar_wait(&b_empty[sb], pb); EV_TW_END(tw_b); }
                  mbar_expect_tx(&b_full[sb], (uint32_t)p.b_tile_bytes);
                  tma_load_3d(b_base + (uint32_t)(sb * p.b_tile_bytes), &tmB, &b_full[sb], wcol, n0, j);
                  if (++sb == B_SLOTS) { sb = 0; pb ^= 1u; }
                }
              }
              continue;
            }
            { EV_TW_BEGIN(); mbar_wait(&a_empty[sa], pa); EV_TW_END(tw_a); }
            if (tile == (int)blockIdx.x && kc == 0 && g == 0) EV_TR(14);
            if (p.debug_nob & 2) { mbar_arrive(&a_full[sa]); if (++sa == A_SLOTS) { sa = 0; pa ^= 1u; } if (resident) continue; goto b_loads; }
            mbar_expect_tx(&a_full[sa], a_bytes);
            {
            const uint32_t dst = a_base + (uint32_t)(sa * p.a_slot_bytes);
            const int sec = (kc >= p.kch1) + (kc >= 2 * p.kch1);   // 3xTF32: K-chunks walk the A sections [hi | hi | lo]; otherwise one section
            const int col = p.grp_col0[g] + p.sec_off[sec] + (kc - sec * p.kch1) * p.bk, row = m0 + p.grp_row0[g];
            tma_load_3d(dst, &tmA, &a_full[sa], col, row, b);
            if (p.a_boxes > 1) tma_load_3d(dst + box_bytes, &tmA, &a_full[sa], col, row + p.a_box_rows, b);
            }
            if (++sa == A_SLOTS) { sa = 0; pa ^= 1u; }
            if (tile == (int)blockIdx.x && kc == 0 && g == 0) EV_TR(3);
            if (resident) continue;
          b_loads:
            const int tap0 = g * grp_taps;
            for (int j = 0; j < grp_taps; ++j) {
              { EV_TW_BEGIN(); mbar_wait(&b_empty[sb], pb); EV_TW_END(tw_b); }
              if (p.debug_nob & 1) { mbar_arrive(&b_full[sb]); }   // timing experiment only: no weight traffic (results are wrong)
              else {
              mbar_expect_tx(&b_full[sb], (uint32_t)p.b_tile_bytes);
              tma_load_3d(b_base + (uint32_t)(sb * p.b_tile_bytes), &tmB, &b_full[sb], kc * p.bk, n0, tap0 + j);
              }
              if (++sb == B_SLOTS) { sb = 0; pb ^= 1u; }
            }
          }
        }
      }
      EV_TW_STORE(18, tw_b); EV_TW_STORE(19, tw_a);
    }
    __syncwarp();
  } else if (warp < ROLE_WARPS) {
    // ---------------- two MMA issuer warps: warp 1 owns m-block 0, warp 2 owns m-block 1 of every tile (independent
    // accumulators), so one warp's barrier / bookkeeping work overlaps the other's MMAs -- the tensor core's instruction
    // queue is shallow and a single issuer left the pipe idle ~half of the time.  Each warp walks the (warp-uniform) loops and waits the (warp-uniform) loops and waits; one elected lane issues.
    // Every tap and m-block re-reads the same smem tile at a row offset.  The loop body is kept to a few dozen
    // instructions per weight tile: ring slots / phases advance incrementally and descriptors by adds (a single
    // warp issues ~1 dependent instruction per 5-8 clk, so 200 instructions per tap would cap the tensor pipe).
    const uint32_t idesc = p.idesc;
    const bool tf32 = p.mma_tf32 != 0;
    const uint32_t hi = desc_hi_word(p.desc_sbo, p.desc_layout);
    const uint32_t mb_step16 = (uint32_t)(BM * p.row_bytes) >> 4, tap_step16 = p.tap_step16;
    const uint32_t b_step16 = (uint32_t)p.b_tile_bytes >> 4, a_step16 = (uint32_t)p.a_slot_bytes >> 4;
    const uint32_t a_lo0 = desc_lo_word(a_base), b_lo0 = desc_lo_word(b_base);
    const int kchunks = p.kchunks, n_groups = p.n_groups, grp_taps = p.grp_taps;
    const bool resident = p.resident != 0, ks4 = p.ksteps == 4;
    const uint32_t acc_stride = (uint32_t)(p.mb * BN);
    const int my_mb = warp - 1, mb_stride = p.n_issuers;   // this issuer owns m-blocks my_mb, my_mb + mb_stride, ...
    int sa = 0, sb = 0, vt = 0;     // vt counts accumulator-set uses: one per tile, or one per flush group (3xTF32)
    // An issuer warp that owns no valid m-block of the tile (the second issuer of a one-m-block tile) has nothing in flight: it keeps
    // the barrier protocol with plain arrivals instead of tcgen05.commit, which would queue behind the other warp's MMAs
    bool idle_issuer = false;
    auto signal = [&](uint64_t* bar) { if (idle_issuer) mbar_arrive(bar); else umma_commit(bar); };
    long long tw_a = 0, tw_b = 0, tw_acc = 0;
    uint32_t pa = 0, pb = 0;        // parity to wait for on the "full" barriers
    int sh_sb = 0; uint32_t sh_pb = 0;   // tf32_share: ring position of the weight tiles that step 2 reuses
    const int flush_kc = p.flush_kc;
    if (resident) { mbar_wait(&b_full[0], 0); tcgen05_fence_after(); }
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      int mt = first_mt;
      if (tile != (int)blockIdx.x) { int b_, nt_; decode_tile(p, tile, b_, mt, nt_); }
      const int vmb = min(p.mb, (p.g.M - mt * tile_rows + BM - 1) / BM);     // m-blocks that hold valid rows
      idle_issuer = p.idle_arrive && my_mb >= vmb && !(mb_stride == 1 && vmb > 1);
      int buf = 0, in_group = 0;
      uint32_t d_tmem = 0;
      uint32_t acc = 0;
      uint32_t b_res_lo = b_lo0;    // resident weights: tiles are laid out in (K-chunk, tap) order
      for (int kc = 0; kc < kchunks; ++kc) {
        if (in_group == 0) {        // open an accumulation group on the next accumulator set
          buf = vt & 1;
          { EV_TW_BEGIN(); mbar_wait(&acc_empty[buf], ((uint32_t)(vt >> 1) & 1u) ^ 1u); EV_TW_END(tw_acc); }   // epilogue has drained this accumulator set
          tcgen05_fence_after();
          d_tmem = tmem_base + (uint32_t)buf * acc_stride;
          acc = 0;
        }
        if (p.tf32_share) {
          // operand-sharing walk (one issuer, one m-block, one tap group): see TcParams::tf32_share
          const int sh_s = kc % 3;
          if (sh_s != 1) { EV_TW_BEGIN(); mbar_wait(&a_full[sa], pa); EV_TW_END(tw_a); tcgen05_fence_after(); }     // step 1 reads step 0's tile again
          const uint32_t a_lo_s = a_lo0 + (uint32_t)sa * a_step16 + p.tap_first16;
          if (sh_s == 1) { sh_sb = sb; sh_pb = pb; }                                  // step 2 walks step 1's weight slots again
          if (sh_s == 2) { sb = sh_sb; pb = sh_pb; }
          uint32_t a_lo = a_lo_s;
          for (int j = 0; j < grp_taps; ++j) {
            if (sh_s != 2) { EV_TW_BEGIN(); mbar_wait(&b_full[sb], pb); EV_TW_END(tw_b); tcgen05_fence_after(); }
            const uint32_t b_lo = b_lo0 + (uint32_t)sb * b_step16;
            if (elect_one()) {     // both issuer warps keep the barrier protocol; only the one that owns a valid m-block issues
              if (my_mb < vmb) {
                if (tf32) issue_tap<4, true>(d_tmem + (uint32_t)(my_mb * BN), hi, a_lo + (uint32_t)my_mb * mb_step16, b_lo, idesc, acc);
                else issue_tap<4, false>(d_tmem + (uint32_t)(my_mb * BN), hi, a_lo + (uint32_t)my_mb * mb_step16, b_lo, idesc, acc);
              }
              if (sh_s != 1) signal(&b_empty[sb]);                              // step 1's weight tiles stay for step 2
            }
            __syncwarp();
            acc = 1;
            a_lo += tap_step16;
            if (++sb == B_SLOTS) { sb = 0; pb ^= 1u; }
          }
          if (sh_s != 0) {                                                            // step 0's activation tile stays for step 1
            if (elect_one()) signal(&a_empty[sa]);
            __syncwarp();
            if (++sa == A_SLOTS) { sa = 0; pa ^= 1u; }
          }
        } else
        for (int g = 0; g < n_groups; ++g) {
          { EV_TW_BEGIN(); mbar_wait(&a_full[sa], pa); EV_TW_END(tw_a); }
          tcgen05_fence_after();
          if (warp == 1 && tile == (int)blockIdx.x && kc == 0 && g == 0) EV_TR(4);
          uint32_t a_lo = a_lo0 + (uint32_t)sa * a_step16 + p.tap_first16;
          for (int j = 0; j < grp_taps; ++j) {
            uint32_t b_lo;
            if (resident) {
              b_lo = b_res_lo;
              b_res_lo += b_step16;
            } else {
              { EV_TW_BEGIN(); mbar_wait(&b_full[sb], pb); EV_TW_END(tw_b); }
              tcgen05_fence_after();
              b_lo = b_lo0 + (uint32_t)sb * b_step16;
            }
            if (elect_one()) {
              // straight-line issue (MB_MAX = 2): this issuer's own m-block, plus m-block 1 when it is the only issuer;
              // an issuer without a valid m-block only keeps the barrier protocol going
              const bool second = mb_stride == 1 && vmb > 1;
              const uint32_t dm = d_tmem + (uint32_t)(my_mb * BN), am = a_lo + (uint32_t)my_mb * mb_step16;
              if (tf32) {
                if (my_mb < vmb) issue_tap<4, true>(dm, hi, am, b_lo, idesc, acc);
                if (second) issue_tap<4, true>(dm + (uint32_t)BN, hi, am + mb_step16, b_lo, idesc, acc);
              } else if (ks4) {
                if (my_mb < vmb) issue_tap<4, false>(dm, hi, am, b_lo, idesc, acc);
                if (second) issue_tap<4, false>(dm + (uint32_t)BN, hi, am + mb_step16, b_lo, idesc, acc);
              } else {
                if (my_mb < vmb) issue_tap<2, false>(dm, hi, am, b_lo, idesc, acc);
                if (second) issue_tap<2, false>(dm + (uint32_t)BN, hi, am + mb_step16, b_lo, idesc, acc);
              }
              if (!resident) signal(&b_empty[sb]);   // weight slot is free once both issuers' MMAs have read it
            }
            __syncwarp();
            acc = 1;
            a_lo += tap_step16;
            if (!resident) { if (++sb == B_SLOTS) { sb = 0; pb ^= 1u; } }
          }
          if (elect_one()) signal(&a_empty[sa]);     // activation tile is free once every tap of the group has read it
          __syncwarp();
          if (++sa == A_SLOTS) { sa = 0; pa ^= 1u; }
        }
        if (++in_group == flush_kc || kc == kchunks - 1) {   // group complete -> epilogue (output pass or partial-sum flush)
          if (elect_one()) signal(&acc_full[buf]);
          __syncwarp();
          if (warp == 1) { if (tile == (int)blockIdx.x) EV_TR(5); EV_TR(6); }
          in_group = 0;
          ++vt;
        }
      }
    }
    if (warp == 1) { EV_TW_STORE(16, tw_b); EV_TW_STORE(17, tw_a); EV_TW_STORE(20, tw_acc); }
  } else {
    // ---------------- epilogue (warps 2..9).  Warp (q, half) owns TMEM lanes [32q, 32q+32) and every second 32-column
    // block of them; the eight warps run free of each other (no CTA barrier):
    //   residual loads issued -> tcgen05.ld (thread = accumulator row) -> private 32 x 32 fp32 transpose buffer ->
    //   row-wise pass: 8 lanes x float4 per row, fused epilogue arithmetic, coalesced fp32 + bf16 stores.
    const int ew = warp - ROLE_WARPS;
    const int q = warp & 3, slot = ew >> 2, n_slots = ((int)(blockDim.x >> 5) - ROLE_WARPS) >> 2;   // 2 or 4 warps per lane quadrant
    const Epilogue& e = p.e;
    bf16* out_act = reinterpret_cast<bf16*>(e.out_act);
    const bool has_res = e.res != nullptr, has_res2 = e.res2 != nullptr, has_f32 = e.out_f32 != nullptr, has_act = e.out_act != nullptr;
    const bool use_div = e.div != 1.0f, snake = e.act == ACT_SNAKE, use_alpha = e.alpha != 1.0f;
    const bool mask_pre = e.mask_pre != 0, mask_act = e.mask_act != 0, polyphase = e.phase_cout != p.g.N;
    const bool f32_act = has_f32 && e.f32_is_act != 0;
    const float inv_div = 1.0f / e.div;   // bf16-operand path: x * (1/3) instead of the reference's x / 3 (1 ulp, far inside tolerance)
    const float slope = e.act == ACT_LRELU ? e.slope : (e.act == ACT_RELU ? 0.0f : 1.0f);
    const float alpha = e.alpha;
    constexpr int NBLK = BN / 32;                      // 32-column blocks per accumulator
    constexpr int U = 8;                               // row-pass iterations: 4 rows x (8 lanes x float4) each
    const int sub = lane >> 3, cl = (lane & 7) * 4;
    float* wstage = stage + ew * (32 * STAGE_LD);
    const bool act_only = p.act_only != 0;
    float* srow_w = wstage + lane * STAGE_LD;
    const float* srow_r = wstage + sub * STAGE_LD + cl;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    const int M = p.g.M, N = p.g.N, T_out = e.T_out;
    const int up_s = e.up_s, up_p = e.up_p;

    int ti = 0;                      // accumulator-set use counter (see the MMA warp's vt)
    const int n_grp = (p.kchunks + p.flush_kc - 1) / p.flush_kc;   // accumulation groups per tile (1 unless 3xTF32)
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ti += n_grp) {
      int nt = first_nt, mt = first_mt, b = first_b;
      if (tile != (int)blockIdx.x) decode_tile(p, tile, b, mt, nt);
      const int m0 = mt * tile_rows, n0 = nt * BN;
      const int vmb = min(p.mb, (M - m0 + BM - 1) / BM);
      const int buf = ti & 1;
      const int len_b = e.mask.lens ? __ldg(e.mask.lens + b) : 0x7fffffff;
      const int n_blk = vmb * NBLK;                    // this quadrant's blocks; the warp takes slot, slot+n_slots, ...
      bool waited = false;
#pragma unroll 1
      for (int blk = slot; blk < n_blk; blk += n_slots) {
        const int mb = blk / NBLK, cb = blk - mb * NBLK;
        if (act_only) {
          // ---- lean path: bias + activation + bf16 pack in the accumulator layout (thread = row), bf16 staging
          if (!waited) {
            mbar_wait(&acc_full[buf], (uint32_t)(ti >> 1) & 1u);
            tcgen05_fence_after();
            waited = true;
          }
          uint32_t raw[32];
          tmem_ld32(lane_addr + (uint32_t)(buf * p.mb * BN + mb * BN + cb * 32), raw);
          if (blk + n_slots >= n_blk) {
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
          }
          const int nb = n0 + cb * 32;                 // first output channel of the block (N % 32 == 0 on this path)
          // the last n-tile of a layer with N % BN != 0 holds blocks past C_out: their accumulator columns are read and released
          // above like any other, but they have no bias, no SnakeBeta parameters and no output columns
          if (nb >= N) continue;
          const int row = m0 + mb * BM + q * 32 + lane;
          const float mv = (mask_act && !((row << e.mask.shift) < len_b)) ? 0.0f : 1.0f;
          uint8_t* brow = reinterpret_cast<uint8_t*>(wstage) + lane * ACT_PITCH;
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            float v[8];
            const float4 b0 = e.bias ? __ldg(reinterpret_cast<const float4*>(e.bias + nb + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
            const float4 b1 = e.bias ? __ldg(reinterpret_cast<const float4*>(e.bias + nb + j + 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
            v[0] = __uint_as_float(raw[j]) + b0.x; v[1] = __uint_as_float(raw[j + 1]) + b0.y;
            v[2] = __uint_as_float(raw[j + 2]) + b0.z; v[3] = __uint_as_float(raw[j + 3]) + b0.w;
            v[4] = __uint_as_float(raw[j + 4]) + b1.x; v[5] = __uint_as_float(raw[j + 5]) + b1.y;
            v[6] = __uint_as_float(raw[j + 6]) + b1.z; v[7] = __uint_as_float(raw[j + 7]) + b1.w;
            if (snake) {
              const float4 sa0 = __ldg(reinterpret_cast<const float4*>(e.snake_a + nb + j)), sa1 = __ldg(reinterpret_cast<const float4*>(e.snake_a + nb + j + 4));
              const float4 sb0 = __ldg(reinterpret_cast<const float4*>(e.snake_invb + nb + j)), sb1 = __ldg(reinterpret_cast<const float4*>(e.snake_invb + nb + j + 4));
              const float sa[8] = {sa0.x, sa0.y, sa0.z, sa0.w, sa1.x, sa1.y, sa1.z, sa1.w};
              const float sb[8] = {sb0.x, sb0.y, sb0.z, sb0.w, sb1.x, sb1.y, sb1.z, sb1.w};
#pragma unroll
              for (int i = 0; i < 8; ++i) { const float sn = __sinf(v[i] * sa[i]); v[i] = mv != 0.0f ? fmaf(sb[i], sn * sn, v[i]) : 0.0f; }
            } else {
#pragma unroll
              for (int i = 0; i < 8; ++i) v[i] = mv != 0.0f ? fmaxf(v[i], v[i] * slope) : 0.0f;
            }
            uint32_t w[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) { __nv_bfloat162 h2 = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]); w[i] = *reinterpret_cast<uint32_t*>(&h2); }
            *reinterpret_cast<uint4*>(brow + j * 2) = make_uint4(w[0], w[1], w[2], w[3]);
          }
          __syncwarp();
          {   // row-wise: 4 lanes x 16 B per row, 8 rows per warp instruction
            const int rsub = lane >> 2, ch = lane & 3;
            bf16* dst = out_act + b * e.act_bs + nb + ch * 8;
            const uint8_t* src = reinterpret_cast<const uint8_t*>(wstage) + ch * 16;
            const int rb = m0 + mb * BM + q * 32 + rsub;
#pragma unroll
            for (int it = 0; it < 4; ++it) {
              const int r = rb + it * 8;
              if (r < M && r < T_out && !(p.debug_nob & 4))
                *reinterpret_cast<uint4*>(dst + (long long)r * e.act_ld) = *reinterpret_cast<const uint4*>(src + (rsub + it * 8) * ACT_PITCH);
            }
          }
          __syncwarp();
          continue;
        }
        const int n = n0 + cb * 32 + cl;
        const bool n_ok = n < N;
        int co = n, phase = 0;
        if (polyphase && n_ok) { phase = n / e.phase_cout; co = n - phase * e.phase_cout; }
        const int r0 = m0 + mb * BM + q * 32 + sub;
        const int t0 = up_s * r0 + phase - up_p, dt = up_s * 4;
        float4 rr[U];
        if (p.vec_ok && (has_res || has_res2)) {   // residual loads fly while the accumulator is fetched and staged
          const float* res_p = has_res ? e.res + b * e.res_bs + co : nullptr;
          // the second residual (MRF partial sum) is fetched here too and folded into rr: read inside the row loop below it would sit
          // behind the previous row's store to the same array (out_f32 == res2) -- one DRAM latency per row instead of one per block
          const float* res2_p = has_res2 ? e.res2 + b * e.res2_bs + co : nullptr;
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int t = t0 + u * dt;
            const bool ok = n_ok && (r0 + 4 * u) < M && (unsigned)t < (unsigned)T_out;
            rr[u] = (ok && has_res) ? *reinterpret_cast<const float4*>(res_p + (long long)t * e.res_ld) : make_float4(0.f, 0.f, 0.f, 0.f);
            if (ok && has_res2) {
              const float4 r2 = *reinterpret_cast<const float4*>(res2_p + (long long)t * e.res2_ld);
              rr[u].x += r2.x; rr[u].y += r2.y; rr[u].z += r2.z; rr[u].w += r2.w;
            }
          }
        }
        if (n_grp > 1) {
          // two-level accumulation (3xTF32 / 3xFP16): this warp owns exactly one block; every group's TMEM partial sum is added
          // with rounded fp32 adds into the master accumulator kept in the warp's transpose buffer (3xFP16: times the power of
          // two that undoes the operands' pre-scaling -- exact, so still one rounding per add)
          const float ds = p.descale ? __ldg(p.descale + 1) : 1.0f;
#pragma unroll 1
          for (int grp = 0; grp < n_grp; ++grp) {
            const int v = ti + grp, vb = v & 1;
            mbar_wait(&acc_full[vb], (uint32_t)(v >> 1) & 1u);
            tcgen05_fence_after();
            uint32_t raw[32];
            tmem_ld32(lane_addr + (uint32_t)(vb * p.mb * BN + mb * BN + cb * 32), raw);
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[vb]);
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              float4 m4 = make_float4(0.f, 0.f, 0.f, 0.f);
              if (grp > 0) m4 = *reinterpret_cast<const float4*>(srow_w + j);
              m4.x = fmaf(__uint_as_float(raw[j]), ds, m4.x); m4.y = fmaf(__uint_as_float(raw[j + 1]), ds, m4.y);
              m4.z = fmaf(__uint_as_float(raw[j + 2]), ds, m4.z); m4.w = fmaf(__uint_as_float(raw[j + 3]), ds, m4.w);
              *reinterpret_cast<float4*>(srow_w + j) = m4;
            }
          }
          __syncwarp();
        } else {
          if (!waited) {
            mbar_wait(&acc_full[buf], (uint32_t)(ti >> 1) & 1u);
            tcgen05_fence_after();
            waited = true;
            if (ew == 0 && tile == (int)blockIdx.x) EV_TR(7);
          }
          {
            uint32_t raw[32];
            tmem_ld32(lane_addr + (uint32_t)(buf * p.mb * BN + mb * BN + cb * 32), raw);
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              *reinterpret_cast<uint4*>(srow_w + j) = make_uint4(raw[j], raw[j + 1], raw[j + 2], raw[j + 3]);
          }
          if (blk + n_slots >= n_blk) {      // last TMEM read of this warp for the tile: hand the accumulators back
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
          }
          __syncwarp();
        }
        if (p.vec_ok) {
          float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f), sa4 = bias4, sb4 = bias4;
          if (n_ok && e.bias) bias4 = __ldg(reinterpret_cast<const float4*>(e.bias + co));
          if (n_ok && snake) {
            sa4 = __ldg(reinterpret_cast<const float4*>(e.snake_a + co));
            sb4 = __ldg(reinterpret_cast<const float4*>(e.snake_invb + co));
          }
          float* f32_p = has_f32 ? e.out_f32 + b * e.f32_bs + co : nullptr;
          bf16* act_p = has_act ? out_act + b * e.act_bs + co : nullptr;
          float gs = 0.0f, gq = 0.0f;
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int t = t0 + u * dt;
            const bool ok = n_ok && (r0 + 4 * u) < M && (unsigned)t < (unsigned)T_out;
            if (!ok) continue;
            const float4 a4 = *reinterpret_cast<const float4*>(srow_r + u * 4 * STAGE_LD);
            float v0 = a4.x + bias4.x, v1 = a4.y + bias4.y, v2 = a4.z + bias4.z, v3 = a4.w + bias4.w;
            const float mv = ((t << e.mask.shift) < len_b) ? 1.0f : 0.0f;
            if (mask_pre && mv == 0.0f) { v0 = v1 = v2 = v3 = 0.0f; }   // a select, not a multiply: a padded row may hold anything
            if (use_alpha) { v0 *= alpha; v1 *= alpha; v2 *= alpha; v3 *= alpha; }
            if (has_res || has_res2) { v0 += rr[u].x; v1 += rr[u].y; v2 += rr[u].z; v3 += rr[u].w; }
            if (use_div) { v0 *= inv_div; v1 *= inv_div; v2 *= inv_div; v3 *= inv_div; }
            if (has_f32 && !f32_act) *reinterpret_cast<float4*>(f32_p + (long long)t * e.f32_ld) = make_float4(v0, v1, v2, v3);
            if (e.gn_sum) { gs += (v0 + v1) + (v2 + v3); gq += (v0 * v0 + v1 * v1) + (v2 * v2 + v3 * v3); }
            if (has_act || f32_act) {
              float a0, a1, a2, a3;
              if (snake) {   // y + sin^2(y*e^alpha) / (e^beta + 1e-9); fast sine is ample for bf16 operands
                const float s0 = __sinf(v0 * sa4.x), s1 = __sinf(v1 * sa4.y), s2 = __sinf(v2 * sa4.z), s3 = __sinf(v3 * sa4.w);
                a0 = fmaf(sb4.x, s0 * s0, v0); a1 = fmaf(sb4.y, s1 * s1, v1); a2 = fmaf(sb4.z, s2 * s2, v2); a3 = fmaf(sb4.w, s3 * s3, v3);
              } else {       // LeakyReLU(slope) for slope in [0,1]: max(v, v*slope); slope = 1 is the identity
                a0 = fmaxf(v0, v0 * slope); a1 = fmaxf(v1, v1 * slope); a2 = fmaxf(v2, v2 * slope); a3 = fmaxf(v3, v3 * slope);
              }
              if (mask_act && mv == 0.0f) { a0 = a1 = a2 = a3 = 0.0f; }
              if (f32_act) *reinterpret_cast<float4*>(f32_p + (long long)t * e.f32_ld) = make_float4(a0, a1, a2, a3);
              if (has_act) {
                __nv_bfloat162 lo = __floats2bfloat162_rn(a0, a1), hi = __floats2bfloat162_rn(a2, a3);
                uint2 pk;
                pk.x = *reinterpret_cast<uint32_t*>(&lo);
                pk.y = *reinterpret_cast<uint32_t*>(&hi);
                *reinterpret_cast<uint2*>(act_p + (long long)t * e.act_ld) = pk;
              }
            }
          }
          if (e.gn_sum && n0 + cb * 32 < N) {   // the block's 32 columns are one GroupNorm group: one fp64 atomic pair per warp and block
                                                // (a block past C_out has no group)
            gs = warp_sum(gs); gq = warp_sum(gq);
            if (lane == 0) {
              double* dst = e.gn_sum + ((long long)b * e.gn_groups + ((n0 + cb * 32) >> 5)) * 2;
              atomicAdd(dst, (double)gs);
              atomicAdd(dst + 1, (double)gq);
            }
          }
        } else {
          scalar_block(p, wstage, b, m0 + mb * BM + q * 32, n0 + cb * 32, lane);
        }
        __syncwarp();                // the transpose buffer may be overwritten by the next block
        if (ew == 0 && tile == (int)blockIdx.x && blk == slot) EV_TR(15);
      }
      if (ew == 0) { if (tile == (int)blockIdx.x) EV_TR(8); EV_TR(9); }
      if (slot >= n_blk) {           // a warp without a block in this tile still keeps step with the accumulator hand-over
        for (int grp = 0; grp < n_grp; ++grp) {
          const int v = ti + grp;
          mbar_wait(&acc_full[v & 1], (uint32_t)(v >> 1) & 1u);
          if (lane == 0) mbar_arrive(&acc_empty[v & 1]);
          __syncwarp();
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
    EV_TR(10);
  }
}

// ------------------------------------------------------------------------------------------------ host side
PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;
int g_halo_mode = -1;   // EV_TC_HALO=0 disables halo reuse (one activation tile per tap) for debugging

bool encode_map(CUtensorMap* map, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t s1_bytes,
                uint64_t s2_bytes, uint32_t b0, uint32_t b1, std::string* err, int swizzle_bytes = 128, bool f32 = false) {
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {s1_bytes, s2_bytes};
  cuuint32_t box[3] = {b0, b1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  const CUtensorMapSwizzle sw = swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B;
  CUresult r = g_encode(map, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    if (err) {
      char buf[256];
      snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled failed (%d): dims %llu,%llu,%llu strides %llu,%llu box %u,%u",
               (int)r, (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2,
               (unsigned long long)s1_bytes, (unsigned long long)s2_bytes, b0, b1);
      *err = buf;
    }
    return false;
  }
  return true;
}

thread_local int g_sm_count = 0;     // SM count of the device of the launch being planned (refreshed per launch, see sm_count_now)
int g_sm_by_dev[64] = {};
int sm_count_now() {    // per-device (a process may drive several GPUs), cached after the first query
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  int& c = g_sm_by_dev[dev & 63];
  if (c <= 0) { int v = 0; cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev); c = v > 0 ? v : 148; }
  return c;
}
int g_resident_mode = 1;   // EV_TC_RESIDENT=0 disables the weights-resident variant (debugging)
int g_mb_mode = 0;         // EV_TC_MB=1|2 forces the m-blocks per tile (0 = heuristic)
int g_bk32_mode = 1;       // EV_TC_BK32=0 disables the 64-byte-swizzle path for C_in <= 32
int g_cta2_mode = 1;       // EV_TC_CTA2=0 keeps one CTA per SM
int g_wide_mode = 1;       // EV_TC_WIDE=0 keeps 8 epilogue warps
int g_lean_mode = 1;       // EV_TC_LEAN=0 disables the activation-only epilogue path
int g_min_b2 = 4;          // EV_TC_MINB2: fewest weight-ring slots accepted for the two-CTAs-per-SM configuration
int g_tf32_share = 1;      // EV_TF32_SHARE=0: every one of the three products loads its own operand tiles
int g_tf32_flush = 1;      // EV_TF32_FLUSH=0: 3xTF32 without two-level accumulation (shows the tensor core's truncation error)

// Shared-memory plan of one launch for `k` CTAs per SM with `epi_warps` epilogue warps; false when the rings do not fit.
// resident: -1 = EV_TC_RESIDENT and the tile-count heuristic; 0 / 1 = streamed / resident weights (1: false when they cannot stay)
template <int BN>
bool plan_smem(TcParams& p, int k, int epi_warps, int* smem_out, int resident) {
  const int staging = epi_warps * STAGING_WARP_BYTES;
  const int per_cta = std::min(SMEM_LIMIT, (228 * 1024) / k - 2048);   // 1 KiB driver reserve + static barriers per CTA
  const int budget = per_cta - 1024 - staging;
  const int w_tiles = p.kchunks * p.g.taps;
  int a_slots, b_slots;
  // resident weights need one n-tile (the producer loads them at n0 = 0) and room beside two activation slots; enough tiles to
  // amortise the up-front load is a preference only, which a forced choice skips
  const bool want = resident >= 0 ? resident != 0 : (g_resident_mode != 0 && p.total_tiles >= 2 * k * g_sm_count);
  p.resident = want && p.n_tiles == 1 && (w_tiles * p.b_tile_bytes + 2 * p.a_slot_bytes <= budget);
  if (resident == 1 && !p.resident) return false;
  if (p.resident) {
    b_slots = w_tiles;
    a_slots = std::min(MAX_A_SLOTS, (budget - w_tiles * p.b_tile_bytes) / p.a_slot_bytes);
  } else {
    a_slots = p.a_slot_bytes <= 24 * 1024 ? 3 : 2;
    b_slots = (budget - a_slots * p.a_slot_bytes) / p.b_tile_bytes;
    if (b_slots < 4 && a_slots == 3) { a_slots = 2; b_slots = (budget - a_slots * p.a_slot_bytes) / p.b_tile_bytes; }
    if (b_slots > MAX_B_SLOTS) b_slots = MAX_B_SLOTS;
    { static const int cap = []() { const char* v = getenv("EV_TC_MAXB"); return v ? atoi(v) : 0; }(); if (cap > 0 && b_slots > cap) b_slots = cap; }   // timing experiments
    if (b_slots < (k > 1 ? g_min_b2 : 3)) return false;
  }
  if (a_slots < 2) return false;
  p.a_slots = a_slots;
  p.b_slots = b_slots;
  *smem_out = 1024 + a_slots * p.a_slot_bytes + b_slots * p.b_tile_bytes + staging;
  return true;
}

cudaError_t refuse(std::string* err, const char* why) {
  if (err) *err = std::string("conv_tc: forced schedule cannot run: ") + why;
  return cudaErrorInvalidValue;
}

template <int BN>
cudaError_t launch_bn(const CUtensorMap& tmA, const CUtensorMap& tmB, TcParams& p, cudaStream_t stream, RaggedPlanner* ragged,
                      const TcSchedule& sc, int split, TcLaunchInfo* info, std::string* err) {
  p.m_tiles = ceil_div(p.g.M, BM * p.mb);
  p.rag = (ragged && !p.tf32) ? ragged->table(BM * p.mb, p.g.M, stream) : nullptr;
  p.n_tiles = ceil_div(p.g.N, BN);
  p.total_tiles = p.m_tiles * p.n_tiles * p.g.B;
  p.div_n = ((1ull << 44) + (unsigned long long)p.n_tiles - 1) / (unsigned long long)p.n_tiles;
  p.div_m = ((1ull << 44) + (unsigned long long)p.m_tiles - 1) / (unsigned long long)p.m_tiles;
  if (p.total_tiles >= (1 << 22)) return cudaErrorInvalidConfiguration;
  uint32_t cols = 32;
  while (cols < (uint32_t)(2 * p.mb * BN)) cols <<= 1;
  p.tmem_cols = cols;
  const int k_tmem = 512 / (int)cols;
  // two CTAs per SM (8 epilogue warps each) when shared memory and TMEM allow and a tile has few 32-column blocks;
  // otherwise one CTA with 16 epilogue warps (the epilogue is issue-bound: more warps hide its dependent latencies)
  int k = 1, smem = 0, threads = NUM_THREADS_WIDE;
  bool ok = false;
  const bool flush = p.flush_kc < p.kchunks;
  if (flush && (BN != 128 || p.mb != 1)) return cudaErrorInvalidConfiguration;   // one block per epilogue warp
  if (sc.ctas_per_sm == 2 && sc.epi_warps == 16) return refuse(err, "two CTAs per SM run 8 epilogue warps each");
  // the EV_TC_CTA2 / EV_TC_WIDE switches, unless this call forces CTAs per SM or epilogue warps; a forced pair of CTAs skips
  // the "more tiles than SMs" preference as EV_TC_CTA2=2 does, never the TMEM and shared-memory conditions
  const bool two_on = sc.ctas_per_sm >= 0 ? sc.ctas_per_sm == 2
                                          : sc.epi_warps != 16 && g_cta2_mode && (p.total_tiles > g_sm_count || g_cta2_mode == 2);
  const bool wide_on = sc.epi_warps >= 0 ? sc.epi_warps == 16 : (g_wide_mode || flush);
  if (!flush && two_on && k_tmem >= 2 && p.mb * (BN / 32) <= 4 && plan_smem<BN>(p, 2, 8, &smem, sc.resident)) {
    k = 2; threads = NUM_THREADS; ok = true;
  }
  if (!ok && sc.ctas_per_sm != 2 && wide_on && plan_smem<BN>(p, 1, 16, &smem, sc.resident)) ok = true;
  if (!ok && sc.ctas_per_sm != 2 && sc.epi_warps != 16 && !flush && plan_smem<BN>(p, 1, 8, &smem, sc.resident)) {
    threads = NUM_THREADS; ok = true;
  }
  if (!ok) {
    if (sc.ctas_per_sm == 2) return refuse(err, "two CTAs per SM need 2*mb*BN <= 256 TMEM columns, no split flush and rings that fit");
    if (sc.epi_warps == 8 && flush) return refuse(err, "the two-level flush of the split paths needs 16 epilogue warps");
    if (sc.resident == 1) return refuse(err, "resident weights need one n-tile and a weight set that fits in shared memory");
    if (sc.epi_warps == 16) return refuse(err, "16 epilogue warps leave no room for the rings");
    return cudaErrorInvalidConfiguration;
  }
  // never let more CTAs become co-resident than TMEM can serve (tcgen05.alloc would spin forever)
  const int min_smem = (228 * 1024) / (k_tmem + 1) + 1;
  if (smem < min_smem && k_tmem < 8) smem = std::min(min_smem, SMEM_LIMIT);
  static DeviceOnce once;
  cudaError_t ce_attr = once.run([&]() { return cudaFuncSetAttribute(conv_tc_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT); });
  if (ce_attr != cudaSuccess) return ce_attr;
  p.n_issuers = threads == NUM_THREADS_WIDE ? 2 : 1;
  // the sharing walk needs one tap group (haloed tile or a 1x1 conv), streamed weights and room for a step's weight tiles
  if (p.tf32_share && (p.n_groups != 1 || p.resident || p.b_slots < p.g.taps + 1 || p.a_slots < 2 || p.kchunks % 3 != 0)) {
    if (sc.share == 1) return refuse(err, "operand sharing needs one tap group, streamed weights and a weight slot per tap and one more");
    p.tf32_share = 0;
  }
  const int grid = std::min(p.total_tiles, k * g_sm_count);
  if (info) {
    TcLaunchInfo& r = *info;
    r.bn = BN; r.mb = p.mb; r.ctas_per_sm = k; r.epi_warps = threads / 32 - 1 - p.n_issuers; r.issuers = p.n_issuers;
    r.resident = p.resident; r.a_slots = p.a_slots; r.b_slots = p.b_slots; r.bk = p.bk; r.halo = p.n_groups == 1 && p.g.taps > 1;
    r.a_boxes = p.a_boxes; r.act_only = p.act_only; r.vec_ok = p.vec_ok; r.split = split;
    r.flush_groups = (p.kchunks + p.flush_kc - 1) / p.flush_kc; r.tf32_share = p.tf32_share; r.ragged = p.rag != nullptr;
    r.grid = grid; r.total_tiles = p.total_tiles;
  }
  return launch_pdl(conv_tc_kernel<BN>, dim3(grid), dim3(threads), (size_t)smem, stream, tmA, tmB, p);
}

}  // namespace

bool tc_encode_bf16_map(::CUtensorMap_st* map, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t s1_bytes,
                        uint64_t s2_bytes, uint32_t b0, uint32_t b1, int swizzle_bytes, std::string* err) {
  if (!g_encode && !conv_tc_init(err)) return false;
  return encode_map(map, base, d0, d1, d2, s1_bytes, s2_bytes, b0, b1, err, swizzle_bytes);
}
int tc_sm_count() { return sm_count_now(); }
cudaError_t conv_tc_read_trace(unsigned long long* host, int n) {
  return cudaMemcpyFromSymbol(host, g_trace, sizeof(unsigned long long) * std::min(n, 512 * 24));
}

int conv_tc_pick_bn(int N) {
  if (N % 128 == 0) return 128;
  if (N <= 32) return 32;
  if (N <= 64) return 64;
  return 128;
}

bool conv_tc_init(std::string* err) {
  if (g_encode) return true;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  cudaError_t ce = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
  if (ce != cudaSuccess || q != cudaDriverEntryPointSuccess || fn == nullptr) {
    if (err) *err = std::string("cuTensorMapEncodeTiled entry point unavailable: ") + cudaGetErrorString(ce);
    return false;
  }
  g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
  g_sm_count = sm_count_now();
  return true;
}

// x: channel-last bf16 activations (b, t, c) at x + b*x_bs + t*x_ld + c, `x_rows` addressable rows per item.
cudaError_t conv_tc_launch(const ConvGeom& g, const void* x, long long x_ld, long long x_bs, int tf32x3,
                           const ConvWeights& w, const Epilogue& e, cudaStream_t stream, std::string* err, RaggedPlanner* ragged,
                           const TcSchedule* sched, TcLaunchInfo* info) {
  if (!g_encode && !conv_tc_init(err)) return cudaErrorNotSupported;
  const TcSchedule sc = sched ? *sched : TcSchedule{};
  {
    auto flag = [](int v) { return v >= -1 && v <= 1; };
    if (!flag(sc.lean) || !flag(sc.resident) || !flag(sc.bk32) || !flag(sc.halo) || !flag(sc.share) || (sc.mb != -1 && sc.mb != 1 && sc.mb != 2) ||
        (sc.ctas_per_sm != -1 && sc.ctas_per_sm != 1 && sc.ctas_per_sm != 2) || (sc.epi_warps != -1 && sc.epi_warps != 8 && sc.epi_warps != 16))
      return refuse(err, "a value outside its choices");
    if (tf32x3 && sc.bk32 >= 0) return refuse(err, "the split paths have a fixed K-chunk width");
    if (tf32x3 && sc.mb == 2) return refuse(err, "the split paths run one m-block per tile (one 32 x 32 block per epilogue warp)");
    if (!tf32x3 && sc.share == 1) return refuse(err, "operand sharing is a walk of the split paths");
    if (sc.bk32 == 1 && g.C_in > 32) return refuse(err, "BK = 32 serves C_in <= 32 only");
  }
  const int esz = tf32x3 == 1 ? 4 : 2;
  if ((x_ld * esz & 15) || (x_bs * esz & 15) || (reinterpret_cast<uintptr_t>(x) & 15)) {
    if (err) *err = "conv_tc: activation tensor is not 16-byte aligned / strided";
    return cudaErrorInvalidValue;
  }
  if (g_halo_mode < 0) {
    auto env_int = [](const char* name, int dflt) { const char* v = getenv(name); return v ? atoi(v) : dflt; };
    g_resident_mode = env_int("EV_TC_RESIDENT", 1);
    g_mb_mode = env_int("EV_TC_MB", 0);
    g_bk32_mode = env_int("EV_TC_BK32", 1);
    g_cta2_mode = env_int("EV_TC_CTA2", 1);
    g_wide_mode = env_int("EV_TC_WIDE", 1);
    g_lean_mode = env_int("EV_TC_LEAN", 1);
    g_tf32_flush = env_int("EV_TF32_FLUSH", 1);
    g_tf32_share = env_int("EV_TF32_SHARE", 1);
    g_min_b2 = env_int("EV_TC_MINB2", 4);
    g_halo_mode = env_int("EV_TC_HALO", 1);
  }
  const int BN = conv_tc_pick_bn(g.N);
  g_sm_count = sm_count_now();
  TcParams p;
  p.g = g;
  p.e = e;
  // K-chunk width: 64 channels under the 128-byte swizzle, or 32 under the 64-byte swizzle when that avoids padded K
  p.tf32 = tf32x3 ? 1 : 0;
  p.mma_tf32 = tf32x3 == 1 ? 1 : 0;
  p.descale = nullptr;
  if (tf32x3 == 2) {      // 3xFP16: 64 halves per 128-byte row, UMMA K = 16; the same walk over [x_hi | x_hi | x_lo] x [w_hi | w_lo | w_hi]
    if (g.conv_stride != 1 || !w.w_f16x3 || !w.f16_scale || g.C_in % 64) { if (err) *err = "conv_tc: the 3xFP16 path needs stride 1, C_in % 64 == 0 and split weights"; return cudaErrorInvalidValue; }
    p.bk = 64;
    p.row_bytes = 128;
    p.ksteps = 4;
    p.kch1 = g.C_in / 64;
    p.kchunks = 3 * p.kch1;
    p.sec_off[0] = 0; p.sec_off[1] = 0; p.sec_off[2] = g.C_in;
    p.idesc = make_idesc(BM, BN) & ~((7u << 7) | (7u << 10));      // kind::f16 with F16 (format 0) operands instead of BF16
    p.flush_kc = std::max(1, 16 / (g.taps * p.ksteps));
    if (g_tf32_flush == 0) p.flush_kc = p.kchunks;
    p.tf32_share = sc.share >= 0 ? sc.share : g_tf32_share;
    p.descale = w.f16_scale;
  } else if (tf32x3) {      // 32 fp32 channels per 128-byte row, UMMA K = 8; K-chunks walk [x_hi | x_hi | x_lo] x [w_hi | w_lo | w_hi]
    if (g.conv_stride != 1 || !w.w_tf32) { if (err) *err = "conv_tc: the 3xTF32 path needs stride 1 and split weights"; return cudaErrorInvalidValue; }
    p.bk = 32;
    p.row_bytes = 128;
    p.ksteps = 4;
    p.kch1 = w.K32 / 32;
    p.kchunks = 3 * p.kch1;
    p.sec_off[0] = 0; p.sec_off[1] = 0; p.sec_off[2] = g.C_in;
    p.idesc = make_idesc_tf32(BM, BN);
    p.flush_kc = std::max(1, 16 / (g.taps * p.ksteps));    // <= 16 truncating tensor-core accumulations per partial sum
    if (g_tf32_flush == 0) p.flush_kc = p.kchunks;
    p.tf32_share = sc.share >= 0 ? sc.share : g_tf32_share;
  } else {
    p.tf32_share = 0;
    p.bk = ((sc.bk32 >= 0 ? sc.bk32 : g_bk32_mode) && g.C_in <= 32) ? 32 : 64;
    p.row_bytes = p.bk * 2;
    p.ksteps = p.bk / UMMA_K;
    p.kchunks = ceil_div(g.C_in, p.bk);
    p.kch1 = p.kchunks;
    p.sec_off[0] = p.sec_off[1] = p.sec_off[2] = 0;
    p.idesc = make_idesc(BM, BN);
    p.flush_kc = p.kchunks;
  }
  p.desc_sbo = 8u * (uint32_t)p.row_bytes;
  p.desc_layout = p.row_bytes == 128 ? 2u : 4u;
  p.b_tile_bytes = BN * p.row_bytes;
  int tap_row[kMaxTaps], tap_col[kMaxTaps];
  CUtensorMap tmA, tmB;
  uint64_t d0, d1, s1;
  if (g.conv_stride == 1) {
    for (int j = 0; j < g.taps; ++j) { tap_row[j] = g.tap_off[j]; tap_col[j] = 0; }
    d0 = (uint64_t)(tf32x3 ? 2 * g.C_in : g.C_in); d1 = (uint64_t)g.T_in; s1 = (uint64_t)x_ld * esz;
  } else if (g.conv_stride == 2) {
    // (T, ld) viewed as (T/2, 2*ld): time 2j+h is row j, columns [h*ld, h*ld + C_in)
    if (g.T_in & 1) { if (err) *err = "conv_tc: stride-2 conv needs an even input length"; return cudaErrorInvalidValue; }
    for (int j = 0; j < g.taps; ++j) {
      const int off = g.tap_off[j];
      const int h = ((off % 2) + 2) % 2;
      tap_row[j] = (off - h) / 2;
      tap_col[j] = h * (int)x_ld;
    }
    d0 = (uint64_t)(x_ld + g.C_in); d1 = (uint64_t)(g.T_in / 2); s1 = (uint64_t)x_ld * 4;
  } else {
    if (err) *err = "conv_tc: unsupported stride";
    return cudaErrorInvalidValue;
  }
  // m-blocks per tile: two accumulators share every weight tile unless that costs a whole extra round of tiles
  {
    auto cost = [&](int mb) {
      const long long tiles = (long long)ceil_div(g.M, BM * mb) * ceil_div(g.N, BN) * g.B;
      const long long rounds = (tiles + g_sm_count - 1) / g_sm_count;
      return (double)rounds * (mb + 0.3);
    };
    p.mb = (g.M > BM && cost(2) <= cost(1)) ? 2 : 1;
    if (g_mb_mode == 1 || g_mb_mode == 2) p.mb = g_mb_mode;
    if (sc.mb > 0) p.mb = sc.mb;
    if (tf32x3) p.mb = 1;            // two-level accumulation: one 32 x 32 block per epilogue warp (16 warps, 128 x 128 tile)
    if (p.mb > MB_MAX) p.mb = MB_MAX;
  }
  // halo reuse: all taps read one tile when they share the column origin and the row span fits two TMA boxes
  int lo = tap_row[0], hi = tap_row[0];
  bool same_col = true;
  for (int j = 1; j < g.taps; ++j) { lo = std::min(lo, tap_row[j]); hi = std::max(hi, tap_row[j]); same_col &= tap_col[j] == tap_col[0]; }
  const bool halo_ok = g.taps > 1 && same_col && (hi - lo) <= 128;
  if (sc.halo == 1 && !halo_ok) return refuse(err, "halo reuse needs several taps that read the same columns within 128 rows");
  const bool halo = (sc.halo >= 0 ? sc.halo != 0 : g_halo_mode != 0) && halo_ok;
  int a_rows;
  if (halo) {
    p.n_groups = 1;
    p.grp_row0[0] = lo; p.grp_col0[0] = tap_col[0]; p.grp_first[0] = 0; p.grp_count[0] = g.taps;
    for (int j = 0; j < g.taps; ++j) p.tap_byte_off[j] = (tap_row[j] - lo) * p.row_bytes;
    a_rows = p.mb * BM + hi - lo;
    p.grp_taps = g.taps;
    p.tap_first16 = (uint32_t)p.tap_byte_off[0] >> 4;
    p.tap_step16 = (uint32_t)(((tap_row[1] - tap_row[0]) * p.row_bytes) / 16);
    for (int j = 1; j < g.taps; ++j)
      if (tap_row[j] - tap_row[j - 1] != tap_row[1] - tap_row[0]) { if (err) *err = "conv_tc: taps must be equally spaced"; return cudaErrorInvalidValue; }
  } else {
    p.n_groups = g.taps;
    for (int j = 0; j < g.taps; ++j) {
      p.grp_row0[j] = tap_row[j]; p.grp_col0[j] = tap_col[j]; p.grp_first[j] = j; p.grp_count[j] = 1; p.tap_byte_off[j] = 0;
    }
    a_rows = p.mb * BM;
    p.grp_taps = 1;
    p.tap_first16 = 0;
    p.tap_step16 = 0;
  }
  p.a_boxes = a_rows > 256 ? 2 : 1;
  p.a_box_rows = (int)align_up((size_t)ceil_div(a_rows, p.a_boxes), 8);
  p.a_slot_bytes = (int)align_up((size_t)p.a_boxes * p.a_box_rows * p.row_bytes, 1024);
  bool ok = encode_map(&tmA, x, d0, d1, (uint64_t)g.B, s1, (uint64_t)x_bs * esz, (uint32_t)p.bk, (uint32_t)p.a_box_rows, err, p.row_bytes, tf32x3 == 1);
  if (!ok) return cudaErrorInvalidValue;
  if (tf32x3 == 2) {
    if (w.N_pad_tc % BN != 0) { if (err) *err = "conv_tc: split weight padding does not match the tile shape"; return cudaErrorInvalidValue; }
    const uint64_t k3 = 3ull * (uint64_t)g.C_in;
    ok = encode_map(&tmB, w.w_f16x3, k3, (uint64_t)w.N_pad_tc, (uint64_t)w.taps, k3 * 2, k3 * w.N_pad_tc * 2, 64u, (uint32_t)BN, err, 128, false);
  } else if (tf32x3) {
    if (w.N_pad_tc % BN != 0 || w.K32 % 32 != 0) { if (err) *err = "conv_tc: split weight padding does not match the tile shape"; return cudaErrorInvalidValue; }
    const uint64_t k3 = 3ull * w.K32;
    ok = encode_map(&tmB, w.w_tf32, k3, (uint64_t)w.N_pad_tc, (uint64_t)w.taps, k3 * 4, k3 * w.N_pad_tc * 4, 32u, (uint32_t)BN, err, 128, true);
  } else {
    if (w.N_pad_tc % BN != 0 || w.K_pad % 64 != 0 || w.K_pad < p.kchunks * p.bk) {
      if (err) *err = "conv_tc: packed weight padding does not match the tile shape";
      return cudaErrorInvalidValue;
    }
    ok = encode_map(&tmB, w.w_bf16, (uint64_t)w.K_pad, (uint64_t)w.N_pad_tc, (uint64_t)w.taps, (uint64_t)w.K_pad * 2,
                    (uint64_t)w.K_pad * w.N_pad_tc * 2, (uint32_t)p.bk, (uint32_t)BN, err, p.row_bytes);
  }
  if (!ok) return cudaErrorInvalidValue;
  if (tf32x3 && e.out_act) { if (err) *err = "conv_tc: the split-operand paths write fp32 outputs only"; return cudaErrorInvalidValue; }
  if (e.act != ACT_NONE && e.act != ACT_RELU && e.act != ACT_LRELU && e.act != ACT_SNAKE) {
    if (err) *err = "conv_tc: the tensor-core epilogue implements identity / (leaky) ReLU / SnakeBeta only";
    return cudaErrorInvalidValue;
  }
  auto al4 = [](long long v) { return (v & 3) == 0; };
  p.vec_ok = (e.phase_cout % 4 == 0) && (g.N % 4 == 0) && al4(e.res_ld) && al4(e.res_bs) && al4(e.res2_ld) && al4(e.res2_bs) &&
             al4(e.f32_ld) && al4(e.f32_bs) && al4(e.act_ld) && al4(e.act_bs) &&
             ((reinterpret_cast<uintptr_t>(e.res) | reinterpret_cast<uintptr_t>(e.res2) |
               reinterpret_cast<uintptr_t>(e.out_f32) | reinterpret_cast<uintptr_t>(e.bias)) & 15) == 0 &&
             (reinterpret_cast<uintptr_t>(e.out_act) & 7) == 0;
  const bool lean_ok = p.vec_ok && e.out_act && !e.out_f32 && !e.res && !e.res2 && e.alpha == 1.0f && e.div == 1.0f &&
                       !e.mask_pre && e.phase_cout == g.N && g.N % 32 == 0 && (e.act_ld % 8) == 0 && (e.act_bs % 8) == 0 &&
                       (reinterpret_cast<uintptr_t>(e.out_act) & 15) == 0;
  if (sc.lean == 1 && !lean_ok) return refuse(err, "the lean epilogue serves a bf16-only output of an ordinary conv with N % 32 == 0 and aligned rows");
  p.act_only = (sc.lean >= 0 ? sc.lean != 0 : g_lean_mode != 0) && lean_ok;
  if (e.gn_sum && (!p.vec_ok || !e.out_f32 || e.phase_cout != g.N || g.N % 32 != 0 || g.N / 32 != e.gn_groups)) {
    if (err) *err = "conv_tc: fused GroupNorm statistics need 32 channels per group on the vector path";
    return cudaErrorInvalidValue;
  }
  { static const int nob = []() { const char* v = getenv("EV_TC_DEBUG_NOB"); return v ? atoi(v) : 0; }(); p.debug_nob = nob; }
  { static const int ia = []() { const char* v = getenv("EV_TC_IDLE_ARRIVE"); return v ? atoi(v) : 1; }(); p.idle_arrive = ia; }
  { static const int tr = []() { const char* v = getenv("EV_TC_TRACE"); return v ? atoi(v) : 0; }(); p.trace = tr; }
  switch (BN) {
    case 32: return launch_bn<32>(tmA, tmB, p, stream, ragged, sc, tf32x3, info, err);
    case 64: return launch_bn<64>(tmA, tmB, p, stream, ragged, sc, tf32x3, info, err);
    default: return launch_bn<128>(tmA, tmB, p, stream, ragged, sc, tf32x3, info, err);
  }
}

}  // namespace ev
