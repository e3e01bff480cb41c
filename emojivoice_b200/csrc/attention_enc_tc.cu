// Text-encoder MultiHeadAttention (text_encoder.py:223-246) on tcgen05 tensor cores at fp32 accuracy.
//
// The duration predictor sits behind this attention and durations must match the reference exactly, so bf16 / tf32 products
// are not an option.  Every operand is therefore split into two fp16 halves of a power-of-two multiple (v * 2^s = hi + lo,
// hi = fp16(v 2^s), lo = fp16(v 2^s - hi): 22 mantissa bits) and every product runs as three kind::f16 MMAs
// (hi hi + hi lo + lo hi) accumulated in fp32 in TMEM -- the same 3xFP16 scheme as the encoder convolutions (weights.cu).
//
// One CTA = 128 queries of one (utterance, head), head width HD = 96 or 128, any number of keys, in blocks of 64 (flash-attention order):
//   stage     q (once) and each k block are read as fp32, rotated (RoPE on the first rope_dim features, rotate-half pairing,
//             text_encoder.py:147-169), split and written as 128B-swizzled K-major fp16 tiles; v goes in split but in its natural
//             [key][feature] layout and is consumed MN-major.  The next block's global loads sit in registers meanwhile.
//   scores    S = Q K^T of the block by tcgen05 into TMEM.  The tensor core TRUNCATES on every accumulation into TMEM (the
//             encoder convs flush into fp32 masters for the same reason), so the full-magnitude hi hi products of the two
//             feature chunks (0-63 and 64..HD-1) go to two accumulators (at most four accumulations each) and are added with a
//             rounded fp32 add.
//   softmax   thread = (query row, half of the block's columns): running maximum (the halves meet through shared memory),
//             p = exp(s - m) with the reference's -1e4 fill where the query OR the key is padded; P is split like the rest.
//   output    O_blk = P V into a FRESH TMEM accumulator per block; the running output lives in registers (HD / 2 per thread)
//             and takes o = o * corr + O_blk with rounded adds.
// HD = 96 (single-speaker models: 192 channels, 2 heads) keeps the tile layout of HD = 128: feature chunk 1 holds features 64-95
// in the first half of each 128-byte row, its score MMAs stop after two K = 16 steps and never read the other half, and the
// P V MMA of chunk 1 stays N = 64 over V columns that are zero beyond feature 95 (those output columns are never read).
// Other head widths stay on the fp32 CUDA-core kernel (attention.cu).
#include "kernels.cuh"
#include "tc_ptx.cuh"

namespace ev {
using namespace tc;

namespace {

constexpr int BQ = 128, BK = 64, THREADS = 256;
constexpr int TILE_Q = BQ * 128, TILE_K = BK * 128; // one 64-feature chunk of Q (16 KB) / of a key block (8 KB); a P half is a TILE_Q
constexpr int Q_BYTES = 4 * TILE_Q;                 // [hi c0 | hi c1 | lo c0 | lo c1]
constexpr int BLK_BYTES = 4 * TILE_K;               // a K or V block [hi c0 | hi c1 | lo c0 | lo c1], and the P block [hi | lo]
constexpr int SMEM_BYTES = 1024 + Q_BYTES + 3 * BLK_BYTES;
constexpr uint32_t TMEM_COLS = 256, S_A = 0, S_B = 64, O_COL = 128;
constexpr float kOpScale = kF16ActScale;            // q, k, v are split as halves of x * 8 (as the conv activations are)
constexpr float kPScale = 4096.0f;                  // p in [0, 1] is split as halves of p * 4096

template <int HD>
struct Geo {
  static_assert(HD == 96 || HD == 128, "head width");
  static constexpr int ROPE = HD / 2, RHALF = HD / 4;                 // rotary width = half a head (text_encoder.py:203-204)
  static constexpr int ROT = RHALF / 8, PLAIN = (HD - ROPE) / 8;     // rotated / plain items of 8 features per row
  static constexpr int NPL = (64 * PLAIN + THREADS - 1) / THREADS;   // plain items per thread in 64 rows
  static constexpr bool FULL_ROT = 64 * ROT % THREADS == 0, FULL_PL = 64 * PLAIN % THREADS == 0;
  static constexpr int KS1 = (HD - 64) / 16;                         // K = 16 steps of feature chunk 1
  static_assert(64 * ROT <= THREADS, "one rotated item per thread");
};

// One thread's share of a 64-row x HD-feature q / k tile: at most one ROTATED item (features [8i, 8i+8) and their partners
// [HD/4+8i, HD/4+8i+8) with the cos / sin of the row) and at most two PLAIN items (8 of the features HD/2..HD-1 each).
// HD = 128: 4 rotated + 8 plain items per row, every thread holds three; HD = 96: 3 + 6 per row, warps 6-7 hold no rotated
// item and warps 4-7 one plain item.  Item kinds are uniform across a warp, so neither the loads nor the conversions diverge.
struct Regs12 { float4 a, b, c, d, cs0, cs1, sn0, sn1, pa[2], pb[2]; };
template <int N> struct RegsV { float4 a[N], b[N]; };                    // the work items of a V block

__device__ __forceinline__ void split8(const float4& x, const float4& y, float scale, uint4* hi, uint4* lo) {
  const float v[8] = {x.x * scale, x.y * scale, x.z * scale, x.w * scale, y.x * scale, y.y * scale, y.z * scale, y.w * scale};
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const __half h0 = __float2half_rn(v[2 * i]), h1 = __float2half_rn(v[2 * i + 1]);
    const __half2 hh = __halves2half2(h0, h1);
    const __half2 ll = __floats2half2_rn(v[2 * i] - __half2float(h0), v[2 * i + 1] - __half2float(h1));
    h[i] = *reinterpret_cast<const uint32_t*>(&hh);
    l[i] = *reinterpret_cast<const uint32_t*>(&ll);
  }
  *hi = make_uint4(h[0], h[1], h[2], h[3]);
  *lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// 64 rows x HD features of q or k: rotated item idx = threadIdx.x, plain item idx = threadIdx.x + it * THREADS
template <int HD>
__device__ __forceinline__ void load_rows(const float* base, long long ld, int t0, int T, const float* rc, const float* rs, Regs12& r) {
  using G = Geo<HD>;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  {
    const unsigned idx = threadIdx.x;
    const int row = idx / G::ROT, i = idx % G::ROT, t = t0 + row;
    r.a = r.b = r.c = r.d = r.sn0 = r.sn1 = z;
    r.cs0 = r.cs1 = make_float4(1.f, 1.f, 1.f, 1.f);
    if ((G::FULL_ROT || idx < 64 * G::ROT) && t < T) {
      const float* p = base + (long long)t * ld + 8 * i;
      r.a = *reinterpret_cast<const float4*>(p); r.b = *reinterpret_cast<const float4*>(p + 4);
      r.c = *reinterpret_cast<const float4*>(p + G::RHALF); r.d = *reinterpret_cast<const float4*>(p + G::RHALF + 4);
      r.cs0 = *reinterpret_cast<const float4*>(rc + t * G::RHALF + 8 * i); r.cs1 = *reinterpret_cast<const float4*>(rc + t * G::RHALF + 8 * i + 4);
      r.sn0 = *reinterpret_cast<const float4*>(rs + t * G::RHALF + 8 * i); r.sn1 = *reinterpret_cast<const float4*>(rs + t * G::RHALF + 8 * i + 4);
    }
  }
#pragma unroll
  for (int it = 0; it < G::NPL; ++it) {
    const unsigned idx = threadIdx.x + it * THREADS;
    const int row = idx / G::PLAIN, i = idx % G::PLAIN, t = t0 + row;
    r.pa[it] = r.pb[it] = z;
    if ((G::FULL_PL || idx < 64 * G::PLAIN) && t < T) {
      const float* p = base + (long long)t * ld + G::ROPE + 8 * i;
      r.pa[it] = *reinterpret_cast<const float4*>(p); r.pb[it] = *reinterpret_cast<const float4*>(p + 4);
    }
  }
}

// out[d] = x[d] cos - x[d + half] sin, out[d + half] = x[d + half] cos + x[d] sin  (text_encoder.py:147-169)
__device__ __forceinline__ float4 rot_lo(const float4& x, const float4& y, const float4& c, const float4& s) {
  return make_float4(x.x * c.x + (-y.x) * s.x, x.y * c.y + (-y.y) * s.y, x.z * c.z + (-y.z) * s.z, x.w * c.w + (-y.w) * s.w);
}
__device__ __forceinline__ float4 rot_hi(const float4& x, const float4& y, const float4& c, const float4& s) {
  return make_float4(y.x * c.x + x.x * s.x, y.y * c.y + x.y * s.y, y.z * c.z + x.z * s.z, y.w * c.w + x.w * s.w);
}

// Rotate, split and store the rows loaded by load_rows as K-major 128B-swizzled fp16 tiles: `dst` = hi half of feature chunk 0,
// chunk 1 `chunk` bytes further, lo halves `lo_off` bytes after the hi halves; `row0` = first tile row of these 64 rows.
// Features HD..127 of chunk 1 are never written (HD = 96): no MMA reads them.
template <int HD>
__device__ __forceinline__ void store_rows(const Regs12& r, uint8_t* dst, int chunk, int lo_off, int row0) {
  using G = Geo<HD>;
  uint4 hi, lo;
  {
    const unsigned idx = threadIdx.x;
    if (G::FULL_ROT || idx < 64 * G::ROT) {
      const int row = row0 + idx / G::ROT, i = idx % G::ROT;
      uint8_t* prow = dst + row * 128;
      split8(rot_lo(r.a, r.c, r.cs0, r.sn0), rot_lo(r.b, r.d, r.cs1, r.sn1), kOpScale, &hi, &lo);
      int off = (i ^ (row & 7)) * 16;
      *reinterpret_cast<uint4*>(prow + off) = hi; *reinterpret_cast<uint4*>(prow + lo_off + off) = lo;
      split8(rot_hi(r.a, r.c, r.cs0, r.sn0), rot_hi(r.b, r.d, r.cs1, r.sn1), kOpScale, &hi, &lo);
      off = ((G::ROT + i) ^ (row & 7)) * 16;
      *reinterpret_cast<uint4*>(prow + off) = hi; *reinterpret_cast<uint4*>(prow + lo_off + off) = lo;
    }
  }
#pragma unroll
  for (int it = 0; it < G::NPL; ++it) {
    const unsigned idx = threadIdx.x + it * THREADS;
    if (G::FULL_PL || idx < 64 * G::PLAIN) {
      const int row = row0 + idx / G::PLAIN, i = idx % G::PLAIN;
      const int c = G::ROPE / 8 + i;        // 16-byte feature group of the head: tile c / 8, group c % 8 of the tile's row
      split8(r.pa[it], r.pb[it], kOpScale, &hi, &lo);
      const int off = (c >> 3) * chunk + row * 128 + ((c & 7) ^ (row & 7)) * 16;
      *reinterpret_cast<uint4*>(dst + off) = hi; *reinterpret_cast<uint4*>(dst + lo_off + off) = lo;
    }
  }
}

// 64 keys x HD features of v: HD / 8 items of 8 features per row, HD / 32 per thread; natural [key][feature] layout
template <int HD>
__device__ __forceinline__ void load_v(const float* base, long long ld, int t0, int T, RegsV<HD / 32>& r) {
#pragma unroll
  for (int it = 0; it < HD / 32; ++it) {
    const unsigned idx = threadIdx.x + it * THREADS;
    const int row = idx / (HD / 8), i = idx % (HD / 8), t = t0 + row;
    r.a[it] = r.b[it] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t < T) {
      const float* p = base + (long long)t * ld + 8 * i;
      r.a[it] = *reinterpret_cast<const float4*>(p); r.b[it] = *reinterpret_cast<const float4*>(p + 4);
    }
  }
}
template <int HD>
__device__ __forceinline__ void store_v(const RegsV<HD / 32>& r, uint8_t* dst) {
#pragma unroll
  for (int it = 0; it < HD / 32; ++it) {
    const unsigned idx = threadIdx.x + it * THREADS;
    const int row = idx / (HD / 8), i = idx % (HD / 8);
    uint4 hi, lo;
    split8(r.a[it], r.b[it], kOpScale, &hi, &lo);
    const int off = (i >> 3) * TILE_K + row * 128 + (((i & 7) ^ (row & 7)) * 16);
    *reinterpret_cast<uint4*>(dst + off) = hi; *reinterpret_cast<uint4*>(dst + 2 * TILE_K + off) = lo;
  }
}

struct Params {
  const float* q; const float* k; const float* v; long long ld, bs;
  int T, n_kb;
  float c1;                        // scale / (kOpScale * kOpScale): TMEM score -> reference logit
  const int* lens; int len_shift;
  const float* rope_cos; const float* rope_sin;
  float* out; long long out_ld, out_bs;
  __half* split; int split_ld;     // optional pre-split copy of the output for the out-projection conv (AttnArgs::split)
  int trace;                       // EV_ENC_ATTN_TRACE=1: CTA (0,0,0) prints clock stamps of its milestones (timing experiments)
};

template <int HD>
__global__ void __launch_bounds__(THREADS, 1) attn_enc_tc_kernel(const Params p) {
  using G = Geo<HD>;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t s_ready, o_ready;
  __shared__ uint32_t tmem_base_smem;
  __shared__ float red_sh[2][BQ];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t q_s = base, k_s = q_s + Q_BYTES, v_s = k_s + BLK_BYTES, p_s = v_s + BLK_BYTES;
  uint8_t* q_gen = gen; uint8_t* k_gen = q_gen + Q_BYTES; uint8_t* v_gen = k_gen + BLK_BYTES; uint8_t* p_gen = v_gen + BLK_BYTES;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * BQ;
  const int n_kb = p.n_kb;

  if (threadIdx.x == 0) {
    mbar_init(&s_ready, 1); mbar_init(&o_ready, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_base_smem;
  long long stamp[32];
  int n_stamp = 0;
  const bool tracer = p.trace && threadIdx.x == 0 && (blockIdx.x | blockIdx.y | blockIdx.z) == 0;
#define EV_STAMP() do { if (tracer && n_stamp < 32) stamp[n_stamp++] = clock64(); } while (0)
  EV_STAMP();
  pdl_trigger();
  pdl_wait();
  EV_STAMP();

  const float* qb = p.q + b * p.bs + h * HD;
  const float* kb_ = p.k + b * p.bs + h * HD;
  const float* vb = p.v + b * p.bs + h * HD;
  constexpr uint32_t idesc_s = make_idesc(BQ, BK, 0, 0) & ~((7u << 7) | (7u << 10));   // fp16 operands, both K-major
  constexpr uint32_t idesc_o = make_idesc(BQ, 64, 0, 1) & ~((7u << 7) | (7u << 10));   // V is MN-major (rows = keys)

  // thread = (query row, half): half of a key block's 64 score columns, and the same half of the HD output features
  const int quarter = warp & 3, hf = warp >> 2, row = quarter * 32 + lane, t = q0 + row;
  const int len = p.lens ? __ldg(p.lens + b) : 0x7fffffff;
  const bool qvalid = (t << p.len_shift) < len;
  const uint32_t lane_addr = tmem_base + ((uint32_t)(quarter * 32) << 16);

  Regs12 rk;
  {
    Regs12 r1;
    load_rows<HD>(qb, p.ld, q0, p.T, p.rope_cos, p.rope_sin, rk);
    load_rows<HD>(qb, p.ld, q0 + 64, p.T, p.rope_cos, p.rope_sin, r1);
    store_rows<HD>(rk, q_gen, TILE_Q, 2 * TILE_Q, 0);
    load_rows<HD>(kb_, p.ld, 0, p.T, p.rope_cos, p.rope_sin, rk);
    store_rows<HD>(r1, q_gen, TILE_Q, 2 * TILE_Q, 64);
  }
  if constexpr (HD < 128) {   // V columns HD..127 of feature chunk 1 (hi and lo) stay zero: store_v never writes them
    uint4* v1 = reinterpret_cast<uint4*>(v_gen + TILE_K);
#pragma unroll
    for (int it = 0; it < TILE_K / 8 / THREADS; ++it) {
      const int i = threadIdx.x + it * THREADS;
      v1[(i / (TILE_K / 16)) * (2 * TILE_K / 16) + i % (TILE_K / 16)] = make_uint4(0u, 0u, 0u, 0u);
    }
  }
  EV_STAMP();
  constexpr int NO = HD / 2;                              // running outputs per thread
  float o[NO];
#pragma unroll
  for (int i = 0; i < NO; ++i) o[i] = 0.0f;
  float m = -INFINITY, l = 0.0f;

  for (int kb = 0; kb < n_kb; ++kb) {
    const uint32_t par = (uint32_t)kb & 1u;
    // every MMA of the previous block has completed (o_ready was awaited): the K, V and P tiles are free
    store_rows<HD>(rk, k_gen, TILE_K, 2 * TILE_K, 0);
    fence_proxy_async();
    __syncthreads();
    if (warp == 0) {
      tcgen05_fence_after();
      if (elect_one()) {
        // The tensor core TRUNCATES when it adds into a TMEM accumulator, so the number of full-magnitude accumulations per
        // accumulator is kept at four: A = the small cross-term MMAs first (16; 12 at HD = 96), then hi hi of feature chunk 0;
        // B = hi hi of chunk 1.  Chunk 1 takes KS1 K = 16 steps (4; 2 at HD = 96: features 64-95).
        uint32_t acc = 0;
#pragma unroll
        for (int term = 1; term < 3; ++term) {            // hi lo, lo hi
          const uint32_t qa = q_s + (term == 2 ? 2u * TILE_Q : 0u), ka = k_s + (term == 1 ? 2u * TILE_K : 0u);
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            const uint64_t dq = make_smem_desc(qa + (uint32_t)(c * TILE_Q)), dk = make_smem_desc(ka + (uint32_t)(c * TILE_K));
#pragma unroll
            for (int k = 0; k < (c ? G::KS1 : 4); ++k) { umma_bf16(tmem_base + S_A, dq + (uint64_t)(2 * k), dk + (uint64_t)(2 * k), idesc_s, acc); acc = 1; }
          }
        }
#pragma unroll
        for (int c = 0; c < 2; ++c) {                     // hi hi
          const uint64_t dq = make_smem_desc(q_s + (uint32_t)(c * TILE_Q)), dk = make_smem_desc(k_s + (uint32_t)(c * TILE_K));
#pragma unroll
          for (int k = 0; k < (c ? G::KS1 : 4); ++k)
            umma_bf16(tmem_base + (c ? S_B : S_A), dq + (uint64_t)(2 * k), dk + (uint64_t)(2 * k), idesc_s, (c == 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(&s_ready);
      }
      __syncwarp();
    }
    RegsV<HD / 32> rv;
    load_v<HD>(vb, p.ld, kb * BK, p.T, rv);                   // in flight under the score MMAs
    EV_STAMP();
    mbar_wait(&s_ready, par);
    EV_STAMP();
    tcgen05_fence_after();
    float sc[32];
    {
      uint32_t raw[32];
      tmem_ld32(lane_addr + S_A + (uint32_t)(hf * 32), raw);
#pragma unroll
      for (int c = 0; c < 32; ++c) sc[c] = __uint_as_float(raw[c]);
      tmem_ld32(lane_addr + S_B + (uint32_t)(hf * 32), raw);
      const int k0 = kb * BK + hf * 32;
      float mx = -INFINITY;
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        const int tk = k0 + c;
        const float sv = (sc[c] + __uint_as_float(raw[c])) * p.c1;
        sc[c] = tk < p.T ? ((qvalid && (tk << p.len_shift) < len) ? sv : -1e4f) : -INFINITY;     // text_encoder.py:241
        mx = fmaxf(mx, sc[c]);
      }
      red_sh[hf][row] = mx;
      __syncthreads();
      mx = fmaxf(mx, red_sh[hf ^ 1][row]);               // every block holds at least one key of the sequence: finite
      const float m_new = fmaxf(m, mx), corr = expf(m - m_new);
      m = m_new;
      l *= corr;
#pragma unroll
      for (int i = 0; i < NO; ++i) o[i] *= corr;
    }
    store_v<HD>(rv, v_gen);
    {
      uint8_t* prow = p_gen + row * 128;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float pv[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) { pv[e] = expf(sc[8 * i + e] - m); l += pv[e]; }       // exp(-inf) = 0 beyond the sequence
        uint4 hi, lo;
        split8(make_float4(pv[0], pv[1], pv[2], pv[3]), make_float4(pv[4], pv[5], pv[6], pv[7]), kPScale, &hi, &lo);
        const int off = ((hf * 4 + i) ^ (row & 7)) * 16;
        *reinterpret_cast<uint4*>(prow + off) = hi; *reinterpret_cast<uint4*>(prow + TILE_Q + off) = lo;
      }
    }
    if (kb + 1 < n_kb) load_rows<HD>(kb_, p.ld, (kb + 1) * BK, p.T, p.rope_cos, p.rope_sin, rk);   // in flight under the P V MMAs
    tcgen05_fence_before();
    fence_proxy_async();
    EV_STAMP();
    __syncthreads();
    if (warp == 0) {
      tcgen05_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int c = 0; c < 2; ++c) {                     // feature chunk -> 64 columns of this block's O (a fresh accumulator); column = feature
          uint32_t acc = 0;
#pragma unroll
          for (int tt = 0; tt < 3; ++tt) {                // P_hi V_lo, P_lo V_hi, then P_hi V_hi
            const int term = tt == 2 ? 0 : tt + 1;
            const uint64_t da = make_smem_desc(p_s + (term == 2 ? (uint32_t)TILE_Q : 0u));
            const uint64_t db = make_smem_desc_ex(v_s + (uint32_t)(c * TILE_K) + (term == 1 ? 2u * TILE_K : 0u), 1024, 8192, 2);
#pragma unroll
            for (int k = 0; k < 4; ++k) { umma_bf16(tmem_base + O_COL + (uint32_t)(c * 64), da + (uint64_t)(2 * k), db + (uint64_t)(k * 128), idesc_o, acc); acc = 1; }
          }
        }
        umma_commit(&o_ready);
      }
      __syncwarp();
    }
    EV_STAMP();
    mbar_wait(&o_ready, par);
    EV_STAMP();
    tcgen05_fence_after();
    constexpr int LDW = NO % 32 == 0 ? 32 : 16;          // TMEM load width: 2 x 32 columns (HD = 128), 3 x 16 (HD = 96)
#pragma unroll
    for (int g = 0; g < NO / LDW; ++g) {                  // rounded fp32 adds into the running output
      uint32_t raw[LDW];
      if constexpr (LDW == 32) tmem_ld32(lane_addr + O_COL + (uint32_t)(hf * NO + g * LDW), raw);
      else tmem_ld16(lane_addr + O_COL + (uint32_t)(hf * NO + g * LDW), raw);
#pragma unroll
      for (int i = 0; i < LDW; ++i) o[g * LDW + i] += __uint_as_float(raw[i]);
    }
    tcgen05_fence_before();
  }
  red_sh[hf][row] = l;
  __syncthreads();
  l = red_sh[0][row] + red_sh[1][row];
  // every MMA has completed: the operand tiles are free.  The 128 x HD fp32 output goes through shared memory (16-byte chunks
  // XOR-swizzled by the row, conflict-free both ways, row pitch 512 bytes) so that a warp stores one full row per instruction.
  {
    const float inv = 1.0f / (l * kPScale * kOpScale);
    float4* stage = reinterpret_cast<float4*>(gen);
#pragma unroll
    for (int i = 0; i < NO / 4; ++i)
      stage[row * 32 + ((hf * (NO / 4) + i) ^ (row & 31))] = make_float4(o[4 * i] * inv, o[4 * i + 1] * inv, o[4 * i + 2] * inv, o[4 * i + 3] * inv);
    __syncthreads();
    float* ob = p.out + b * p.out_bs + h * HD;
#pragma unroll 4
    for (int r = warp; r < BQ; r += THREADS / 32) {
      const int tr = q0 + r;
      if (tr < p.T && lane < HD / 4) {
        const float4 y = stage[r * 32 + (lane ^ (r & 31))];
        *reinterpret_cast<float4*>(ob + (long long)tr * p.out_ld + 4 * lane) = y;
        if (p.split) {   // [hi | lo] halves of y * 8, exactly what split_f16_kernel would make of the stored row
          const float v0 = y.x * kF16ActScale, v1 = y.y * kF16ActScale, v2 = y.z * kF16ActScale, v3 = y.w * kF16ActScale;
          const __half h0 = __float2half_rn(v0), h1 = __float2half_rn(v1), h2 = __float2half_rn(v2), h3 = __float2half_rn(v3);
          const __half2 ha = __halves2half2(h0, h1), hb = __halves2half2(h2, h3);
          const __half2 la = __floats2half2_rn(v0 - __half2float(h0), v1 - __half2float(h1));
          const __half2 lb = __floats2half2_rn(v2 - __half2float(h2), v3 - __half2float(h3));
          __half* sp = p.split + ((long long)b * p.T + tr) * 2 * p.split_ld + h * HD + 4 * lane;
          *reinterpret_cast<uint2*>(sp) = make_uint2(*reinterpret_cast<const uint32_t*>(&ha), *reinterpret_cast<const uint32_t*>(&hb));
          *reinterpret_cast<uint2*>(sp + p.split_ld) = make_uint2(*reinterpret_cast<const uint32_t*>(&la), *reinterpret_cast<const uint32_t*>(&lb));
        }
      }
    }
  }
  EV_STAMP();
  if (tracer) {
    printf("attn_enc_tc trace (clk since start; per key block: S issued, S ready, P written, PV issued, O ready):");
    for (int i = 1; i < n_stamp; ++i) printf(" %lld", stamp[i] - stamp[0]);
    printf("\n");
  }
#undef EV_STAMP
  __syncthreads();
  if (warp == 0) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

template <int HD>
cudaError_t launch_enc_tc(const Params& p, dim3 grid, cudaStream_t s) {
  static DeviceOnce once;
  cudaError_t ce = once.run([&]() { return cudaFuncSetAttribute(attn_enc_tc_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES); });
  if (ce != cudaSuccess) return ce;
  return launch_pdl(attn_enc_tc_kernel<HD>, grid, dim3(THREADS), (size_t)SMEM_BYTES, s, p);
}

}  // namespace

bool attention_enc_tc_supported(const AttnArgs& a) {
  if (a.mode != 0 || (a.D != 96 && a.D != 128) || a.rope_dim != a.D / 2 || !a.rope_cos || !a.rope_sin) return false;
  return !((a.ld & 3) || (a.bs & 3) || (a.out_ld & 3) || (a.out_bs & 3) || (reinterpret_cast<uintptr_t>(a.q) & 15) ||
           (reinterpret_cast<uintptr_t>(a.k) & 15) || (reinterpret_cast<uintptr_t>(a.v) & 15) || (reinterpret_cast<uintptr_t>(a.out) & 15));
}

cudaError_t attention_enc_tc(const AttnArgs& a, cudaStream_t s) {
  if (!attention_enc_tc_supported(a)) return cudaErrorNotSupported;
  Params p;
  p.q = a.q; p.k = a.k; p.v = a.v; p.ld = a.ld; p.bs = a.bs;
  p.T = a.T; p.n_kb = ceil_div(a.T, BK);
  p.c1 = a.scale / (kOpScale * kOpScale);
  p.lens = a.lens; p.len_shift = a.len_shift;
  p.rope_cos = a.rope_cos; p.rope_sin = a.rope_sin;
  p.out = reinterpret_cast<float*>(a.out); p.out_ld = a.out_ld; p.out_bs = a.out_bs;
  p.split = reinterpret_cast<__half*>(a.split); p.split_ld = a.H * a.D;
  static const int trace = []() { const char* v = getenv("EV_ENC_ATTN_TRACE"); return (v && v[0] == '1') ? 1 : 0; }();
  p.trace = trace;
  const dim3 grid(ceil_div(a.T, BQ), a.H, a.B);
  return a.D == 96 ? launch_enc_tc<96>(p, grid, s) : launch_enc_tc<128>(p, grid, s);
}

}  // namespace ev
