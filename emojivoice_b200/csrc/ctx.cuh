// Context, weight store and the conv dispatch shared by matcha.cu / hifigan.cu / api.cu.
#pragma once
#include <map>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/emojivoice_b200.h"
#include "conv.cuh"
#include "kernels.cuh"

namespace ev {

struct ResnetW {
  ConvWeights conv1, conv2, res;
  float *gn1_g = nullptr, *gn1_b = nullptr, *gn2_g = nullptr, *gn2_b = nullptr;
  int c_in = 0;
};
struct TransformerW {
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln3_g = nullptr, *ln3_b = nullptr;
  ConvWeights qkv, out, ff1, ff2;
  float *snake_a = nullptr, *snake_invb = nullptr;
};
struct EncLayerW {
  ConvWeights qkv, o, ffn1, ffn2;
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
};

struct MatchaW {
  bool loaded = false;
  ev_matcha_cfg cfg{};
  float* spk_table = nullptr;
  float* tok_emb = nullptr;
  ConvWeights pre_conv[3], pre_proj;
  float *pre_g[3] = {}, *pre_b[3] = {};
  std::vector<EncLayerW> enc;
  ConvWeights proj_m, dp_conv1, dp_conv2, dp_proj;
  float *dp_g1 = nullptr, *dp_b1 = nullptr, *dp_g2 = nullptr, *dp_b2 = nullptr;
  float *rope_cos = nullptr, *rope_sin = nullptr;
  int rope_T = 0;
  // estimator
  ConvWeights time1, time2, temb_proj;  // temb_proj stacks the 6 resnet mlp.1 layers (N = 6*C)
  ResnetW rn[6];                        // down0, down1, mid0, mid1, up0, up1
  TransformerW tf[6];
  ConvWeights down0, down1_conv, up0, up1_conv, final_conv, final_proj;
  float *final_g = nullptr, *final_b = nullptr;
};

struct DenoiseTables {         // tables of the bias denoiser's FFT (denoiser.cu)
  float* win_sq = nullptr;     // hann^2 [1024]
  float2* twiddle = nullptr;   // [1024] exp(-2 pi i n / 1024)
  bool ready = false;
};

struct HifiganW {
  bool loaded = false;
  ev_hifigan_cfg cfg{};
  ConvWeights conv_pre;
  ConvWeights ups[8];
  ConvWeights c1[8][4][3], c2[8][4][3];
  float* bacc[8][4][3] = {};  // cumulative conv2 biases of each ResBlock (fused kernel: residual stream kept bias-free in TMEM)
  bool fuse_resblocks = true; // EV_RB_FUSE=0: layer-by-layer convs everywhere
  float* post_w = nullptr;   // [7][C_last]
  float* post_b = nullptr;
  int c_last = 0, total_up = 1;
  float* denoise_bias = nullptr;  // (n_fft/2+1) once ev_denoiser_init ran
  DenoiseTables dn;
};

}  // namespace ev

namespace ev {
struct ProfRecord { int kid; double flops, bytes; cudaEvent_t e0, e1; };
}

struct ev_ctx {
  int device = 0;
  int sm_count = 0;
  std::string err;
  long long launches = 0;
  std::vector<void*> owned;     // cudaMalloc'ed by this context
  ev::MatchaW matcha;
  ev::HifiganW hifigan;
  // optional per-launch CUDA-event timing (ev_profile_begin/end); off in normal operation
  // text encoder convs on tcgen05 via the 3xTF32 split with TWO-LEVEL ACCUMULATION (EV_ENC_TC=0: fp32 CUDA cores).
  // The tensor core's fp32 accumulation truncates: over K ~ 3000 a single TMEM accumulator measures 2e-6..2e-5 relative
  // error; flushing the partial sum into an fp32 master accumulator (rounded adds) every <= 16 MMAs brings it to
  // 4.0-4.9e-7, the same as the fp32 CUDA-core kernel (2e-7..6e-7) -- accurate enough for ceil(exp(logw)).
  bool enc_tc = true;
  bool profiling = false;
  bool prof_detail = false;    // EV_PROF_DETAIL=1: conv kernel classes carry the layer shape
  const char* prof_tag = "";   // appended to conv kernel names while profiling (enc / dec / voc)
  std::vector<ev::ProfRecord> prof;
  std::vector<std::string> kernel_names;
  std::vector<cudaEvent_t> event_pool;
  // decoder lanes: the batch is cut into up to EV_MAX_LANES independent slices whose kernels run on separate streams
  // (forked from / joined into the caller's stream, so a CUDA-graph capture sees parallel branches).  The decoder's
  // kernels at B = 32 are launch/prologue-latency bound (3 us of MMA in a 13 us kernel); concurrent lanes overlap them.
  static constexpr int kMaxLanes = 4;
  int dec_lanes = 1;            // EV_DEC_LANES (default 1: measured 16.86 ms -> 16.5 ms with 2 lanes, 17.5 ms with 4 -- the decoder's
                                // kernels already cover most SMs, so concurrent lanes mostly queue behind each other)
  // ragged vocoding (ev_vocode_ragged): active only while that call issues its launches
  ev::RaggedPlanner rag;
  double prof_scale = 1.0;      // profiling: algorithmic FLOPs/bytes of the launches are scaled by the valid-row fraction
  cudaStream_t lane_stream[kMaxLanes - 1] = {};
  cudaEvent_t lane_fork = nullptr, lane_join[kMaxLanes - 1] = {};
  // side branch of a ResNet block: res_conv(x) only depends on the block's input, so it runs on the last lane stream next to
  // conv1 -> GroupNorm -> conv2 and is joined before the residual add (EV_DEC_SIDE=0: serial).  Single-lane decoding only.
  bool dec_side = true;
  cudaEvent_t side_fork = nullptr, side_join = nullptr;
};

namespace ev {

int fail(ev_ctx* ctx, int code, const std::string& msg);
int cuda_fail(ev_ctx* ctx, cudaError_t ce, const char* what);
#define EV_CUDA(ctx, expr)                                          \
  do {                                                              \
    cudaError_t _ce = (expr);                                       \
    if (_ce != cudaSuccess) return ev::cuda_fail(ctx, _ce, #expr);  \
  } while (0)
#define EV_TRY(expr)            \
  do {                          \
    int _rc = (expr);           \
    if (_rc != 0) return _rc;   \
  } while (0)

// Every kernel launch goes through one of these: counts the launch and, while profiling, brackets it with events
// recorded on the launching stream.
struct LaunchScope {
  ev_ctx* ctx; cudaStream_t s; int idx;
  LaunchScope(ev_ctx* c, cudaStream_t st, const char* name, double flops, double bytes);
  ~LaunchScope();
};
#define EV_LAUNCH(ctx, s, name, flops, bytes, expr)                 \
  do {                                                              \
    cudaError_t _ce;                                                \
    { ev::LaunchScope _ls(ctx, s, name, flops, bytes); _ce = (expr); } \
    if (_ce != cudaSuccess) return ev::cuda_fail(ctx, _ce, name);   \
  } while (0)

// Bump allocator over the caller's workspace (256-byte granules).
struct Workspace {
  char* base;
  size_t size, off = 0;
  bool overflow = false;
  Workspace(void* p, size_t n) : base(reinterpret_cast<char*>(p)), size(n) {}
  template <typename T> T* take(size_t count) {
    size_t bytes = align_up(count * sizeof(T), 256);
    if (base == nullptr) { off += bytes; return nullptr; }   // sizing pass
    if (off + bytes > size) { overflow = true; return nullptr; }
    T* p = reinterpret_cast<T*>(base + off);
    off += bytes;
    return p;
  }
};

// name -> tensor lookup over the caller's ev_tensor list
struct WeightStore {
  std::map<std::string, const ev_tensor*> by_name;
  ev_ctx* ctx;
  cudaStream_t stream;
  WeightStore(ev_ctx* c, const ev_tensor* w, int n, cudaStream_t s);
  const ev_tensor* get(const std::string& name, std::initializer_list<long long> shape);
  bool has(const std::string& name) const { return by_name.count(name) != 0; }
  // plain fp32 copy owned by the context
  int copy_vec(const std::string& name, long long n, float** out);
};

enum ConvKind { CONV_NORMAL = 0, CONV_TRANSPOSED = 1 };
enum TcMode { TC_NONE = 0, TC_BF16 = 1, TC_TF32X3 = 2 };   // which tensor-core operand layout make_conv also packs
// Allocate + pack one conv / linear layer.  `names` may list several tensors stacked along N (fused QKV, stacked mlps).
int make_conv(ev_ctx* ctx, WeightStore& ws, const std::vector<std::string>& weight_names, const std::vector<std::string>& bias_names,
              int c_out_each, int c_in, int ksize, int stride, int pad, int dilation, ConvKind kind, int tc_mode,
              ConvWeights* out);
int device_alloc(ev_ctx* ctx, size_t bytes, void** out, bool zero, cudaStream_t s);

// Derive the GEMM geometry of `w` applied to B items of T_in rows; returns T_out.
int conv_geometry(const ConvWeights& w, int B, int T_in, ConvGeom* g);

// Launch `w` on x (ActT = float -> CUDA-core fp32, bf16 -> tcgen05); e carries the fused epilogue.
// fp32-accurate tensor-core convolution (3xTF32 split); `scratch` holds B*T_in*2*C_in floats
// presplit: `scratch` already holds the 3xFP16 [hi | lo] operand of x (written by the producer: LnArgs::split / AttnArgs::split);
// honoured only when the 3xFP16 path runs (enc_split_f16()), otherwise x is split here as usual
// sched / info: conv_tc_launch's per-call schedule and launch report (conv.cuh); left untouched when the CUDA-core kernel runs
int run_conv_tf32(ev_ctx* ctx, const ConvWeights& w, const float* x, long long x_ld, long long x_bs, int B, int T_in, Epilogue e,
                  float* scratch, cudaStream_t s, bool presplit = false, const TcSchedule* sched = nullptr, TcLaunchInfo* info = nullptr);
bool enc_split_f16();   // EV_ENC_SPLIT=tf32 selects the round-1 3xTF32 products (their operand has another layout)

template <typename ActT>
int run_conv(ev_ctx* ctx, const ConvWeights& w, const ActT* x, long long x_ld, long long x_bs, int B, int T_in,
             Epilogue e, cudaStream_t s, const TcSchedule* sched = nullptr, TcLaunchInfo* info = nullptr);

// ---- one HiFi-GAN ResBlock1 (hifigan.cu): what the vocoder runs per block, and what ev_test_resblock runs alone
// Packs `<prefix>convs1.{0,1,2}` / `<prefix>convs2.{0,1,2}` (C x C x k, dilations dil[0..2] and 1) and the cumulative conv2 biases
// bacc[l] = sum_{i <= l} convs2.i.bias the fused kernel adds to its residual stream.
int load_resblock(ev_ctx* ctx, WeightStore& ws, const std::string& prefix, int C, int k, const int dil[3], ConvWeights c1[3],
                  ConvWeights c2[3], float* bacc[3], cudaStream_t s);
template <typename ActT>
struct ResBlockArgs {
  int C = 0, k = 0;
  const ConvWeights* c1[3] = {};
  const ConvWeights* c2[3] = {};
  const float* bacc[3] = {};
  const float* x = nullptr;        // fp32 (B, L, C) block input
  const ActT* x_act = nullptr;     // lrelu(x) as the convs' operand (layer path)
  float* xb = nullptr; ActT* xba = nullptr; ActT* mid = nullptr;   // layer-path scratch, (B, L, C) each
  float* sum = nullptr;            // fp32 (B, L, C) multi-receptive-field accumulator
  ActT* act_out = nullptr;         // mode 2: lrelu(mean, slope_out) (the next stage's operand), or nullptr
  int B = 0, L = 0;
  // 0: sum = y   1: sum += y   2: sum = (sum + y) * inv_n (written only if write_f32)   3: as 2 without the sum read (a lone branch;
  // layer path only)
  int mode = 0, write_f32 = 1;
  float inv_n = 1.0f, slope_out = 0.1f;
  bool fused = false;              // resblock_tc (bf16 only) or six conv launches
  const RbSchedule* sched = nullptr;
  RbLaunchInfo* info = nullptr;
};
// Ragged batches: ctx->rag, as for run_conv.
template <typename ActT>
int run_resblock(ev_ctx* ctx, const ResBlockArgs<ActT>& a, cudaStream_t s);

}  // namespace ev
