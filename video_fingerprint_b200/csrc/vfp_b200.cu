// C-ABI implementation (include/vfp_b200.h): weight preparation, forward orchestration, similarity join.
// Single translation unit: all kernels are included as headers so the library is one nvcc invocation.
#include "../../include/vfp_b200.h"

#include <math.h>
#include <string.h>

#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "conv1_kernel.cuh"
#include "attention_tc_kernel.cuh"
#include "conv3_ts_kernel.cuh"
#include "ffn_kernel.cuh"
#include "gemm_launch.cuh"
#include "join_kernels.cuh"
#include "metrics_kernels.cuh"
#include "model3d_kernels.cuh"
#include "preprocess_kernels.cuh"
#include "stem_ts_kernel.cuh"
#include "token_kernels.cuh"
#include "topk_kernels.cuh"

using namespace vfp;

namespace {

thread_local std::string g_last_error;

int fail(const std::string& msg) {
  g_last_error = msg;
  return 1;
}
int fail_cuda(const char* what, cudaError_t e) {
  g_last_error = std::string(what) + ": " + cudaGetErrorString(e);
  return 2;
}
#define VFP_CUDA(call)                                  \
  do {                                                  \
    cudaError_t e__ = (call);                           \
    if (e__ != cudaSuccess) return fail_cuda(#call, e__); \
  } while (0)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

constexpr float kBnEps = 1e-5f;

// ---------------------------------------------------------------------------------------------
// optional stage profiler: CUDA events recorded between the stages of a forward pass, on the caller's
// stream (bench.py reads per-kernel time from here; it is off unless vfp_profile_enable(1) was called)
// ---------------------------------------------------------------------------------------------
enum Stage : int {
  kStConv1 = 0, kStConv2, kStConv3, kStConv4, kStTokEmbed, kStTemporalConv, kStLayerNorm, kStQkv, kStAttention,
  kStOutProj, kStPoolGemm, kStPool, kStFinal, kStMisc, kStStemFused, kStFfn, kNumStages
};
const char* const kStageNames[kNumStages] = {"conv1_stem", "conv2_igemm", "conv3_igemm", "conv4_igemm_pool", "token_embed_gemm",
                                             "temporal_conv", "layernorm", "qkv_gemm", "attention", "out_proj_gemm",
                                             "pool_logits_gemm", "temporal_pool",
                                             "final_projection", "misc", "stem_fused", "ffn_fused"};
struct Profiler {
  bool enabled = false;
  std::vector<cudaEvent_t> pool;
  std::vector<std::pair<int, cudaEvent_t>> marks;  // (stage that ENDS at this event, event); stage -1 = pass start
  size_t next = 0;
  double ms[kNumStages] = {0};
  unsigned long long launches = 0;
  void mark(int stage, cudaStream_t st) {
    if (!enabled) return;
    if (next == pool.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      pool.push_back(e);
    }
    cudaEvent_t e = pool[next++];
    cudaEventRecord(e, st);
    marks.emplace_back(stage, e);
  }
  void drain() {
    if (marks.empty()) return;
    cudaEventSynchronize(marks.back().second);
    for (size_t i = 1; i < marks.size(); ++i) {
      if (marks[i].first < 0) continue;
      float t = 0.f;
      cudaEventElapsedTime(&t, marks[i - 1].second, marks[i].second);
      ms[marks[i].first] += t;
    }
    marks.clear();
    next = 0;
  }
};
Profiler g_prof;
const int kTemporalKernels[4] = {3, 5, 7, 11};

// conv2 reads conv1's output in space-to-depth form [frame][16][16][(sh*2+sw)*32 + c] (a cell = 2x2 pixels).
// A 3x3/stride-2 tap (kh, kw) lives in cell offset d = {-1,0,0}[k], sub-position s = {1,0,1}[k]. K blocks are
// 64 channels (= two horizontally adjacent sub-pixels, one full 128-byte TMA row): {channel half, dw, dh}.
// Sub-pixels a block does not need (dw = -1 only uses sw = 1) get zero weights, so K = 6 * 64 = 384 (288 real).
struct Conv2KBlock { int c_half, dw, dh; };
const Conv2KBlock kConv2KBlocks[6] = {{1, 0, -1}, {0, 0, 0}, {1, 0, 0}, {1, -1, -1}, {0, -1, 0}, {1, -1, 0}};
inline int conv2_tap_index(int d, int sub) { return d == -1 ? (sub == 1 ? 0 : -1) : (sub == 0 ? 1 : 2); }

struct AttnBlockWeights {
  float *ln1_w, *ln1_b, *ln2_w, *ln2_b;
  __nv_bfloat16 *wqkv, *wo, *w1, *w2;
  float *bqkv, *bo, *b1, *b2;
  CUtensorMap tm_qkv, tm_o;
  CUtensorMap tm_w1_ffn, tm_w2_ffn;   // fused feed-forward kernel: boxes of 128 rows x 64 columns (one CTA's half of a 256-row block)
};

}  // namespace

struct vfp_weights {
  int embedding_dim = 0;
  int n_attn = 0;
  std::vector<void*> allocs;
  // frame encoder
  uint32_t* c1_wpack = nullptr;
  float* c1_bias = nullptr;
  __nv_bfloat16 *c2_w = nullptr, *c3_w = nullptr, *c4_w = nullptr;
  float *c2_b = nullptr, *c3_b = nullptr, *c4_b = nullptr;
  CUtensorMap tm_c2;
  CUtensorMap tm_c4h;   // conv4 filters with boxes of half the rows: one CTA's half of the CTA-pair GEMM's B tile
  __nv_bfloat16* c2f_w = nullptr;  // conv2 weights in the K order of the fused stem kernel
  CUtensorMap tm_c2f;
  __nv_bfloat16* c1ts_w = nullptr;  // conv1 weights stacked for the TS-mode stem kernel: [64 = (sw, c_out)][128 = (kh, 24 window values)]
  CUtensorMap tm_c1ts;
  // token embedding (Linear 256->S o Linear S->256, folded) + positional table
  __nv_bfloat16* wtok = nullptr;
  float* btok = nullptr;
  float* pe = nullptr;
  int pe_len = 0;
  CUtensorMap tm_tok;
  // temporal conv blocks
  float* tc_w[2] = {nullptr, nullptr};
  float* tc_b[2] = {nullptr, nullptr};
  std::vector<AttnBlockWeights> attn;
  // pooling + head
  __nv_bfloat16* wpool = nullptr;
  float* bpool = nullptr;
  CUtensorMap tm_pool;
  float *w0t = nullptr, *b0 = nullptr, *w3t = nullptr, *b3 = nullptr;
  // head on tensor cores (embedding_dim <= 256 and a multiple of 32): bf16 K-major copies of both layers
  bool head_on_tensor_cores = false;
  __nv_bfloat16 *w0_bf = nullptr, *w3_bf = nullptr;
  CUtensorMap tm_head0, tm_head3;
};

namespace {

struct TensorTable {
  std::map<std::string, const vfp_tensor_desc*> by_name;
  const float* get(const std::string& name, int64_t numel, std::string* err) const {
    auto it = by_name.find(name);
    if (it == by_name.end()) {
      *err = "missing checkpoint tensor: " + name;
      return nullptr;
    }
    if (it->second->numel != numel) {
      *err = "checkpoint tensor " + name + " has " + std::to_string(it->second->numel) + " elements, expected " +
             std::to_string(numel);
      return nullptr;
    }
    return static_cast<const float*>(it->second->data);
  }
  bool has(const std::string& name) const { return by_name.count(name) != 0; }
  int64_t numel(const std::string& name) const {
    auto it = by_name.find(name);
    return it == by_name.end() ? -1 : it->second->numel;
  }
};

template <class T>
int upload(vfp_weights* w, const std::vector<T>& host, T** dev) {
  void* p = nullptr;
  VFP_CUDA(cudaMalloc(&p, host.size() * sizeof(T)));
  w->allocs.push_back(p);
  VFP_CUDA(cudaMemcpy(p, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice));
  *dev = static_cast<T*>(p);
  return 0;
}

std::vector<__nv_bfloat16> to_bf16(const std::vector<float>& v) {
  std::vector<__nv_bfloat16> o(v.size());
  for (size_t i = 0; i < v.size(); ++i) o[i] = __float2bfloat16(v[i]);
  return o;
}

// eval-mode BN as per-channel scale/shift:  y = (x - mean) * gamma / sqrt(var + eps) + beta
struct BnFold {
  std::vector<float> scale, shift;
};
bool load_bn(const TensorTable& t, const std::string& prefix, int c, BnFold* out, std::string* err) {
  const float* g = t.get(prefix + ".weight", c, err);
  const float* b = g ? t.get(prefix + ".bias", c, err) : nullptr;
  const float* m = b ? t.get(prefix + ".running_mean", c, err) : nullptr;
  const float* v = m ? t.get(prefix + ".running_var", c, err) : nullptr;
  if (!v) return false;
  out->scale.resize(c);
  out->shift.resize(c);
  for (int i = 0; i < c; ++i) {
    const double s = (double)g[i] / sqrt((double)v[i] + (double)kBnEps);
    out->scale[i] = (float)s;
    out->shift[i] = (float)((double)b[i] - (double)m[i] * s);
  }
  return true;
}

// 3x3 conv weights (cout, cin, 3, 3) -> K-major GEMM operand [cout][(kh*3+kw)*cin + c], BN folded
int prep_conv3x3(vfp_weights* w, const TensorTable& t, int conv_idx, int cin, int cout, __nv_bfloat16** dw, float** db,
                 std::string* err) {
  const std::string p = "spatial_encoder.encoder.";
  const float* cw = t.get(p + std::to_string(conv_idx) + ".weight", (int64_t)cout * cin * 9, err);
  const float* cb = cw ? t.get(p + std::to_string(conv_idx) + ".bias", cout, err) : nullptr;
  BnFold bn;
  if (!cb || !load_bn(t, p + std::to_string(conv_idx + 1), cout, &bn, err)) return 1;
  std::vector<float> wf((size_t)cout * 9 * cin), bf(cout);
  for (int co = 0; co < cout; ++co) {
    for (int c = 0; c < cin; ++c)
      for (int kh = 0; kh < 3; ++kh)
        for (int kw = 0; kw < 3; ++kw)
          wf[(size_t)co * 9 * cin + (kh * 3 + kw) * cin + c] = cw[(((size_t)co * cin + c) * 3 + kh) * 3 + kw] * bn.scale[co];
    bf[co] = cb[co] * bn.scale[co] + bn.shift[co];
  }
  if (upload(w, to_bf16(wf), dw) || upload(w, bf, db)) return 1;
  return 0;
}

int prep_dense_bf16(vfp_weights* w, const float* src, size_t n, __nv_bfloat16** dev) {
  std::vector<float> v(src, src + n);
  return upload(w, to_bf16(v), dev);
}
int prep_f32(vfp_weights* w, const float* src, size_t n, float** dev) {
  std::vector<float> v(src, src + n);
  return upload(w, v, dev);
}

// ---------------------------------------------------------------------------------------------
// forward workspace. Two regions with different granularity:
//   * the TOKEN region holds one "token pass" (up to all clips of the call): 7.5 KB per frame/token. The token
//     GEMMs, LayerNorm, attention, pooling and the head each run ONCE per token pass, so their launches are large;
//   * the CONV region holds the activations of one "conv pass" (up to 65 536 frames by default, 48 KB per frame, plus 64 KB
//     per frame for 16 384 frames of conv1 output that only the two-kernel stem uses): the frame encoder walks the token
//     pass in such slices and only leaves the 512 B/frame pooled features behind.
// ---------------------------------------------------------------------------------------------
constexpr int64_t kConvPassFrames = 262144;  // workspace is sized for this many frames per conv pass (48 KB per frame)
// ... and for this many frames of conv1 output (64 KB per frame, two-kernel stem only), which steps through a conv pass in
// sub-passes of this size. Measured on B200 (10k x 64-frame clips): 512 -> 71.3 ms/step, 1024 -> 62.9, 2048 -> 60.7,
// 4096 -> 58.9, 16384 -> 55.8: short L2-sized sub-passes lose more to small launches than they save in HBM traffic.
constexpr int64_t kStemPassFrames = 16384;
// frames actually walked per conv pass (vfp_set_tuning key 3, <= kConvPassFrames). Every launch of the three persistent
// frame-encoder kernels costs ~13-16 us that do not scale with its size (cluster launch, TMEM allocation, the filters' trip
// into tensor memory, pipeline ramp and drain), so passes are LARGE: 10 000 x 64-frame clips take 32.9 ms per step with
// 16 384-frame passes, 32.1 with 65 536 and the same with 131 072 / 262 144 (profiles/r02_conv_pass_sweep.txt). Passes small
// enough to keep c2 / c3 in the 126 MB L2 (2 048 - 4 096 frames) lose far more to those fixed costs than they save in
// HBM traffic: 36.3 - 39.4 ms, 35.1 - 36.7 with programmatic dependent launch.
int64_t g_conv_pass_frames = 65536;
// conv1+conv2 in one kernel (stem_ts_kernel.cuh: conv1's output stays in shared memory as conv2's UMMA operand).
// Measured on B200 (10k x 64-frame clips): 13.3 ms vs 13.4 + 12.9 ms for the two HBM-bound kernels, so it is the
// default for u8 / bf16 frames; vfp_set_tuning(1, 0) selects the two-kernel path (always used for fp32 frames).
int g_fused_stem = 2;
int g_attention_tc = 1;    // key 17: attention on tcgen05 (attention_tc_kernel.cuh) instead of the mma.sync kernel

struct TokenWs {
  size_t cu, frame_src, att_items, frame_addr, tok_pos, tok_len, feat, xa, xb, xn, qkv, att, delta, delta2, logits, xbf, pooled, pooled_bf, head_h, total;
};
struct ConvWs {
  size_t c1, c2, c3, total;
};
TokenWs token_ws_layout(int64_t F, int64_t C) {
  TokenWs L{};
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off = align_up(off + bytes, 1024);
    return o;
  };
  // cu, frame_src and att_items are consecutive: the host stages the three per-pass tables in one buffer, one copy
  L.cu = take((size_t)(C + 1) * 4);
  L.frame_src = take((size_t)C * sizeof(FrameSrc));    // where each clip's frames are
  L.att_items = take((size_t)(F / 64 + C + 1) * 16);   // attention work items: <= F / 64 + C of them
  L.frame_addr = take((size_t)F * 8);                  // device address of every frame of the pass (token_map_kernel)
  L.tok_pos = take((size_t)F * 4);
  L.tok_len = take((size_t)F * 4);
  L.feat = take((size_t)F * 256 * 2);
  L.xa = take((size_t)F * kDim * 4);
  L.xb = take((size_t)F * kDim * 4);
  L.xn = take((size_t)F * kDim * 2);
  L.qkv = take((size_t)F * 3 * kDim * 2);
  L.att = take((size_t)F * kDim * 2);
  L.delta = take((size_t)F * kDim * 2);
  L.delta2 = take((size_t)F * kDim * 2);
  L.logits = take((size_t)F * kDim * 4);
  L.xbf = take((size_t)F * kDim * 2);
  L.pooled = take((size_t)C * 3 * kDim * 4);
  L.pooled_bf = take((size_t)C * 3 * kDim * 2);
  L.head_h = take((size_t)C * kDim * 2);
  L.total = off;
  return L;
}
ConvWs conv_ws_layout(int64_t F) {   // F = frames per conv pass
  ConvWs L{};
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off = align_up(off + bytes, 1024);
    return o;
  };
  L.c1 = take((size_t)std::min<int64_t>(F, kStemPassFrames) * 32 * 32 * 32 * 2);
  L.c2 = take((size_t)F * 16 * 16 * 64 * 2);
  L.c3 = take((size_t)F * 8 * 8 * 128 * 2);
  L.total = off;
  return L;
}
size_t forward_ws_total(int64_t F, int64_t C) {
  return token_ws_layout(F, C).total + conv_ws_layout(std::min<int64_t>(F, g_conv_pass_frames)).total;   // follows tuning key 3: size and call under the same setting
}

// Pipelines of vfp_forward (vfp_set_tuning key 9): token passes are dealt round-robin onto this many internal streams.
// Measured on B200 (10 000 x 64-frame clips): 1 pipeline 38.6-38.9 ms per step, 2 pipelines 38.6-39.6, 3 pipelines 39.9 -
// the kernels of one pass already fill the GPU, so the default is ONE pipeline (the caller's stream, no fork / join).
constexpr int kMaxPipes = 4;
int g_forward_pipes = 1;

// Internal non-blocking streams, created once per device and shared by all calls (work of different calls on the same
// pipeline stream simply queues up; the fork / join events are per call).
int pipe_streams(int n, cudaStream_t* out) {
  static std::mutex mu;
  static cudaStream_t pool[kMaxDevices][kMaxPipes] = {};
  std::lock_guard<std::mutex> g(mu);
  const int dev = current_device();
  for (int i = 0; i < n; ++i) {
    if (!pool[dev][i]) VFP_CUDA(cudaStreamCreateWithFlags(&pool[dev][i], cudaStreamNonBlocking));
    out[i] = pool[dev][i];
  }
  return 0;
}

}  // namespace

// =============================================================================================
// exported functions
// =============================================================================================
extern "C" {

int vfp_abi_version(void) { return VFP_ABI_VERSION; }
const char* vfp_last_error(void) { return g_last_error.c_str(); }

int vfp_device_sm_count(void) {
  int n = 0, dev = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  int sms = 0;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
  return sms;
}

int vfp_set_tuning(int key, long long value) {
  if (key == 1 && (value == 0 || value == 2)) { g_fused_stem = (int)value; return 0; }
  if (key == 3 && value >= 64 && value <= kConvPassFrames) { g_conv_pass_frames = value; return 0; }
  if (key == 17 && value >= 0 && value <= 1) { g_attention_tc = (int)value; return 0; }
  if (key == 9 && value >= 1 && value <= kMaxPipes) { g_forward_pipes = (int)value; return 0; }        // pipelines (internal streams) of vfp_forward
  if (key == 2) {  // hang diagnosis: timed-out mbarrier waits are logged and abandoned instead of trapping
    const int mode = value != 0;
    const unsigned int zero = 0;
    if (cudaMemcpyToSymbol(g_vfp_hang_mode, &mode, sizeof(mode)) != cudaSuccess) return 2;
    if (cudaMemcpyToSymbol(g_vfp_hang_count, &zero, sizeof(zero)) != cudaSuccess) return 2;
    return 0;
  }
  return 1;
}

int vfp_profile_enable(int on) {
  g_prof.drain();
  g_prof.enabled = on != 0;
  return 0;
}
int vfp_profile_num_stages(void) { return kNumStages; }
const char* vfp_profile_stage_name(int i) { return (i >= 0 && i < kNumStages) ? kStageNames[i] : ""; }
int vfp_profile_read(double* stage_ms, int n_stages, uint64_t* launches, int reset) {
  g_prof.drain();
  for (int i = 0; i < n_stages && i < kNumStages; ++i) stage_ms[i] = g_prof.ms[i];
  if (launches) *launches = g_prof.launches;
  if (reset) {
    for (int i = 0; i < kNumStages; ++i) g_prof.ms[i] = 0;
    g_prof.launches = 0;
  }
  return 0;
}

unsigned int vfp_device_error_word(void) {
  unsigned int v = 0, zero = 0;
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(&v, g_vfp_device_error, sizeof(v));
  if (v) cudaMemcpyToSymbol(g_vfp_device_error, &zero, sizeof(zero));
  return v;
}

#ifdef VFP_FFN_TRACE
int vfp_debug_ffn_trace(long long* out, int max_pairs) {   // development builds only (not declared in the header): copies + clears
  (void)max_pairs;
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out, g_ffn_trace, sizeof(long long) * 8192 / 2);
  static long long zeros[4096];
  cudaMemcpyToSymbol(g_ffn_trace, zeros, sizeof(zeros));
  return 2048;
}
#endif

int vfp_debug_hang_log(unsigned int* out, int max_entries) {
  unsigned int n = 0;
  cudaDeviceSynchronize();
  if (cudaMemcpyFromSymbol(&n, g_vfp_hang_count, sizeof(n)) != cudaSuccess) return -1;
  if (n > 64) n = 64;
  if ((int)n > max_entries) n = (unsigned int)max_entries;
  if (n && cudaMemcpyFromSymbol(out, g_vfp_hang_log, (size_t)n * 16) != cudaSuccess) return -1;
  return (int)n;
}

void vfp_weights_destroy(vfp_weights* w) {
  if (!w) return;
  for (void* p : w->allocs) cudaFree(p);
  delete w;
}

int vfp_weights_embedding_dim(const vfp_weights* w) { return w ? w->embedding_dim : 0; }

int vfp_weights_create(const vfp_tensor_desc* tensors, int n_tensors, vfp_weights** out) {
  if (!tensors || !out) return fail("vfp_weights_create: null argument");
  if (vfp_device_sm_count() <= 0) return fail("vfp_weights_create: no CUDA device (there is no CPU fallback)");
  if (!tensor_map_encoder()) return fail("vfp_weights_create: cuTensorMapEncodeTiled not available from the driver");
  TensorTable t;
  for (int i = 0; i < n_tensors; ++i) t.by_name[tensors[i].name] = &tensors[i];
  std::string err;
  vfp_weights* w = new vfp_weights();
  auto bail = [&](const std::string& m) {
    vfp_weights_destroy(w);
    return fail("vfp_weights_create: " + (m.empty() ? g_last_error : m));
  };
  const std::string enc = "spatial_encoder.encoder.";

  // ---- conv1 (3->32, k5): BN folded, packed as mma.sync B fragments [kh][n-tile][lane][2] ----
  {
    const float* cw = t.get(enc + "0.weight", 32 * 3 * 25, &err);
    const float* cb = cw ? t.get(enc + "0.bias", 32, &err) : nullptr;
    BnFold bn;
    if (!cb || !load_bn(t, enc + "1", 32, &bn, &err)) return bail(err);
    auto wk = [&](int co, int kh, int k) -> float {  // k = kw*3 + c, k == 15 is the zero pad
      if (k >= 15) return 0.0f;
      const int kw = k / 3, c = k % 3;
      return cw[((co * 3 + c) * 5 + kh) * 5 + kw] * bn.scale[co];
    };
    // column g of n-tile nt is channel nt*8 + g
    std::vector<uint32_t> pack(5 * 4 * 32 * 2);
    for (int kh = 0; kh < 5; ++kh)
      for (int nt = 0; nt < 4; ++nt)
        for (int lane = 0; lane < 32; ++lane) {
          const int g = lane >> 2, tig = lane & 3, co = nt * 8 + g;
          for (int r = 0; r < 2; ++r) {
            const int k0 = 2 * tig + 8 * r;
            const __nv_bfloat16 lo = __float2bfloat16(wk(co, kh, k0)), hi = __float2bfloat16(wk(co, kh, k0 + 1));
            uint16_t l16, h16;
            memcpy(&l16, &lo, 2);
            memcpy(&h16, &hi, 2);
            pack[((kh * 4 + nt) * 32 + lane) * 2 + r] = (uint32_t)l16 | ((uint32_t)h16 << 16);
          }
        }
    std::vector<float> bias(32);
    for (int co = 0; co < 32; ++co) bias[co] = cb[co] * bn.scale[co] + bn.shift[co];
    if (upload(w, pack, &w->c1_wpack) || upload(w, bias, &w->c1_bias)) return bail("");
    // stem_ts_kernel.cuh: an A row is a horizontal pair of output pixels (sw = 0, 1) of output row oh; per filter row kh it
    // holds 24 consecutive HWC values starting at pixel 4cx-3 channel 1: k = kh*24 + 2 + 3*p + ci is pixel 4cx-2+p, channel
    // ci. Output pixel ow = 2cx + sw reads pixels 4cx + 2sw - 2 + kw, i.e. p = 2sw + kw. Everything else is zero.
    std::vector<float> wts((size_t)64 * 128, 0.0f);
    for (int sw = 0; sw < 2; ++sw)
      for (int co = 0; co < 32; ++co)
        for (int kh = 0; kh < 5; ++kh)
          for (int kw = 0; kw < 5; ++kw)
            for (int ci = 0; ci < 3; ++ci)
              wts[(size_t)(sw * 32 + co) * 128 + kh * 24 + 2 + 3 * (2 * sw + kw) + ci] = cw[((co * 3 + ci) * 5 + kh) * 5 + kw] * bn.scale[co];
    // K columns 120 / 121 of every A row are 1.0: the folded bias rides along as two bf16 (hi + lo)
    for (int sw = 0; sw < 2; ++sw)
      for (int co = 0; co < 32; ++co) {
        const float hi = __bfloat162float(__float2bfloat16(bias[co]));
        wts[(size_t)(sw * 32 + co) * 128 + 120] = hi;
        wts[(size_t)(sw * 32 + co) * 128 + 121] = bias[co] - hi;
      }
    if (upload(w, to_bf16(wts), &w->c1ts_w)) return bail("");
  }
  // ---- conv2..4 ----
  {  // conv2: K laid out to match kConv2KBlocks (see there)
    const float* cw = t.get(enc + "3.weight", 64 * 32 * 9, &err);
    const float* cb = cw ? t.get(enc + "3.bias", 64, &err) : nullptr;
    BnFold bn;
    if (!cb || !load_bn(t, enc + "4", 64, &bn, &err)) return bail(err);
    std::vector<float> wf((size_t)64 * 384, 0.0f), bf(64);
    for (int co = 0; co < 64; ++co) {
      for (int kb = 0; kb < 6; ++kb)
        for (int j = 0; j < 2; ++j) {
          const int block = 2 * kConv2KBlocks[kb].c_half + j, sh = block >> 1, sw = block & 1;
          const int kh = conv2_tap_index(kConv2KBlocks[kb].dh, sh), kw = conv2_tap_index(kConv2KBlocks[kb].dw, sw);
          if (kh < 0 || kw < 0) continue;
          for (int c = 0; c < 32; ++c)
            wf[(size_t)co * 384 + kb * 64 + j * 32 + c] = cw[((co * 32 + c) * 3 + kh) * 3 + kw] * bn.scale[co];
        }
      bf[co] = cb[co] * bn.scale[co] + bn.shift[co];
    }
    if (upload(w, to_bf16(wf), &w->c2_w) || upload(w, bf, &w->c2_b)) return bail("");
    // fused stem kernel (stem_common.cuh), five K blocks of 64 = [half 0: 32 ch | half 1: 32 ch], per block and
    // half the (kh, kw) tap it holds (-1 = zero):
    //   blk0 G_A (AL0, dh=0):  (1,1) | (2,1)      blk1 G_B (AL1, dh=0): (2,2) | (1,2)      blk2 G_C (AL1, dh=0, shifted): (2,0) | (1,0)
    //   blk3 G_E | G_D (dh=-1): (0,2) | (0,1)     blk4 G_F (dh=-1, shifted): (0,0) | zero
    // (blk1;blk2 and blk3;blk4 are adjacent in shared memory: each pair is the stacked 128-row operand of one N=128 UMMA)
    const int fused_tap[5][2][2] = {{{1, 1}, {2, 1}}, {{2, 2}, {1, 2}}, {{2, 0}, {1, 0}}, {{0, 2}, {0, 1}}, {{0, 0}, {-1, -1}}};
    std::vector<float> wfu((size_t)64 * 320, 0.0f);
    for (int co = 0; co < 64; ++co)
      for (int kb = 0; kb < 5; ++kb)
        for (int half = 0; half < 2; ++half) {
          const int kh = fused_tap[kb][half][0], kw = fused_tap[kb][half][1];
          if (kh < 0) continue;
          for (int c = 0; c < 32; ++c)
            wfu[(size_t)co * 320 + kb * 64 + half * 32 + c] = cw[((co * 32 + c) * 3 + kh) * 3 + kw] * bn.scale[co];
        }
    if (upload(w, to_bf16(wfu), &w->c2f_w)) return bail("");
  }
  if (prep_conv3x3(w, t, 6, 64, 128, &w->c3_w, &w->c3_b, &err)) return bail(err);
  if (prep_conv3x3(w, t, 9, 128, 256, &w->c4_w, &w->c4_b, &err)) return bail(err);

  // ---- Linear(256->S) o Linear(S->256) folded, + positional table ----
  {
    const int64_t s_numel = t.numel(enc + "14.bias");
    if (s_numel <= 0) return bail("missing checkpoint tensor: " + enc + "14.bias");
    const int S = (int)s_numel;
    const float* ws = t.get(enc + "14.weight", (int64_t)S * 256, &err);
    const float* bs = ws ? t.get(enc + "14.bias", S, &err) : nullptr;
    const float* wt = bs ? t.get("temporal_projection.weight", (int64_t)kDim * S, &err) : nullptr;
    const float* bt = wt ? t.get("temporal_projection.bias", kDim, &err) : nullptr;
    if (!bt) return bail(err.empty() ? "temporal_dim must be 256" : err);
    std::vector<float> wf((size_t)kDim * 256), bf(kDim);
    for (int o = 0; o < kDim; ++o) {
      for (int i = 0; i < 256; ++i) {
        double acc = 0;
        for (int s = 0; s < S; ++s) acc += (double)wt[(size_t)o * S + s] * (double)ws[(size_t)s * 256 + i];
        wf[(size_t)o * 256 + i] = (float)acc;
      }
      double acc = bt[o];
      for (int s = 0; s < S; ++s) acc += (double)wt[(size_t)o * S + s] * (double)bs[s];
      bf[o] = (float)acc;
    }
    if (upload(w, to_bf16(wf), &w->wtok) || upload(w, bf, &w->btok)) return bail("");
    const int64_t pe_numel = t.numel("pos_encoding.pe");
    if (pe_numel <= 0 || pe_numel % kDim) return bail("missing or malformed checkpoint tensor: pos_encoding.pe");
    w->pe_len = (int)(pe_numel / kDim);
    if (prep_f32(w, t.get("pos_encoding.pe", pe_numel, &err), (size_t)pe_numel, &w->pe)) return bail("");
  }
  // ---- temporal conv blocks: BN folded, 11 centred taps, layout [ci][tap][o] ----
  for (int blk = 0; blk < 2; ++blk) {
    std::vector<float> wf(4 * 11 * kDim, 0.0f), bf(kDim);
    for (int j = 0; j < 4; ++j) {
      const int k = kTemporalKernels[j], off = (11 - k) / 2;
      const std::string p = "temporal_conv_blocks." + std::to_string(blk) + ".convs." + std::to_string(j);
      const float* cw = t.get(p + ".0.weight", 64 * 4 * k, &err);
      const float* cb = cw ? t.get(p + ".0.bias", 64, &err) : nullptr;
      BnFold bn;
      if (!cb || !load_bn(t, p + ".1", 64, &bn, &err)) return bail(err);
      for (int g = 0; g < 64; ++g) {
        const int o = j * 64 + g;
        for (int ci = 0; ci < 4; ++ci)
          for (int dt = 0; dt < k; ++dt) wf[(ci * 11 + off + dt) * kDim + o] = cw[(g * 4 + ci) * k + dt] * bn.scale[g];
        bf[o] = cb[g] * bn.scale[g] + bn.shift[g];
      }
    }
    if (upload(w, wf, &w->tc_w[blk]) || upload(w, bf, &w->tc_b[blk])) return bail("");
  }
  // ---- attention blocks ----
  while (t.has("attention_blocks." + std::to_string(w->n_attn) + ".norm1.weight")) ++w->n_attn;
  w->attn.resize(w->n_attn);
  for (int b = 0; b < w->n_attn; ++b) {
    const std::string p = "attention_blocks." + std::to_string(b);
    AttnBlockWeights& a = w->attn[b];
    struct F32Item { const char* key; int64_t n; float** dst; };
    const F32Item f32s[] = {
        {".norm1.weight", kDim, &a.ln1_w}, {".norm1.bias", kDim, &a.ln1_b}, {".norm2.weight", kDim, &a.ln2_w},
        {".norm2.bias", kDim, &a.ln2_b},   {".attn.in_proj_bias", 3 * kDim, &a.bqkv},
        {".attn.out_proj.bias", kDim, &a.bo}, {".conv1.bias", 4 * kDim, &a.b1}, {".conv2.bias", kDim, &a.b2}};
    for (const F32Item& it : f32s) {
      const float* src = t.get(p + it.key, it.n, &err);
      if (!src) return bail(err);
      if (prep_f32(w, src, (size_t)it.n, it.dst)) return bail("");
    }
    struct BfItem { const char* key; int64_t n; __nv_bfloat16** dst; };
    const BfItem bfs[] = {{".attn.in_proj_weight", 3 * kDim * kDim, &a.wqkv}, {".attn.out_proj.weight", kDim * kDim, &a.wo},
                          {".conv1.weight", 4 * kDim * kDim, &a.w1},          {".conv2.weight", 4 * kDim * kDim, &a.w2}};
    for (const BfItem& it : bfs) {
      const float* src = t.get(p + it.key, it.n, &err);
      if (!src) return bail(err);
      if (prep_dense_bf16(w, src, (size_t)it.n, it.dst)) return bail("");
    }
    if (make_tmap_rows_bf16(&a.tm_qkv, a.wqkv, 3 * kDim, kDim, kDim, 256, 64) ||
        make_tmap_rows_bf16(&a.tm_o, a.wo, kDim, kDim, kDim, 256, 64))
      return bail("tensor map encode failed (attention weights)");
    if (make_tmap_rows_bf16(&a.tm_w1_ffn, a.w1, 4 * kDim, kDim, kDim, 128, 64) ||
        make_tmap_rows_bf16(&a.tm_w2_ffn, a.w2, kDim, 4 * kDim, 4 * kDim, 128, 64))
      return bail("tensor map encode failed (feed-forward weights)");
  }
  // ---- pooling + head ----
  {
    const float* wp = t.get("temporal_pool.0.weight", kDim * kDim, &err);
    const float* bp = wp ? t.get("temporal_pool.0.bias", kDim, &err) : nullptr;
    const float* w0 = bp ? t.get("final_projection.0.weight", (int64_t)kDim * 3 * kDim, &err) : nullptr;
    const float* b0 = w0 ? t.get("final_projection.0.bias", kDim, &err) : nullptr;
    if (!b0) return bail(err);
    const int64_t d_numel = t.numel("final_projection.3.bias");
    if (d_numel <= 0 || d_numel > 512) return bail("final_projection.3.bias missing or embedding_dim > 512");
    const int D = (int)d_numel;
    const float* w3 = t.get("final_projection.3.weight", (int64_t)D * kDim, &err);
    const float* b3 = w3 ? t.get("final_projection.3.bias", D, &err) : nullptr;
    if (!b3) return bail(err);
    w->embedding_dim = D;
    std::vector<float> w0t((size_t)3 * kDim * kDim), w3t((size_t)kDim * D);
    for (int o = 0; o < kDim; ++o)
      for (int k = 0; k < 3 * kDim; ++k) w0t[(size_t)k * kDim + o] = w0[(size_t)o * 3 * kDim + k];
    for (int o = 0; o < D; ++o)
      for (int k = 0; k < kDim; ++k) w3t[(size_t)k * D + o] = w3[(size_t)o * kDim + k];
    if (prep_dense_bf16(w, wp, (size_t)kDim * kDim, &w->wpool) || prep_f32(w, bp, kDim, &w->bpool) ||
        upload(w, w0t, &w->w0t) || prep_f32(w, b0, kDim, &w->b0) || upload(w, w3t, &w->w3t) ||
        prep_f32(w, b3, (size_t)D, &w->b3))
      return bail("");
    if (D <= 256 && D % 32 == 0) {
      if (prep_dense_bf16(w, w0, (size_t)kDim * 3 * kDim, &w->w0_bf) || prep_dense_bf16(w, w3, (size_t)D * kDim, &w->w3_bf))
        return bail("");
      if (make_tmap_rows_bf16(&w->tm_head0, w->w0_bf, kDim, 3 * kDim, 3 * kDim, 256, 64) ||
          make_tmap_rows_bf16(&w->tm_head3, w->w3_bf, (uint64_t)D, kDim, kDim, 256, 64))
        return bail("tensor map encode failed (head)");
      w->head_on_tensor_cores = true;
    }
  }
  if (make_tmap_rows_bf16(&w->tm_c2, w->c2_w, 64, 384, 384, 64, 64) ||
      make_tmap_rows_bf16(&w->tm_c2f, w->c2f_w, 64, 320, 320, 64, 64) ||
      make_tmap_rows_bf16(&w->tm_c1ts, w->c1ts_w, 64, 128, 128, 64, 64) ||
      make_tmap_rows_bf16(&w->tm_c4h, w->c4_w, 256, 1152, 1152, 128, 64) ||
      make_tmap_rows_bf16(&w->tm_tok, w->wtok, kDim, 256, 256, 256, 64) ||
      make_tmap_rows_bf16(&w->tm_pool, w->wpool, kDim, kDim, kDim, 256, 64))
    return bail("tensor map encode failed (weights)");
  VFP_CUDA(cudaDeviceSynchronize());
  *out = w;
  return 0;
}

size_t vfp_forward_workspace_bytes(int64_t frames_per_pass, int64_t clips_per_pass) {
  if (frames_per_pass <= 0) return 0;
  if (clips_per_pass <= 0 || clips_per_pass > frames_per_pass) clips_per_pass = frames_per_pass;
  return forward_ws_total(frames_per_pass, clips_per_pass);
}

}  // extern "C"

namespace {

// Frame encoder over the F frames at frame_addr[0 .. F) (device table, one address per frame) -> feat_out (bf16 [frames][256]).
// `fused_ok`: every frame address is 16-byte aligned, as the fused stem's bulk copies need.
int encode_frames_pass(const vfp_weights* w, const unsigned long long* frame_addr, int frame_dtype, bool fused_ok, int64_t F,
                       __nv_bfloat16* feat_out, uint8_t* conv_ws, cudaStream_t st) {
  const ConvWs L = conv_ws_layout(F);
  __nv_bfloat16* c1a = reinterpret_cast<__nv_bfloat16*>(conv_ws + L.c1);
  __nv_bfloat16* c2a = reinterpret_cast<__nv_bfloat16*>(conv_ws + L.c2);
  __nv_bfloat16* c3a = reinterpret_cast<__nv_bfloat16*>(conv_ws + L.c3);
  CUtensorMap ta;
  // the fused stem streams raw frame planes with 16-byte bulk copies; fp32 frames (48 KB) do not fit its smem ring
  const bool fused = g_fused_stem && frame_dtype != VFP_FRAME_F32 && fused_ok;
  if (fused) {
    StemTsParams sp{};
    sp.tmap_w2 = w->tm_c2f;
    sp.tmap_w1 = w->tm_c1ts;
    if (make_tmap_out(&sp.tmap_out, c2a, (uint64_t)F * 256, 64, true)) return fail("tensor map encode failed (stem out)");
    sp.frame_addr = frame_addr; sp.frame_dtype = frame_dtype; sp.n_frames = F;
    sp.c2_bias = w->c2_b;
    VFP_CUDA(ensure_dynamic_smem(reinterpret_cast<const void*>(stem_ts_kernel), StemTsSmem::kTotal));
    g_prof.launches += 1;
    const int grid = (int)std::min<int64_t>(F, device_sm_count());
    VFP_CUDA(launch_kernel(stem_ts_kernel, dim3(grid), dim3(kStemThreads), StemTsSmem::kTotal, st, sp));
    g_prof.mark(kStStemFused, st);
  }
  for (int64_t s0 = 0; s0 < F && !fused; s0 += kStemPassFrames) {
    const int64_t n = std::min<int64_t>(kStemPassFrames, F - s0);
    g_prof.launches += 2;
    {
      const long long grid = std::min<long long>(n, (long long)device_sm_count() * 10);
      conv1_stem_kernel<<<(unsigned)grid, kC1Threads, 0, st>>>(frame_addr + s0, frame_dtype, n, w->c1_wpack,
                                                              w->c1_bias, c1a);
      g_prof.mark(kStConv1, st);
    }
    {  // conv2: c1 is stored space-to-depth [frame][16][16][4*32] -> dense 2x2/stride-1 taps; tile = 8 rows x 16 cols
      if (make_tmap_nhwc_bf16(&ta, c1a, n, 16, 16, 128, 64, 16, 8, 1, 1)) return fail("tensor map encode failed (conv2)");
      GemmShape s{};
      s.m_tiles = (int)(2 * n); s.n_tiles = 1; s.k_blocks = 6; s.group_m = 16; s.a_conv = 1;
      s.tiles_per_frame = 2; s.frames_per_tile = 1; s.tile_out_rows = 8; s.h_mul = 1; s.n_segments = 1;
      for (int kb = 0; kb < 6; ++kb) {
        s.tap_c_blk[kb] = (signed char)kConv2KBlocks[kb].c_half;
        s.tap_w[kb] = (signed char)kConv2KBlocks[kb].dw;
        s.tap_h[kb] = (signed char)kConv2KBlocks[kb].dh;
      }
      EpiBiasActTma<true>::Params ep{};
      if (make_tmap_out(&ep.tmap_out, c2a + (size_t)s0 * 256 * 64, (uint64_t)n * 256, 64, true)) return fail("tensor map encode failed (conv2 out)");
      ep.bias = w->c2_b; ep.N = 64; ep.act = 1;
      // N = 64 is narrow: three row tiles per CTA tile, round-robin over three accumulators (see gemm_sm100.cuh)
      VFP_CUDA((launch_gemm<64, 64, 3, EpiBiasActTma<true>, 3>(ta, w->tm_c2, s, ep, st)));
      g_prof.mark(kStConv2, st);
    }
  }
  g_prof.launches += 2;
  {  // conv3: 16x16x64 -> 8x8x128 with its filters in tensor memory, three frames per tile (conv3_ts_kernel.cuh). (A weight-resident
     // variant - launch_gemm_bres<128, 64, 3, 9>, all nine filter blocks in shared memory, M = 128 pixels - measured 2.01 ms vs
     // 1.25 ms per 131 072 frames: the kernel is bound by the nine-fold L2 -> SM re-read of the input pixels, not by the weights.)
    Conv3Params cp{};
    if (make_tmap_nhwc_bf16(&cp.tmap_in, c2a, F, 16, 16, 64, 64, 8, 8, kC3Frames, 2) || make_tmap_out(&cp.tmap_out, c3a, (uint64_t)F * 64, 128, true))
      return fail("tensor map encode failed (conv3)");
    cp.w = w->c3_w; cp.bias = w->c3_b; cp.n_tiles = (int)((F + kC3Frames - 1) / kC3Frames);
    VFP_CUDA(ensure_dynamic_smem(reinterpret_cast<const void*>(conv3_ts_kernel<7>), Conv3Smem<7>::kTotal));
    VFP_CUDA(launch_kernel(conv3_ts_kernel<7>, dim3(std::min(cp.n_tiles, device_sm_count())), dim3(kC3Threads), Conv3Smem<7>::kTotal, st, cp));
    g_prof.mark(kStConv3, st);
  }
  {  // conv4: 8x8x128 -> 4x4x256 + ReLU + global average pool, tile = 8 frames
    if (make_tmap_nhwc_bf16(&ta, c3a, F, 8, 8, 128, 64, 4, 4, 8, 2)) return fail("tensor map encode failed (conv4)");
    GemmShape s{};
    s.m_tiles = (int)((F + 7) / 8); s.n_tiles = 1; s.k_blocks = 18; s.group_m = 16; s.a_conv = 1;
    s.tiles_per_frame = 1; s.frames_per_tile = 8; s.tile_out_rows = 4;
    conv_taps_strided(&s, 2);
    EpiConvPool16::Params ep{};
    ep.bias = w->c4_b; ep.out_bf16 = feat_out; ep.frames = (int)F; ep.N = 256;
    // CTA pairs: one M256 N256 UMMA per K step. Measured (10 000 clips): 5.19 ms with one CTA per tile, 4.9 ms on pairs.
    VFP_CUDA((launch_gemm_pair<64, 6, EpiConvPool16>(ta, w->tm_c4h, s, ep, st)));
    g_prof.mark(kStConv4, st);
  }
  return 0;
}

// One token pass: clips [c0, c1), whose frames are src[c0 .. c1) (host records), = rows [f0, f0 + F) of the packed
// features (cu_host: prefix sums of the clip lengths).
int forward_pass(const vfp_weights* w, const FrameSrc* src, int frame_dtype, bool fused_ok, const int64_t* cu_host, int c0,
                 int c1, float* emb_out, float* features_out, uint8_t* ws, cudaStream_t st) {
  const int C = c1 - c0;
  const int64_t f0 = cu_host[c0];
  const int64_t F = cu_host[c1] - f0;
  const TokenWs L = token_ws_layout(F, C);
  uint8_t* conv_ws = ws + L.total;
  int* d_cu = reinterpret_cast<int*>(ws + L.cu);
  const FrameSrc* d_src = reinterpret_cast<const FrameSrc*>(ws + L.frame_src);
  unsigned long long* frame_addr = reinterpret_cast<unsigned long long*>(ws + L.frame_addr);
  int* tok_pos = reinterpret_cast<int*>(ws + L.tok_pos);
  int* tok_len = reinterpret_cast<int*>(ws + L.tok_len);
  __nv_bfloat16* feat = reinterpret_cast<__nv_bfloat16*>(ws + L.feat);
  float* xa = reinterpret_cast<float*>(ws + L.xa);
  float* xb = reinterpret_cast<float*>(ws + L.xb);
  __nv_bfloat16* xn = reinterpret_cast<__nv_bfloat16*>(ws + L.xn);
  __nv_bfloat16* qkv = reinterpret_cast<__nv_bfloat16*>(ws + L.qkv);
  __nv_bfloat16* att = reinterpret_cast<__nv_bfloat16*>(ws + L.att);
  __nv_bfloat16* delta = reinterpret_cast<__nv_bfloat16*>(ws + L.delta);     // attention out-projection of the current block
  __nv_bfloat16* delta_f = reinterpret_cast<__nv_bfloat16*>(ws + L.delta2);  // MLP output of the previous block
  float* logits = reinterpret_cast<float*>(ws + L.logits);
  __nv_bfloat16* xbf = reinterpret_cast<__nv_bfloat16*>(ws + L.xbf);
  float* pooled = reinterpret_cast<float*>(ws + L.pooled);
  __nv_bfloat16* pooled_bf = reinterpret_cast<__nv_bfloat16*>(ws + L.pooled_bf);
  __nv_bfloat16* head_h = reinterpret_cast<__nv_bfloat16*>(ws + L.head_h);

  // The per-pass tables, staged in one host buffer laid out like the workspace from L.cu on and copied with one call:
  // clip prefix sums relative to this pass, the clips' frame records, and the attention work items (64 query tokens of
  // one clip each, {first query token, clip start, clip end, 0}).
  std::vector<int32_t> cu_rel(C + 1);
  for (int i = 0; i <= C; ++i) cu_rel[i] = (int32_t)(cu_host[c0 + i] - f0);
  size_t n_items = 0;
  for (int i = 0; i < C; ++i) n_items += (size_t)(cu_rel[i + 1] - cu_rel[i] + kAttRows - 1) / kAttRows;
  std::vector<uint8_t> tables(L.att_items - L.cu + n_items * 16);
  memcpy(tables.data(), cu_rel.data(), (size_t)(C + 1) * 4);
  memcpy(tables.data() + (L.frame_src - L.cu), src + c0, (size_t)C * sizeof(FrameSrc));
  int32_t* items_host = reinterpret_cast<int32_t*>(tables.data() + (L.att_items - L.cu));
  for (int i = 0; i < C; ++i)
    for (int q = cu_rel[i]; q < cu_rel[i + 1]; q += kAttRows) {
      items_host[0] = q; items_host[1] = cu_rel[i]; items_host[2] = cu_rel[i + 1]; items_host[3] = 0;
      items_host += 4;
    }
  g_prof.mark(-1, st);
  g_prof.launches += 8 + 7 * (unsigned long long)w->n_attn;
  int4* att_items = reinterpret_cast<int4*>(ws + L.att_items);
  // pageable source: the copy is staged before the call returns, so the vector may die with this scope
  VFP_CUDA(cudaMemcpyAsync(d_cu, tables.data(), tables.size(), cudaMemcpyHostToDevice, st));
  VFP_CUDA(launch_kernel(token_map_kernel, dim3((unsigned)((F + 255) / 256)), dim3(256), 0, st, (const int*)d_cu, d_src, C, (int)F,
                         tok_pos, tok_len, frame_addr));
  g_prof.mark(kStMisc, st);

  // ---- frame encoder, one conv pass at a time (frames are independent: slices ignore clip boundaries) ----
  for (int64_t s0 = 0; s0 < F; s0 += g_conv_pass_frames) {
    const int64_t n = std::min<int64_t>(g_conv_pass_frames, F - s0);
    if (int rc = encode_frames_pass(w, frame_addr + s0, frame_dtype, fused_ok, n, feat + s0 * 256, conv_ws, st))
      return rc;
  }
  // ---- token embedding: x = Wtok feat + btok + pe[pos] ----
  auto token_gemm = [&](const __nv_bfloat16* A, int64_t M, int K, const CUtensorMap& tb, int N, const EpiBiasAct::Params& ep) -> int {
    CUtensorMap tma;
    if (make_tmap_rows_bf16(&tma, A, (uint64_t)M, (uint64_t)K, (uint64_t)K, 128, 64)) return fail("tensor map encode failed (tokens)");
    GemmShape s = plain_shape(M, N, K, 256, 64, 32);
    if (K == 256) {  // the whole 256x256 weight block of a column tile stays in shared memory
      VFP_CUDA((launch_gemm_bres<256, 64, 4, 4, EpiBiasAct>(tma, tb, s, ep, st)));
    } else {
      VFP_CUDA((launch_gemm<256, 64, 4, EpiBiasAct>(tma, tb, s, ep, st)));
    }
    return 0;
  };
  // bf16-output token GEMM, result written by the TMA unit (coalesced); act: 0 none, 2 gelu. The whole 256x256 weight block of
  // a column tile stays in shared memory: on CTA pairs (gemm_pair_tcgen05_kernel) QKV took 1.91 ms instead of 1.25 and the
  // out-projection 0.64 instead of 0.48 (10 000 clips).
  auto token_gemm_bf16 = [&](const __nv_bfloat16* A, int64_t M, int K, const CUtensorMap& tb, int N, const float* bias, int act,
                             __nv_bfloat16* out) -> int {
    CUtensorMap tma;
    if (make_tmap_rows_bf16(&tma, A, (uint64_t)M, (uint64_t)K, (uint64_t)K, 128, 64)) return fail("tensor map encode failed (tokens)");
    EpiBiasActTma<true>::Params ep{};
    if (make_tmap_out(&ep.tmap_out, out, (uint64_t)M, (uint64_t)N, true)) return fail("tensor map encode failed (token out)");
    ep.bias = bias; ep.N = N; ep.act = act;
    GemmShape s = plain_shape(M, N, K, 256, 64, 32);
    VFP_CUDA((launch_gemm_bres<256, 64, 4, 4, EpiBiasActTma<true>>(tma, tb, s, ep, st)));
    return 0;
  };
  {  // fp32 stream written through the TMA store path (row-per-thread fp32 stores touch 32 lines per instruction)
    CUtensorMap tma;
    if (make_tmap_rows_bf16(&tma, feat, (uint64_t)F, 256, 256, 128, 64)) return fail("tensor map encode failed (tokens)");
    EpiBiasActTma<false>::Params ep{};
    if (make_tmap_out(&ep.tmap_out, xa, (uint64_t)F, kDim, false)) return fail("tensor map encode failed (token embedding out)");
    ep.bias = w->btok; ep.N = kDim; ep.act = 0; ep.pe = w->pe; ep.token_pos = tok_pos; ep.M = (int)F;
    GemmShape s = plain_shape(F, kDim, 256, 256, 64, 32);
    VFP_CUDA((launch_gemm_bres<256, 64, 2, 4, EpiBiasActTma<false>>(tma, w->tm_tok, s, ep, st)));
    g_prof.mark(kStTokEmbed, st);
  }
  // ---- multi-scale temporal convolutions (residual) ----
  {
    // input rows staged by TMA, persistent CTAs (token_kernels.cuh)
    VFP_CUDA(ensure_dynamic_smem(reinterpret_cast<const void*>(temporal_conv_tma_kernel), kTc2SmemBytes));
    float* bufs[3] = {xa, xb, xa};
    for (int blk = 0; blk < 2; ++blk) {
      TemporalConvParams tp{};
      if (make_tmap_rows_f32(&tp.tmap_x, bufs[blk], (uint64_t)F, kDim, kTc2Rows)) return fail("tensor map encode failed (temporal conv)");
      tp.tok_pos = tok_pos; tp.tok_len = tok_len; tp.w = w->tc_w[blk]; tp.bias = w->tc_b[blk]; tp.y = bufs[blk + 1];
      tp.n_tokens = (int)F; tp.n_tiles = (int)((F + kTc2Tok - 1) / kTc2Tok);
      const int grid = std::min(tp.n_tiles, 2 * device_sm_count());
      VFP_CUDA(launch_kernel(temporal_conv_tma_kernel, dim3((unsigned)grid), dim3(kTc2Threads), kTc2SmemBytes, st, tp));
    }
    g_prof.mark(kStTemporalConv, st);
  }
  // ---- attention blocks ----
  const unsigned ln_grid = (unsigned)((F * 32 + 255) / 256);
  VFP_CUDA(ensure_dynamic_smem(reinterpret_cast<const void*>(attention_fa_kernel), kAttSmemBytes));
  AttnTcParams atc{};
  if (g_attention_tc) {
    if (make_tmap_rows_bf16(&atc.tmap_qkv, qkv, (uint64_t)F, 3 * kDim, 3 * kDim, 64, 64)) return fail("tensor map encode failed (attention)");
    atc.items = att_items; atc.out = att; atc.n_units = (int)n_items * 4;
    VFP_CUDA(ensure_dynamic_smem(reinterpret_cast<const void*>(attention_tc_kernel), kAtcSmemBytes));
  }
  // residual updates travel as bf16 `delta` and are folded into the fp32 stream by the next LayerNorm (see there)
  for (int b = 0; b < w->n_attn; ++b) {
    const AttnBlockWeights& a = w->attn[b];
    VFP_CUDA(launch_kernel(add_layernorm_bf16_kernel, dim3(ln_grid), dim3(256), 0, st, xa, b > 0 ? delta : nullptr, b > 0 ? delta_f : nullptr, a.ln1_w, a.ln1_b, xn, (int)F, 1));
    g_prof.mark(kStLayerNorm, st);
    if (token_gemm_bf16(xn, F, kDim, a.tm_qkv, 3 * kDim, a.bqkv, 0, qkv)) return 1;
    g_prof.mark(kStQkv, st);
    if (g_attention_tc) {
      const int grid = std::min(atc.n_units, 2 * device_sm_count());
      VFP_CUDA(launch_kernel(attention_tc_kernel, dim3((unsigned)grid), dim3(kAtcThreads), kAtcSmemBytes, st, atc));
    } else {
      VFP_CUDA(launch_kernel(attention_fa_kernel, dim3((unsigned)n_items), dim3(kAttThreads), kAttSmemBytes, st, qkv, att_items, att, (int)F));
    }
    g_prof.mark(kStAttention, st);
    if (token_gemm_bf16(att, F, kDim, a.tm_o, kDim, a.bo, 0, delta)) return 1;
    g_prof.mark(kStOutProj, st);
    VFP_CUDA(launch_kernel(add_layernorm_bf16_kernel, dim3(ln_grid), dim3(256), 0, st, xa, delta, (const __nv_bfloat16*)nullptr, a.ln2_w, a.ln2_b, xn, (int)F, 0));
    g_prof.mark(kStLayerNorm, st);
    {   // both GEMMs in one kernel on CTA pairs, the hidden activation stays on the SM (ffn_kernel.cuh)
      FfnParams fp{};
      if (make_tmap_rows_bf16(&fp.tmap_x, xn, (uint64_t)F, kDim, kDim, 128, 64)) return fail("tensor map encode failed (feed-forward)");
      fp.tmap_w1 = a.tm_w1_ffn; fp.tmap_w2 = a.tm_w2_ffn;
      if (make_tmap_out(&fp.tmap_out, delta_f, (uint64_t)F, kDim, true)) return fail("tensor map encode failed (feed-forward out)");
      fp.b1 = a.b1; fp.b2 = a.b2; fp.M = (int)F; fp.pair_tiles = (int)((F + 255) / 256);
      const int grid = 2 * std::min(fp.pair_tiles, device_sm_count() / 2);
      VFP_CUDA(ensure_dynamic_smem(reinterpret_cast<const void*>(ffn_pair_kernel<5>), FfnSmem<5>::kTotal));
      VFP_CUDA(launch_kernel_cluster(2, ffn_pair_kernel<5>, dim3(grid), dim3(kFfnThreads), FfnSmem<5>::kTotal, st, fp));
      g_prof.mark(kStFfn, st);
    }
  }
  // close the last block's residual and make the bf16 copy the pooling GEMM reads
  VFP_CUDA(launch_kernel(add_convert_bf16_kernel, dim3((unsigned)((F * kDim / 8 + 255) / 256)), dim3(256), 0, st, xa, w->n_attn > 0 ? delta : nullptr,
                         w->n_attn > 0 ? delta_f : nullptr, xbf, (long long)(F * kDim / 8)));
  if (features_out)
    VFP_CUDA(cudaMemcpyAsync(features_out + (size_t)f0 * kDim, xa, (size_t)F * kDim * 4, cudaMemcpyDeviceToDevice, st));
  // ---- pooling + head ----
  {
    // fp32 logits through the TMA store path (row-per-thread fp32 stores touch 32 lines per instruction)
    CUtensorMap tma;
    if (make_tmap_rows_bf16(&tma, xbf, (uint64_t)F, kDim, kDim, 128, 64)) return fail("tensor map encode failed (pool in)");
    EpiBiasActTma<false>::Params ep{};
    if (make_tmap_out(&ep.tmap_out, logits, (uint64_t)F, kDim, false)) return fail("tensor map encode failed (pool logits)");
    ep.bias = w->bpool; ep.N = kDim; ep.act = 1;
    GemmShape s = plain_shape(F, kDim, kDim, 256, 64, 32);
    VFP_CUDA((launch_gemm_bres<256, 64, 2, 4, EpiBiasActTma<false>>(tma, w->tm_pool, s, ep, st)));   // the 256 x 256 weight block stays in shared memory
    g_prof.mark(kStPoolGemm, st);
  }
  VFP_CUDA(launch_kernel(temporal_pool_kernel, dim3((unsigned)C), dim3(256), 0, st, xa, logits, d_cu, pooled, pooled_bf));
  g_prof.mark(kStPool, st);
  float* emb_dst = emb_out + (size_t)c0 * w->embedding_dim;
  if (w->head_on_tensor_cores) {
    // final_projection as two tcgen05 GEMMs: [C,768]x[768,256] + ReLU, then [C,256]x[256,D] + bias + L2 normalise
    EpiBiasAct::Params ep{};
    ep.bias = w->b0; ep.act = 1; ep.out_bf16 = head_h; ep.ld_out = kDim; ep.M = C; ep.N = kDim;
    if (token_gemm(pooled_bf, C, 3 * kDim, w->tm_head0, kDim, ep)) return 1;
    CUtensorMap tma;
    if (make_tmap_rows_bf16(&tma, head_h, (uint64_t)C, kDim, kDim, 128, 64)) return fail("tensor map encode failed (head)");
    GemmShape s = plain_shape(C, w->embedding_dim, kDim, 256, 64, 32);
    EpiBiasL2Norm::Params en{};
    en.bias = w->b3; en.out_f32 = emb_dst; en.M = C; en.N = w->embedding_dim;
    VFP_CUDA((launch_gemm<256, 64, 4, EpiBiasL2Norm>(tma, w->tm_head3, s, en, st)));
  } else {
    VFP_CUDA(launch_kernel(final_projection_kernel<8>, dim3((unsigned)((C + 7) / 8)), dim3(256), 0, st, pooled, w->w0t, w->b0, w->w3t, w->b3,
                           w->embedding_dim, C, emb_dst));
  }
  g_prof.mark(kStFinal, st);
  if (g_prof.marks.size() > 4096) g_prof.drain();
  VFP_CUDA(cudaGetLastError());
  return 0;
}

// The one planner of the attention model. Clip i is len[i] frames, frame t at device address src[i].addr + t * src[i].pitch:
// clips may be packed back to back, separate allocations, views with any frame stride, overlapping or repeated. Checks the
// lengths and the workspace, then runs the clips in token passes cut on clip boundaries, dealt round-robin onto the pipelines.
// `aligned`: every address and pitch is a multiple of 16 bytes, which the fused stem's bulk copies need.
int forward_clips(const std::string& name, const vfp_weights* w, const FrameSrc* src, const int32_t* len, int n_clips,
                  int frame_dtype, bool aligned, float* emb_out, float* features_out, void* workspace, size_t workspace_bytes,
                  void* stream) {
  std::vector<int64_t> cu((size_t)n_clips + 1, 0);   // prefix sums: clip i owns rows cu[i] .. cu[i+1] of the features
  int max_T = 0, longest = 0;
  for (int i = 0; i < n_clips; ++i) {
    const int T = len[i];
    if (T <= 0) return fail(name + ": clip " + std::to_string(i) + " has no frames");
    if (T > w->pe_len)   // the positional table of the checkpoint (model.py:77: max_len 10000) is the only length limit
      return fail(name + ": clip " + std::to_string(i) + " has " + std::to_string(T) + " frames; the positional table holds " +
                  std::to_string(w->pe_len));
    if (T > max_T) { max_T = T; longest = i; }
    cu[i + 1] = cu[i] + T;
  }
  const int64_t total = cu[n_clips];
  // The workspace is cut into equal slices, one per pipeline; a pipeline = an internal stream that takes every
  // n_pipes-th token pass. Passes are independent (disjoint clips, own workspace slice), so the tail of one pass's
  // kernels overlaps the head of another's, and HBM-bound stages of one pass run beside tensor-bound stages of another.
  auto fit = [&](size_t bytes) {   // largest pass (in frames) `bytes` can hold; a pass never has more clips than frames
    int64_t lo = 0, hi = total;
    while (lo < hi) {
      const int64_t mid = (lo + hi + 1) / 2;
      if (forward_ws_total(mid, std::min<int64_t>(mid, n_clips)) <= bytes) lo = mid; else hi = mid - 1;
    }
    return lo;
  };
  int n_pipes = g_prof.enabled ? 1 : std::max(1, std::min(g_forward_pipes, kMaxPipes));   // stage timing needs one stream
  n_pipes = (int)std::min<int64_t>(n_pipes, std::max<int64_t>(1, total / kConvPassFrames));  // small calls: one pass on the caller's stream
  auto slice_bytes = [&](int n) { return workspace_bytes / n / 1024 * 1024; };
  while (n_pipes > 1 && fit(slice_bytes(n_pipes)) < max_T) --n_pipes;
  const int64_t pass_frames = fit(slice_bytes(n_pipes));
  if (pass_frames < max_T)
    return fail(name + ": workspace of " + std::to_string(workspace_bytes) + " bytes cannot hold the longest clip (clip " +
                std::to_string(longest) + ": " + std::to_string(max_T) + " frames need " + std::to_string(forward_ws_total(max_T, 1)) + ")");
  const size_t slice = slice_bytes(n_pipes);
  // passes of about equal size, a multiple of n_pipes of them
  int64_t n_pass = (total + pass_frames - 1) / pass_frames;
  n_pass = (n_pass + n_pipes - 1) / n_pipes * n_pipes;
  const int64_t target = (total + n_pass - 1) / n_pass;
  cudaStream_t caller = static_cast<cudaStream_t>(stream);
  cudaStream_t pipe[kMaxPipes] = {caller, nullptr, nullptr, nullptr};
  cudaEvent_t fork = nullptr;
  if (n_pipes > 1) {
    if (int rc = pipe_streams(n_pipes, pipe)) return rc;
    VFP_CUDA(cudaEventCreateWithFlags(&fork, cudaEventDisableTiming));
    VFP_CUDA(cudaEventRecord(fork, caller));
    for (int p = 0; p < n_pipes; ++p) VFP_CUDA(cudaStreamWaitEvent(pipe[p], fork, 0));
  }
  int rc = 0;
  int c0 = 0, pass = 0;
  while (c0 < n_clips && rc == 0) {
    int c1 = c0 + 1;   // a clip always fits (pass_frames >= max_T); add clips up to the target, never past the slice capacity
    while (c1 < n_clips && cu[c1 + 1] - cu[c0] <= pass_frames && cu[c1] - cu[c0] < target) ++c1;
    const int p = pass % n_pipes;
    rc = forward_pass(w, src, frame_dtype, aligned, cu.data(), c0, c1, emb_out, features_out,
                      static_cast<uint8_t*>(workspace) + (size_t)p * slice, pipe[p]);
    c0 = c1;
    ++pass;
  }
  if (n_pipes > 1) {   // join: the caller's stream continues when every pipeline has drained (also on the error path)
    for (int p = 0; p < n_pipes; ++p) {
      cudaEvent_t done = nullptr;
      if (cudaEventCreateWithFlags(&done, cudaEventDisableTiming) == cudaSuccess) {
        cudaEventRecord(done, pipe[p]);
        cudaStreamWaitEvent(caller, done, 0);
        cudaEventDestroy(done);   // released by the runtime once the recorded work has completed
      }
    }
    cudaEventDestroy(fork);
  }
  return rc;
}

size_t frame_bytes_of(int frame_dtype) {
  return (size_t)12288 * (frame_dtype == VFP_FRAME_BF16 ? 2 : frame_dtype == VFP_FRAME_F32 ? 4 : 1);
}

// Embedding widths the search accepts: the rule of vfp_pair_stats (every fp32 row is 16-byte aligned for float4 loads and
// every bf16 screen row is a whole number of 32-byte sectors). The screen runs ceil(dim / 64) K blocks of 64 columns.
bool search_dim_ok(int dim) { return dim >= 16 && dim <= 512 && dim % 16 == 0; }

// Database column tiles (of kAres2BlockN = 256 rows) per L2 panel of the join: 65 536 rows, 32 MB of bf16 at dim 256.
constexpr int kJoinPanelTiles = 256;

}  // namespace

extern "C" {

int vfp_forward(const vfp_weights* w, const void* frames, int frame_dtype, const int32_t* cu, int n_clips,
                float* emb_out, float* features_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!w || !frames || !cu || !emb_out || !workspace) return fail("vfp_forward: null argument");
  if (n_clips <= 0) return fail("vfp_forward: n_clips must be positive");
  if (frame_dtype < 0 || frame_dtype > 3) return fail("vfp_forward: unknown frame dtype");
  const size_t frame_bytes = frame_bytes_of(frame_dtype);
  if (cu[0] != 0) return fail("vfp_forward: cu_seqlens[0] must be 0");
  // the packed frames as clip records with a dense pitch; an unaligned buffer takes the two-kernel stem, as it always has
  std::vector<FrameSrc> src((size_t)n_clips);
  std::vector<int32_t> len((size_t)n_clips);
  for (int i = 0; i < n_clips; ++i) {
    src[i].addr = reinterpret_cast<uintptr_t>(frames) + (unsigned long long)cu[i] * frame_bytes;
    src[i].pitch = (long long)frame_bytes;
    len[i] = cu[i + 1] - cu[i];
  }
  const bool aligned = (reinterpret_cast<uintptr_t>(frames) & 15) == 0;
  return forward_clips("vfp_forward", w, src.data(), len.data(), n_clips, frame_dtype, aligned, emb_out, features_out, workspace,
                       workspace_bytes, stream);
}

int vfp_forward_clips(const vfp_weights* w, const void* const* clip_frames_host, const int64_t* frame_pitch_bytes_host,
                      const int32_t* lengths_host, int n_clips, int frame_dtype, float* emb_out, float* features_out,
                      void* workspace, size_t workspace_bytes, void* stream) {
  const std::string name = "vfp_forward_clips";
  if (!w || !clip_frames_host || !lengths_host || !emb_out || !workspace) return fail(name + ": null argument");
  if (n_clips <= 0) return fail(name + ": n_clips must be positive");
  if (frame_dtype < 0 || frame_dtype > 3) return fail(name + ": unknown frame_dtype " + std::to_string(frame_dtype));
  const long long frame_bytes = (long long)frame_bytes_of(frame_dtype);
  std::vector<FrameSrc> src((size_t)n_clips);
  for (int i = 0; i < n_clips; ++i) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(clip_frames_host[i]);
    const long long pitch = frame_pitch_bytes_host ? (long long)frame_pitch_bytes_host[i] : frame_bytes;
    if (!a) return fail(name + ": clip " + std::to_string(i) + " has a null frame pointer");
    if (a % 16)
      return fail(name + ": clip " + std::to_string(i) + "'s frame pointer is not 16-byte aligned (frames are read in 16-byte copies)");
    if (pitch < frame_bytes || pitch % 16)
      return fail(name + ": clip " + std::to_string(i) + " has a frame pitch of " + std::to_string(pitch) +
                  " bytes; it must be a multiple of 16 and at least one frame (" + std::to_string(frame_bytes) + " bytes)");
    src[i].addr = a;
    src[i].pitch = pitch;
  }
  return forward_clips(name, w, src.data(), lengths_host, n_clips, frame_dtype, true, emb_out, features_out, workspace,
                       workspace_bytes, stream);
}

// ---------------------------------------------------------------------------------------------
// similarity join
// ---------------------------------------------------------------------------------------------
size_t vfp_join_workspace_bytes_dim(int64_t n_q, int64_t n_db, int64_t candidate_capacity, int dim) {
  if (n_q <= 0 || n_db <= 0 || !search_dim_ok(dim)) return 0;
  if (candidate_capacity < 1024) candidate_capacity = 1024;
  return align_up((size_t)n_q * 2 * dim, 1024) + align_up((size_t)n_db * 2 * dim, 1024) +
         3 * align_up((size_t)candidate_capacity * 4, 1024) + 1024;
}
size_t vfp_join_workspace_bytes(int64_t n_q, int64_t n_db, int64_t candidate_capacity) {
  return vfp_join_workspace_bytes_dim(n_q, n_db, candidate_capacity, 256);
}

int vfp_join_threshold(const float* q, const float* db, int64_t n_q, int64_t n_db, int dim, int64_t q_row0, float thr,
                       float screen_margin, int32_t* out_i, int32_t* out_j, float* out_s, int64_t capacity,
                       uint64_t* counts_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!q || !db || !out_i || !out_j || !out_s || !counts_out || !workspace) return fail("vfp_join_threshold: null argument");
  if (!search_dim_ok(dim))
    return fail("vfp_join_threshold: dim " + std::to_string(dim) + " is not supported (16 <= dim <= 512, dim % 16 == 0)");
  if (n_q <= 0 || n_db <= 0) return fail("vfp_join_threshold: empty operand");
  if (n_q > 0x7fffff00LL || n_db > 0x7fffff00LL || q_row0 + n_q > 0x7fffff00LL) return fail("vfp_join_threshold: more than 2^31 rows");
  if (!(screen_margin >= 0.0f)) return fail("vfp_join_threshold: screen_margin must be >= 0");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  const bool self_join = (q == db && n_q == n_db);
  const int kb = (dim + 63) / 64;
  const size_t row_bytes = (size_t)2 * dim;   // one bf16 screen row
  const size_t q_bytes = align_up((size_t)n_q * row_bytes, 1024), db_bytes = align_up((size_t)n_db * row_bytes, 1024);
  const size_t fixed = q_bytes + db_bytes + 1024;
  if (workspace_bytes < fixed + 3 * 4096)
    return fail("vfp_join_threshold: workspace too small for dim " + std::to_string(dim) + "; see vfp_join_workspace_bytes_dim");
  const int64_t cand_cap = (int64_t)((workspace_bytes - fixed) / 3 / 1024 * 1024 / 4);
  __nv_bfloat16* qbf = reinterpret_cast<__nv_bfloat16*>(ws);
  __nv_bfloat16* dbbf = self_join ? qbf : reinterpret_cast<__nv_bfloat16*>(ws + q_bytes);
  int* cand_i = reinterpret_cast<int*>(ws + q_bytes + db_bytes);
  int* cand_j = cand_i + cand_cap;
  float* cand_s = reinterpret_cast<float*>(cand_j + cand_cap);
  unsigned long long* cand_count = reinterpret_cast<unsigned long long*>(ws + q_bytes + db_bytes + 3 * (size_t)cand_cap * 4);
  unsigned long long* counts = reinterpret_cast<unsigned long long*>(counts_out);

  VFP_CUDA(cudaMemsetAsync(cand_count, 0, 8, st));
  VFP_CUDA(cudaMemsetAsync(counts, 0, 16, st));
  const long long q8 = n_q * dim / 8, db8 = n_db * dim / 8;   // 8 elements per thread
  f32_to_bf16_kernel<<<(unsigned)((q8 + 255) / 256), 256, 0, st>>>(q, qbf, q8);
  if (!self_join) f32_to_bf16_kernel<<<(unsigned)((db8 + 255) / 256), 256, 0, st>>>(db, dbbf, db8);
  // a self join's score matrix is symmetric: screen the upper triangle only, the re-score kernel emits both orders
  const int tri = self_join ? 1 : 0;
  EpiJoinThreshold::Params ep{};
  ep.thr = thr - screen_margin;
  ep.q_rows = n_q; ep.db_rows = n_db; ep.q_row0 = q_row0;
  ep.out_i = cand_i; ep.out_j = cand_j; ep.out_s = cand_s; ep.count = cand_count; ep.capacity = cand_cap;
  // The screen operands are the unpadded bf16 rows: the tensor maps have an inner extent of dim columns and a 2 * dim-byte
  // pitch, and TMA zero-fills the columns past dim in the last 64-column K block.
  // A-resident, panel-major schedule on CTA pairs (cta_group::2 UMMAs, gemm_sm100.cuh)
  CUtensorMap ta, tb;
  if (make_tmap_rows_bf16(&ta, qbf, (uint64_t)n_q, dim, dim, 128, 64) ||
      make_tmap_rows_bf16(&tb, dbbf, (uint64_t)n_db, dim, dim, 128, 64))
    return fail("vfp_join_threshold: tensor map encode failed");
  AresShape s{};
  s.block_n = kAres2BlockN;
  s.m_super = (int)((n_q + kAresMT * kBlockM - 1) / (kAresMT * kBlockM));   // 256 query rows per work item
  s.n_tiles = (int)((n_db + s.block_n - 1) / s.block_n);
  // a panel of <= 65 536 database rows (32 MB of bf16) stays in L2 while every query super-tile passes over it; small
  // problems get shorter panels so that there are enough items to balance the SMs
  int panel = kJoinPanelTiles;
  const int workers = device_sm_count() / 2;
  while (panel > 8 && (long long)s.m_super * ((s.n_tiles + panel - 1) / panel) < 16LL * workers) panel /= 2;
  s.panel_tiles = panel;
  s.n_panels = (s.n_tiles + panel - 1) / panel;
  s.tri = tri;
  s.q_row0 = 0;   // tri compares LOCAL row and column indices: q and db are the same matrix
  ep.tri = tri;
  // Stages of the database ring: 8 up to kb = 6; above that the resident query rows (16 KB per K block) leave room for
  // 14 - kb stages of 16 KB within the 227 KB a block may have.
  cudaError_t e = cudaErrorInvalidValue;
  switch (kb) {
    case 1: e = launch_gemm_ares2<8, 1, EpiJoinThreshold>(ta, tb, s, ep, st); break;
    case 2: e = launch_gemm_ares2<8, 2, EpiJoinThreshold>(ta, tb, s, ep, st); break;
    case 3: e = launch_gemm_ares2<8, 3, EpiJoinThreshold>(ta, tb, s, ep, st); break;
    case 4: e = launch_gemm_ares2<8, 4, EpiJoinThreshold>(ta, tb, s, ep, st); break;
    case 5: e = launch_gemm_ares2<8, 5, EpiJoinThreshold>(ta, tb, s, ep, st); break;
    case 6: e = launch_gemm_ares2<8, 6, EpiJoinThreshold>(ta, tb, s, ep, st); break;
    case 7: e = launch_gemm_ares2<7, 7, EpiJoinThreshold>(ta, tb, s, ep, st); break;
    case 8: e = launch_gemm_ares2<6, 8, EpiJoinThreshold>(ta, tb, s, ep, st); break;
  }
  VFP_CUDA(e);
  rescore_pairs_kernel<<<device_sm_count() * 4, 256, 0, st>>>(q, db, dim, q_row0, cand_i, cand_j, cand_count, cand_cap, thr,
                                                              out_i, out_j, out_s, counts, capacity, tri);
  // counts[1] = candidate count (device-side copy so the caller reads both with one transfer)
  VFP_CUDA(cudaMemcpyAsync(counts + 1, cand_count, 8, cudaMemcpyDeviceToDevice, st));
  VFP_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------
// flat inner-product top-k
// ---------------------------------------------------------------------------------------------
size_t vfp_topk_workspace_bytes_dim(int64_t n_q, int64_t n_db, int k, int dim) {
  return search_dim_ok(dim) ? topk_workspace_bytes(n_q, n_db, k, dim) : 0;
}
size_t vfp_topk_workspace_bytes(int64_t n_q, int64_t n_db, int k) { return topk_workspace_bytes(n_q, n_db, k, 256); }

int vfp_topk_ip(const float* q, const float* db, int64_t n_q, int64_t n_db, int dim, int k, float screen_margin,
                float* out_s, int64_t* out_idx, uint64_t* flags_out, void* workspace, size_t workspace_bytes,
                void* stream) {
  if (!q || !db || !out_s || !out_idx || !flags_out || !workspace) return fail("vfp_topk_ip: null argument");
  if (!search_dim_ok(dim))
    return fail("vfp_topk_ip: dim " + std::to_string(dim) + " is not supported (16 <= dim <= 512, dim % 16 == 0)");
  if (k <= 0 || k > 32) return fail("vfp_topk_ip: k must be in [1, 32]");
  if (n_q <= 0 || n_db <= 0) return fail("vfp_topk_ip: empty operand");
  if (n_db < k) return fail("vfp_topk_ip: k exceeds the number of database rows");
  if (n_q > 0x7fffff00LL || n_db > 0x7fffff00LL) return fail("vfp_topk_ip: more than 2^31 rows");
  if (workspace_bytes < topk_workspace_bytes(n_q, n_db, k, dim))
    return fail("vfp_topk_ip: workspace too small for dim " + std::to_string(dim) + "; see vfp_topk_workspace_bytes_dim");
  std::string err;
  const int rc = topk_run(q, db, n_q, n_db, dim, k, screen_margin, out_s, out_idx, reinterpret_cast<unsigned long long*>(flags_out),
                          static_cast<uint8_t*>(workspace), static_cast<cudaStream_t>(stream), &err);
  if (rc) return fail("vfp_topk_ip: " + err);
  return 0;
}

// ---------------------------------------------------------------------------------------------
// evaluation metrics over an embedding set (train.py:285-358, 439-481)
// ---------------------------------------------------------------------------------------------
int vfp_pair_scores(const float* e, int64_t n, int dim, const int32_t* pair_i, const int32_t* pair_j, int64_t m, float* out_s,
                    void* stream) {
  if (!e || (m > 0 && (!pair_i || !pair_j || !out_s))) return fail("vfp_pair_scores: null argument");
  if (n <= 0 || dim <= 0 || n > 0x7fffff00LL || m > 0x7fffff00LL) return fail("vfp_pair_scores: bad size");
  if (m == 0) return 0;
  pair_scores_kernel<<<(unsigned)((m + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(e, dim, pair_i, pair_j, (int)m, out_s);
  VFP_CUDA(cudaGetLastError());
  return 0;
}

int vfp_pair_stats(const float* e, const int32_t* video_ids, int64_t n, int dim, const int32_t* row_ptr, const int32_t* pos_idx,
                   const float* pos_score, const float* sorted_intra, int64_t m, const float* thresholds, int n_thresholds,
                   uint32_t* rank_greater, uint32_t* rank_tie_before, double* sums, uint64_t* counts, void* stream) {
  if (!e || !video_ids || !row_ptr || !sums || !counts) return fail("vfp_pair_stats: null argument");
  if (m > 0 && (!pos_idx || !pos_score || !sorted_intra || !rank_greater || !rank_tie_before)) return fail("vfp_pair_stats: null argument");
  if (n <= 0 || n > 0x7fffff00LL || m < 0 || m > 0x7fffff00LL) return fail("vfp_pair_stats: bad size");
  if (dim <= 0 || dim % kMsK != 0) return fail("vfp_pair_stats: dim must be a multiple of 16");
  if (n_thresholds < 0 || n_thresholds > kMsMaxThr || (n_thresholds > 0 && !thresholds)) return fail("vfp_pair_stats: at most 8 thresholds");
  if ((reinterpret_cast<uintptr_t>(e) & 15) != 0) return fail("vfp_pair_stats: embeddings must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  PairStatsParams p{};
  p.e = e; p.ids = video_ids; p.n = (int)n; p.dim = dim; p.row_ptr = row_ptr; p.pos_idx = pos_idx; p.pos_score = pos_score;
  p.sorted_intra = sorted_intra; p.m = (int)m; p.n_thr = n_thresholds;
  for (int t = 0; t < n_thresholds; ++t) p.thr[t] = thresholds[t];   // HOST array
  p.rank_greater = rank_greater; p.rank_tie_before = rank_tie_before; p.sums = sums;
  p.counts = reinterpret_cast<unsigned long long*>(counts);
  VFP_CUDA(cudaMemsetAsync(sums, 0, 4 * sizeof(double), st));
  VFP_CUDA(cudaMemsetAsync(counts, 0, (4 + 2 * kMsMaxThr) * sizeof(uint64_t), st));
  if (m > 0) {
    VFP_CUDA(cudaMemsetAsync(rank_greater, 0, (size_t)m * 4, st));
    VFP_CUDA(cudaMemsetAsync(rank_tie_before, 0, (size_t)m * 4, st));
  }
  const unsigned tiles = (unsigned)((n + kMsTile - 1) / kMsTile);
  pair_stats_kernel<<<dim3(tiles, tiles), 256, 0, st>>>(p);
  VFP_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------
// frame preprocessing (fingerprint.py:186-214): INTER_AREA resize of the short side to 64 + centre crop
// ---------------------------------------------------------------------------------------------
namespace {
// OpenCV computeResizeAreaTab (imgproc/src/resize.cpp), one destination axis, entries of destination indices [d0, d0 + 64)
void area_table(int ssize, int dsize, double scale, int d0, std::vector<int>* begin, std::vector<int>* si, std::vector<float>* alpha) {
  begin->assign(65, 0);
  si->clear();
  alpha->clear();
  for (int d = d0; d < d0 + 64; ++d) {
    (*begin)[d - d0] = (int)si->size();
    const double fsx1 = d * scale, fsx2 = fsx1 + scale;
    const double cell = std::min(scale, ssize - fsx1);
    int sx1 = (int)ceil(fsx1), sx2 = (int)floor(fsx2);
    sx2 = std::min(sx2, ssize - 1);
    sx1 = std::min(sx1, sx2);
    if (sx1 - fsx1 > 1e-3) { si->push_back(sx1 - 1); alpha->push_back((float)((sx1 - fsx1) / cell)); }
    for (int sx = sx1; sx < sx2; ++sx) { si->push_back(sx); alpha->push_back((float)(1.0 / cell)); }
    if (fsx2 - sx2 > 1e-3) { si->push_back(sx2); alpha->push_back((float)(std::min(std::min(fsx2 - sx2, 1.0), cell) / cell)); }
  }
  (*begin)[64] = (int)si->size();
}
// cv::resize's coefficient loop with area_mode = true, ksize = 2, 8-bit fixed point (imgproc/src/resize.cpp), destination
// indices [d0, d0 + 64): sx = cvFloor(dx * scale), fx = (float)((dx + 1) - (sx + 1) * inv_scale) reduced to [0, 1); at the last
// source sample the pair degenerates to (2048, 0); coefficients = saturate_cast<short>(c * 2048) (round half to even)
void linear_area_table(int ssize, int dsize, int d0, int* ofs, short (*coef)[2]) {
  const double inv_scale = (double)dsize / ssize, scale = 1.0 / inv_scale;
  for (int d = d0; d < d0 + 64; ++d) {
    int s = (int)floor(d * scale);
    float f = (float)((d + 1) - (s + 1) * inv_scale);
    f = f <= 0 ? 0.0f : f - floorf(f);
    if (s >= ssize - 1) { f = 0.0f; s = ssize - 1; }
    ofs[d - d0] = s;
    coef[d - d0][0] = (short)lrintf((1.0f - f) * 2048.0f);
    coef[d - d0][1] = (short)lrintf(f * 2048.0f);
  }
}
}  // namespace

size_t vfp_preprocess_workspace_bytes(int height, int width) {
  // tables: two axes x (65 ints + entries * (int + float)); an axis has at most 64 * (scale + 2) entries
  const size_t per_axis = 65 * 4 + (size_t)(64 * 2 + std::max(height, width) + 64) * 8;
  return 2 * per_axis + 256;
}

int vfp_preprocess_frames(const uint8_t* frames_hwc, int n_frames, int height, int width, uint8_t* out_hwc64, void* workspace,
                          size_t workspace_bytes, void* stream) {
  if (!frames_hwc || !out_hwc64 || !workspace) return fail("vfp_preprocess_frames: null argument");
  if (n_frames <= 0 || n_frames > 65535) return fail("vfp_preprocess_frames: 1 .. 65535 frames per call");
  if (height < 1 || width < 1) return fail("vfp_preprocess_frames: empty frames");
  if (workspace_bytes < vfp_preprocess_workspace_bytes(height, width)) return fail("vfp_preprocess_frames: workspace too small");
  // fingerprint.py:190-196
  int new_w, new_h;
  if (height < width) { new_h = 64; new_w = (int)((double)width * 64 / height); }
  else { new_w = 64; new_h = (int)((double)height * 64 / width); }
  if (height < 64 || width < 64) {   // a side below 64 px: both axes are up-scaled (preprocess_kernels.cuh, end of file)
    PreprocessUpParams up{};
    up.src = frames_hwc; up.dst = out_hwc64; up.H = height; up.W = width;
    linear_area_table(width, new_w, (new_w - 64) / 2, up.xo, up.xa);
    linear_area_table(height, new_h, (new_h - 64) / 2, up.yo, up.yb);
    preprocess_linear_kernel<<<dim3(64, (unsigned)n_frames), 192, 0, static_cast<cudaStream_t>(stream)>>>(up);
    VFP_CUDA(cudaGetLastError());
    return 0;
  }
  // cv::resize: inv_scale = dsize / ssize, scale = 1. / inv_scale (not ssize / dsize: the last bit can differ)
  const double scale_x = 1.0 / ((double)new_w / width), scale_y = 1.0 / ((double)new_h / height);
  const int start_h = (new_h - 64) / 2, start_w = (new_w - 64) / 2;   // fingerprint.py:201-202
  const int isx = (int)lrint(scale_x), isy = (int)lrint(scale_y);
  const bool fast = fabs(scale_x - isx) < 2.220446049250313e-16 && fabs(scale_y - isy) < 2.220446049250313e-16;
  std::vector<int> xb, xs, yb, ys;
  std::vector<float> xa, ya;
  if (fast) {   // integer box: every source column / row of the box with weight 1
    xb.resize(65); yb.resize(65);
    for (int d = 0; d <= 64; ++d) { xb[d] = d * isx; yb[d] = d * isy; }
    for (int d = 0; d < 64; ++d) {
      for (int k = 0; k < isx; ++k) { xs.push_back((start_w + d) * isx + k); xa.push_back(1.0f); }
      for (int k = 0; k < isy; ++k) { ys.push_back((start_h + d) * isy + k); ya.push_back(1.0f); }
    }
  } else {
    area_table(width, new_w, scale_x, start_w, &xb, &xs, &xa);
    area_table(height, new_h, scale_y, start_h, &yb, &ys, &ya);
  }
  int sx_min = xs[0], sx_max = xs[0];
  for (int v : xs) { sx_min = std::min(sx_min, v); sx_max = std::max(sx_max, v); }
  PreprocessParams p{};
  p.sx_min = sx_min; p.sx_count = sx_max - sx_min + 1;
  if (p.sx_count * 3 > kPreMaxSpan) return fail("vfp_preprocess_frames: scale factor too large (source span of one output row exceeds 8192 bytes)");
  // pack the tables into one host buffer -> one copy
  std::vector<int32_t> host;
  auto put_i = [&](const std::vector<int>& v) { size_t o = host.size(); host.insert(host.end(), v.begin(), v.end()); return o; };
  auto put_f = [&](const std::vector<float>& v) { size_t o = host.size(); host.resize(o + v.size()); memcpy(host.data() + o, v.data(), v.size() * 4); return o; };
  const size_t o_xb = put_i(xb), o_xs = put_i(xs), o_xa = put_f(xa), o_yb = put_i(yb), o_ys = put_i(ys), o_ya = put_f(ya);
  if (host.size() * 4 > workspace_bytes) return fail("vfp_preprocess_frames: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int32_t* dev = static_cast<int32_t*>(workspace);
  VFP_CUDA(cudaMemcpyAsync(dev, host.data(), host.size() * 4, cudaMemcpyHostToDevice, st));   // pageable source: staged before return
  p.src = frames_hwc; p.dst = out_hwc64; p.H = height; p.W = width;
  p.mode = fast ? ((isx == 2 && isy == 2) ? 2 : 1) : 0;
  p.inv_area = (float)(1.0 / (isx * isy));
  p.x_begin = dev + o_xb; p.x_si = dev + o_xs; p.x_alpha = reinterpret_cast<const float*>(dev + o_xa);
  p.y_begin = dev + o_yb; p.y_si = dev + o_ys; p.y_beta = reinterpret_cast<const float*>(dev + o_ya);
  const size_t pre_smem = (size_t)kPreRowsPerStage * ((p.sx_count * 3 + 32 + 15) & ~15);
  VFP_CUDA(ensure_dynamic_smem(reinterpret_cast<const void*>(preprocess_area_kernel), kPreRowsPerStage * (kPreMaxSpan + 48)));
  preprocess_area_kernel<<<dim3(64, (unsigned)n_frames), 192, pre_smem, st>>>(p);
  VFP_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------
// VideoFingerprint3D (model.py:406-512): the reference's second model behind create_model("3d" | "cnn3d")
// ---------------------------------------------------------------------------------------------
}  // extern "C"

struct vfp3d_weights {
  int fs = 0, embedding_dim = 0;
  int kp[4] = {0, 0, 0, 0};            // padded K of the four conv GEMMs
  __nv_bfloat16* w[4] = {nullptr, nullptr, nullptr, nullptr};   // [Np][Kp] K-major, BN folded
  float* b[4] = {nullptr, nullptr, nullptr, nullptr};           // [Np]
  uint2* l1_pack = nullptr;   // layer 1 as mma.sync B fragments (conv3d_l1_kernel)
  CUtensorMap tm[4];
  float *tc_w = nullptr, *tc_b = nullptr, *ta_w = nullptr, *ta_b = nullptr, *p0_w = nullptr, *p0_b = nullptr, *p3_w = nullptr, *p3_b = nullptr;
  std::vector<void*> allocs;
};

namespace {
constexpr int k3dCin[4] = {3, 16, 32, 64}, k3dCout[4] = {16, 32, 64, 128};
constexpr int k3dCinPad[4] = {3, 32, 32, 64}, k3dNp[4] = {32, 32, 64, 128};   // channel counts as stored (padded to the 32-column store box)

template <class T>
int upload3d(vfp3d_weights* w, const std::vector<T>& host, T** dev) {
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, host.size() * sizeof(T));
  if (e != cudaSuccess) return fail_cuda("cudaMalloc", e);
  w->allocs.push_back(p);
  e = cudaMemcpy(p, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) return fail_cuda("cudaMemcpy", e);
  *dev = static_cast<T*>(p);
  return 0;
}
// temporal positions of one clip of T frames: G groups of fs frames after layer 1 (and 2), T3 after the stride-2 layer 3
struct Dims3d { int G, T3; };
Dims3d dims3d(int T, int fs) {
  Dims3d d;
  d.G = (T + fs - 1) / fs;
  d.T3 = (d.G - 1) / 2 + 1;
  return d;
}
// Workspace of one packed pass whose clips sum to sG groups and sT3 layer-3 positions:
// [tables][im2col matrix A (layers 2-4, reused)][act 0][act 1][act 2][act 3]. Tables, in int32 units: layer-1 groups (L1Group,
// 16 bytes, x sG), the im2col slots of layers 2, 3, 4 (int4 x sG, sT3, sT3) and the head's clips (int2 x C).
struct Ws3d {
  long long m[4];             // packed rows of the four conv layers
  size_t t_slots[3], t_head;  // table offsets (int32 units)
  size_t tables, a, act[4], total;   // byte offsets / sizes
};
Ws3d ws3d(const vfp3d_weights* w, long long sG, long long sT3, long long C) {
  Ws3d L;
  L.m[0] = sG * 1024; L.m[1] = sG * 256; L.m[2] = sT3 * 64; L.m[3] = sT3 * 16;
  L.t_slots[0] = (size_t)sG * 4;
  L.t_slots[1] = L.t_slots[0] + (size_t)sG * 4;
  L.t_slots[2] = L.t_slots[1] + (size_t)sT3 * 4;
  L.t_head = L.t_slots[2] + (size_t)sT3 * 4;
  L.tables = align_up((L.t_head + (size_t)C * 2) * 4, 1024);
  size_t a_bytes = 0;
  for (int l = 1; l < 4; ++l) a_bytes = std::max(a_bytes, align_up((size_t)L.m[l] * w->kp[l] * 2, 1024));   // layer 1 needs no im2col matrix
  L.a = L.tables;
  size_t off = L.a + a_bytes;
  for (int l = 0; l < 4; ++l) { L.act[l] = off; off += align_up((size_t)L.m[l] * k3dNp[l] * 2, 1024); }
  L.total = off + 1024;
  return L;
}

size_t frame_bytes3d(int frame_dtype) {
  return (size_t)12288 * (frame_dtype == VFP_FRAME_BF16 ? 2 : frame_dtype == VFP_FRAME_F32 ? 4 : 1);
}

// One packed pass: clips [c0, c1) of the input, clip i = len[i] frames from device address clip[i].
int forward3d_pass(const vfp3d_weights* w, int frame_dtype, const void* const* clip, const int32_t* len, int c0, int c1,
                   float* emb_out, uint8_t* ws, cudaStream_t st) {
  const int C = c1 - c0, fs = w->fs;
  const size_t frame_bytes = frame_bytes3d(frame_dtype);
  long long sG = 0, sT3 = 0;
  for (int i = c0; i < c1; ++i) { const Dims3d d = dims3d(len[i], fs); sG += d.G; sT3 += d.T3; }
  const Ws3d L = ws3d(w, sG, sT3, C);
  // the per-pass tables (pageable host memory: the copy is staged before cudaMemcpyAsync returns, so the vector may go)
  std::vector<int32_t> tab(L.t_head + (size_t)C * 2, 0);
  int32_t* groups = tab.data();
  int32_t* slots[3] = {tab.data() + L.t_slots[0], tab.data() + L.t_slots[1], tab.data() + L.t_slots[2]};
  int32_t* head = tab.data() + L.t_head;
  long long gb = 0, tb = 0;   // first group / layer-3 position of the clip in the pass
  for (int i = c0; i < c1; ++i) {
    const int T = len[i];
    const Dims3d d = dims3d(T, fs);
    for (int g = 0; g < d.G; ++g) {   // L1Group {first frame of the group, frames left in the clip, 0}
      const void* first = static_cast<const uint8_t*>(clip[i]) + (size_t)g * fs * frame_bytes;
      memcpy(groups + (gb + g) * 4, &first, sizeof(first));
      groups[(gb + g) * 4 + 2] = T - g * fs;
    }
    auto slot = [](int32_t* s, long long in_base, int Ti, int t0) { s[0] = (int32_t)in_base; s[1] = Ti; s[2] = t0; s[3] = 0; };
    for (int to = 0; to < d.G; ++to) slot(slots[0] + (gb + to) * 4, gb, d.G, to - 1);         // layer 2: G -> G, stride 1
    for (int to = 0; to < d.T3; ++to) slot(slots[1] + (tb + to) * 4, gb, d.G, 2 * to - 1);    // layer 3: G -> T3, stride 2
    for (int to = 0; to < d.T3; ++to) slot(slots[2] + (tb + to) * 4, tb, d.T3, to - 1);       // layer 4: T3 -> T3, stride 1
    head[(i - c0) * 2] = (int32_t)tb; head[(i - c0) * 2 + 1] = d.T3;
    gb += d.G; tb += d.T3;
  }
  VFP_CUDA(cudaMemcpyAsync(ws, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice, st));
  const int32_t* dtab = reinterpret_cast<const int32_t*>(ws);
  __nv_bfloat16* A = reinterpret_cast<__nv_bfloat16*>(ws + L.a);
  __nv_bfloat16* act[4];
  for (int l = 0; l < 4; ++l) act[l] = reinterpret_cast<__nv_bfloat16*>(ws + L.act[l]);
  for (int l = 0; l < 4; ++l) {
    if (l == 0) {   // layer 1 straight from the frames on the register-fragment tensor path, no im2col matrix
      const size_t smem = (((size_t)fs * 5 * 204 * 2 + 4 + 15) & ~size_t(15)) + 4 * 16 * 32 * 4;
      VFP_CUDA(ensure_dynamic_smem(reinterpret_cast<const void*>(conv3d_l1_kernel), 64 * 5 * 204 * 2 + 32 + 4 * 16 * 32 * 4));
      conv3d_l1_kernel<<<(unsigned)(sG * 32), 128, smem, st>>>(frame_dtype, reinterpret_cast<const L1Group*>(dtab), fs, w->l1_pack,
                                                             w->b[0], act[0]);
      continue;
    }
    const long long items = L.m[l] * (w->kp[l] / 8);
    const unsigned grid = (unsigned)std::min<long long>((items + 255) / 256, (long long)device_sm_count() * 32);
    const int Hi = 64 >> l;
    im2col3d_ndhwc_kernel<<<grid, 256, 0, st>>>(act[l - 1], reinterpret_cast<const int4*>(dtab + L.t_slots[l - 1]), l == 1 ? sG : sT3,
                                                Hi, Hi, k3dCinPad[l], Hi / 2, Hi / 2, w->kp[l], A);
    CUtensorMap ta;
    if (make_tmap_rows_bf16(&ta, A, (uint64_t)L.m[l], (uint64_t)w->kp[l], (uint64_t)w->kp[l], 128, 64)) return fail("vfp3d_forward: tensor map encode failed (A)");
    EpiBiasActTma<true>::Params ep{};
    if (make_tmap_out(&ep.tmap_out, act[l], (uint64_t)L.m[l], (uint64_t)k3dNp[l], true)) return fail("vfp3d_forward: tensor map encode failed (out)");
    ep.bias = w->b[l]; ep.N = k3dNp[l]; ep.act = 1;
    GemmShape s = plain_shape(L.m[l], k3dNp[l], w->kp[l], k3dNp[l], 64, 32);
    if (l <= 1) VFP_CUDA((launch_gemm<32, 64, 4, EpiBiasActTma<true>>(ta, w->tm[l], s, ep, st)));
    else if (l == 2) VFP_CUDA((launch_gemm<64, 64, 4, EpiBiasActTma<true>>(ta, w->tm[l], s, ep, st)));
    else VFP_CUDA((launch_gemm<128, 64, 4, EpiBiasActTma<true>>(ta, w->tm[l], s, ep, st)));
  }
  Head3dParams hp{};
  hp.act = act[3]; hp.clips = reinterpret_cast<const int2*>(dtab + L.t_head);
  hp.tc_w = w->tc_w; hp.tc_b = w->tc_b; hp.ta_w = w->ta_w; hp.ta_b = w->ta_b;
  hp.p0_w = w->p0_w; hp.p0_b = w->p0_b; hp.p3_w = w->p3_w; hp.p3_b = w->p3_b; hp.D = w->embedding_dim;
  hp.out = emb_out + (size_t)c0 * w->embedding_dim;
  head3d_kernel<<<(unsigned)C, 128, 0, st>>>(hp);
  VFP_CUDA(cudaGetLastError());
  return 0;
}

// The one planner of the 3-D model: checks clip i = len[i] frames at device address clip[i] (any placement: packed, separate
// allocations, overlapping, aliased) and runs the clips in passes cut on clip boundaries, each as large as the workspace holds.
int forward3d_clips(const std::string& name, const vfp3d_weights* w, const void* const* clip, const int32_t* len, int n_clips,
                    int frame_dtype, float* emb_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!w || !clip || !len || !emb_out || !workspace) return fail(name + ": null argument");
  if (n_clips <= 0) return fail(name + ": n_clips must be positive");
  if (frame_dtype != VFP_FRAME_U8 && frame_dtype != VFP_FRAME_BF16 && frame_dtype != VFP_FRAME_F32 && frame_dtype != VFP_FRAME_U8_HWC)
    return fail(name + ": unknown frame_dtype " + std::to_string(frame_dtype));
  for (int i = 0; i < n_clips; ++i) {
    const int T = len[i];
    if (T <= 0) return fail(name + ": clip " + std::to_string(i) + " has length " + std::to_string(T));
    if (!clip[i]) return fail(name + ": clip " + std::to_string(i) + " has a null frame pointer");
    if (reinterpret_cast<uintptr_t>(clip[i]) % 16)
      return fail(name + ": clip " + std::to_string(i) + "'s frame pointer is not 16-byte aligned (the frames are read in 16-byte vectors)");
    const Dims3d d = dims3d(T, w->fs);
    if (d.T3 > kHead3dMaxT)
      return fail(name + ": clip " + std::to_string(i) + " too long: " + std::to_string(T) + " frames give " + std::to_string(d.T3) +
                  " temporal positions after the strides (at most 32, i.e. " + std::to_string(64 * w->fs) + " frames)");
    const size_t need = ws3d(w, d.G, d.T3, 1).total;
    if (need > workspace_bytes)
      return fail(name + ": workspace of " + std::to_string(workspace_bytes) + " bytes is too small for clip " + std::to_string(i) + " (" +
                  std::to_string(T) + " frames need " + std::to_string(need) + ")");
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (int c0 = 0; c0 < n_clips;) {
    int c1 = c0;   // every clip fits on its own (checked above): add clips while the pass still fits
    long long sG = 0, sT3 = 0;
    while (c1 < n_clips) {
      const Dims3d d = dims3d(len[c1], w->fs);
      if (c1 > c0 && ws3d(w, sG + d.G, sT3 + d.T3, c1 - c0 + 1).total > workspace_bytes) break;
      sG += d.G; sT3 += d.T3; ++c1;
    }
    if (int rc = forward3d_pass(w, frame_dtype, clip, len, c0, c1, emb_out, static_cast<uint8_t*>(workspace), st)) return rc;
    c0 = c1;
  }
  return 0;
}

// A packed input (clips back to back, prefix sums cu): the clip pointers are frames + cu[i] frames.
int forward3d_packed(const char* who, const vfp3d_weights* w, const void* frames, int frame_dtype, const int32_t* cu, int n_clips,
                     float* emb_out, void* workspace, size_t workspace_bytes, void* stream) {
  const std::string name(who);
  if (!w || !frames || !cu || !emb_out || !workspace) return fail(name + ": null argument");
  if (n_clips <= 0) return fail(name + ": n_clips must be positive");
  if (frame_dtype == VFP_FRAME_U8_HWC) return fail(name + ": decoder-layout (HWC) frames are not supported here; pass planar (T, 3, 64, 64) frames, or use vfp3d_forward_clips");
  if (frame_dtype != VFP_FRAME_U8 && frame_dtype != VFP_FRAME_BF16 && frame_dtype != VFP_FRAME_F32) return fail(name + ": planar u8 / bf16 / fp32 frames only");
  if (cu[0] != 0) return fail(name + ": cu_seqlens[0] must be 0");
  const size_t frame_bytes = frame_bytes3d(frame_dtype);
  std::vector<const void*> clip((size_t)n_clips);
  std::vector<int32_t> len((size_t)n_clips);
  for (int i = 0; i < n_clips; ++i) {
    if (cu[i + 1] < cu[i]) return fail(name + ": cu_seqlens is not monotone (decreases at clip " + std::to_string(i) + ")");
    clip[i] = static_cast<const uint8_t*>(frames) + (size_t)cu[i] * frame_bytes;
    len[i] = cu[i + 1] - cu[i];
  }
  return forward3d_clips(name, w, clip.data(), len.data(), n_clips, frame_dtype, emb_out, workspace, workspace_bytes, stream);
}
}  // namespace

extern "C" {

void vfp3d_weights_destroy(vfp3d_weights* w) {
  if (!w) return;
  for (void* p : w->allocs) cudaFree(p);
  delete w;
}
int vfp3d_weights_embedding_dim(const vfp3d_weights* w) { return w ? w->embedding_dim : 0; }

int vfp3d_weights_create(const vfp_tensor_desc* tensors, int n_tensors, int frame_stride, vfp3d_weights** out) {
  if (!tensors || !out || n_tensors <= 0) return fail("vfp3d_weights_create: null argument");
  if (frame_stride < 1 || frame_stride > 64) return fail("vfp3d_weights_create: frame_stride must be in [1, 64]");
  TensorTable t;
  for (int i = 0; i < n_tensors; ++i) t.by_name[tensors[i].name] = &tensors[i];
  std::string err;
  vfp3d_weights* w = new vfp3d_weights();
  auto bail = [&](const std::string& m) {
    vfp3d_weights_destroy(w);
    return fail("vfp3d_weights_create: " + (m.empty() ? g_last_error : m));
  };
  w->fs = frame_stride;
  for (int l = 0; l < 4; ++l) {
    const std::string pre = "encoder." + std::to_string(l);
    const int kt = l == 0 ? frame_stride : 3, ks = l == 0 ? 5 : 3, cin = k3dCin[l], cout = k3dCout[l], cpad = k3dCinPad[l];
    const int taps = kt * ks * ks;
    const float* cw = t.get(pre + ".conv.weight", (int64_t)cout * cin * taps, &err);
    const float* cb = cw ? t.get(pre + ".conv.bias", cout, &err) : nullptr;
    if (!cb) return bail(err);
    // eval-mode BatchNorm3d folded (the tensors are named .bn.* here, not encoder.N like the attention model)
    BnFold bn;
    if (!load_bn(t, pre + ".bn", cout, &bn, &err)) return bail(err);
    // layer 0: per (kt, kh) a run of 16 = (kw, c) taps + 1 zero (im2col3d_frames_kernel); layers 1-3: k = tap * cpad + c
    const int kreal = l == 0 ? kt * 5 * 16 : taps * cpad;
    w->kp[l] = (kreal + 63) / 64 * 64;
    std::vector<float> wf((size_t)k3dNp[l] * w->kp[l], 0.0f), bf(k3dNp[l], 0.0f);
    for (int co = 0; co < cout; ++co) {
      for (int c = 0; c < cin; ++c)
        for (int tap = 0; tap < taps; ++tap) {   // reference layout (cout, cin, kt, kh, kw), tap = (kt*ks + kh)*ks + kw
          const size_t k = l == 0 ? (size_t)(tap / 5) * 16 + (size_t)(tap % 5) * 3 + c : (size_t)tap * cpad + c;
          wf[(size_t)co * w->kp[l] + k] = cw[((size_t)co * cin + c) * taps + tap] * bn.scale[co];
        }
      bf[co] = cb[co] * bn.scale[co] + bn.shift[co];
    }
    if (upload3d(w, to_bf16(wf), &w->w[l]) || upload3d(w, bf, &w->b[l])) return bail("");
    if (l == 0) {   // B fragments of mma.sync m16n8k16 per K run of 16: lane (g, tig) holds W[n = nt*8 + g][k0 + 2tig, +1] and [.. + 8, + 9]
      const int n_runs = kt * 5;
      std::vector<uint2> pack((size_t)n_runs * 2 * 32);
      auto bf16bits = [](float x) { __nv_bfloat16 h = __float2bfloat16(x); uint16_t u; memcpy(&u, &h, 2); return (uint32_t)u; };
      for (int run = 0; run < n_runs; ++run)
        for (int nt = 0; nt < 2; ++nt)
          for (int lane = 0; lane < 32; ++lane) {
            const int g = lane >> 2, tig = lane & 3, co = nt * 8 + g;
            const float* row = wf.data() + (size_t)co * w->kp[0] + (size_t)run * 16 + 2 * tig;
            pack[((size_t)run * 2 + nt) * 32 + lane] = make_uint2(bf16bits(row[0]) | (bf16bits(row[1]) << 16), bf16bits(row[8]) | (bf16bits(row[9]) << 16));
          }
      if (upload3d(w, pack, &w->l1_pack)) return bail("");
    }
    if (make_tmap_rows_bf16(&w->tm[l], w->w[l], (uint64_t)k3dNp[l], (uint64_t)w->kp[l], (uint64_t)w->kp[l], (uint32_t)std::min(k3dNp[l], 256), 64))
      return bail("tensor map encode failed");
  }
  auto f32 = [&](const std::string& name, int64_t n, float** dev) -> bool {
    const float* src = t.get(name, n, &err);
    if (!src) return false;
    std::vector<float> h(src, src + n);
    return upload3d(w, h, dev) == 0;
  };
  const int64_t d = t.numel("projector.3.bias");
  if (d <= 0 || d > 512) return bail("projector.3.bias missing or embedding_dim > 512");
  w->embedding_dim = (int)d;
  if (!f32("temporal_conv.weight", 128 * 128 * 3, &w->tc_w) || !f32("temporal_conv.bias", 128, &w->tc_b) ||
      !f32("temporal_attention.weight", 128, &w->ta_w) || !f32("temporal_attention.bias", 1, &w->ta_b) ||
      !f32("projector.0.weight", 128 * 128, &w->p0_w) || !f32("projector.0.bias", 128, &w->p0_b) ||
      !f32("projector.3.weight", d * 128, &w->p3_w) || !f32("projector.3.bias", d, &w->p3_b))
    return bail(err);
  *out = w;
  return 0;
}

size_t vfp3d_forward_workspace_bytes(const vfp3d_weights* w, int64_t clips_per_pass, int n_frames) {
  if (!w || clips_per_pass <= 0 || n_frames <= 0) return 0;
  const Dims3d d = dims3d(n_frames, w->fs);
  return ws3d(w, clips_per_pass * d.G, clips_per_pass * d.T3, clips_per_pass).total;
}

size_t vfp3d_forward_packed_workspace_bytes(const vfp3d_weights* w, int64_t frames_per_pass, int64_t clips_per_pass) {
  if (!w || frames_per_pass <= 0 || clips_per_pass <= 0) return 0;
  const int64_t C = std::min(clips_per_pass, frames_per_pass);                  // a clip has at least one frame
  const int64_t G = std::min(frames_per_pass, frames_per_pass / w->fs + C);     // sum ceil(T/fs) <= F/fs + C, and <= F
  const int64_t T3 = std::min(G, (G + C) / 2);                                  // sum ceil(G/2) <= (sum G + C) / 2
  return ws3d(w, G, T3, C).total;
}

// The equal-length batch is the packed path with uniform clip lengths: one kernel set, one indexing scheme.
int vfp3d_forward(const vfp3d_weights* w, const void* frames, int frame_dtype, int64_t n_clips, int n_frames, float* emb_out,
                  void* workspace, size_t workspace_bytes, void* stream) {
  if (!w || !frames || !emb_out || !workspace) return fail("vfp3d_forward: null argument");
  if (n_clips <= 0 || n_frames <= 0) return fail("vfp3d_forward: empty input");
  if (n_clips > INT32_MAX || n_clips * (int64_t)n_frames > INT32_MAX) return fail("vfp3d_forward: more than 2^31 - 1 frames in one call");
  std::vector<int32_t> cu((size_t)n_clips + 1);
  for (int64_t i = 0; i <= n_clips; ++i) cu[i] = (int32_t)(i * n_frames);
  return forward3d_packed("vfp3d_forward", w, frames, frame_dtype, cu.data(), (int)n_clips, emb_out, workspace, workspace_bytes, stream);
}

int vfp3d_forward_packed(const vfp3d_weights* w, const void* frames, int frame_dtype, const int32_t* cu_seqlens_host, int n_clips,
                         float* emb_out, void* workspace, size_t workspace_bytes, void* stream) {
  return forward3d_packed("vfp3d_forward_packed", w, frames, frame_dtype, cu_seqlens_host, n_clips, emb_out, workspace, workspace_bytes,
                          stream);
}

int vfp3d_forward_clips(const vfp3d_weights* w, const void* const* clip_frames_host, const int32_t* lengths_host, int n_clips,
                        int frame_dtype, float* emb_out, void* workspace, size_t workspace_bytes, void* stream) {
  return forward3d_clips("vfp3d_forward_clips", w, clip_frames_host, lengths_host, n_clips, frame_dtype, emb_out, workspace,
                         workspace_bytes, stream);
}

}  // extern "C"
