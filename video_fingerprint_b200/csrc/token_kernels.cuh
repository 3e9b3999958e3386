// Token-stream kernels of the temporal encoder that are NOT dense contractions: clip bookkeeping,
// LayerNorm, the grouped multi-scale temporal convolution, self-attention over one clip, the three-way
// temporal pooling and the final projection + L2 normalisation. Tokens of all clips are PACKED
// ([sum T][256], clip v owns rows cu[v] .. cu[v+1]) - there is no padding, so the reference's B=1
// semantics for variable-length clips (fingerprint.py:244-249) hold by construction: the temporal conv
// zero-pads at clip ends, attention/pooling only ever see a clip's own rows.
#pragma once
#include "sm100_primitives.cuh"
#include "epilogues.cuh"

namespace vfp {

constexpr int kDim = 256;      // temporal_dim
constexpr int kHeads = 8;
constexpr int kHeadDim = 32;

// ---------------------------------------------------------------------------------------------
// token -> (clip, position) maps from the prefix sums, and the frame address table of the pass
// ---------------------------------------------------------------------------------------------
// Where a clip's frames are: frame t of the clip starts at addr + t * pitch (bytes). Clips may sit anywhere in device memory.
struct FrameSrc {
  unsigned long long addr;
  long long pitch;
};

// Token t of the pass is frame tok_pos[t] of clip v; frame_addr[t] receives that frame's device address, which is all the
// frame encoder's loaders read (the frames themselves need not be packed).
__global__ void token_map_kernel(const int* __restrict__ cu, const FrameSrc* __restrict__ src, int n_clips, int n_tokens,
                                 int* __restrict__ tok_pos, int* __restrict__ tok_len, unsigned long long* __restrict__ frame_addr) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_tokens) return;
  int lo = 0, hi = n_clips;  // find v with cu[v] <= t < cu[v+1]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (cu[mid] <= t) lo = mid; else hi = mid;
  }
  const int pos = t - cu[lo];
  tok_pos[t] = pos;
  tok_len[t] = cu[lo + 1] - cu[lo];
  const FrameSrc s = src[lo];
  frame_addr[t] = s.addr + (unsigned long long)((long long)pos * s.pitch);
}

// ---------------------------------------------------------------------------------------------
// v = (x + delta_a) + delta_f ; y = LayerNorm(v) over 256 channels; x = v if write_x. fp32 residual stream, bf16 normalised
// copy out. The residual GEMMs (attention out-projection, MLP down-projection) emit their result as bf16 deltas through the
// TMA store path; the add into the fp32 stream happens here, where the row is being read anyway, instead of in the GEMM
// epilogue (whose row-per-thread layout makes fp32 read-modify-write uncoalesced). The stream is only WRITTEN once per block:
// a block's second LayerNorm (before the MLP) normalises x + delta_a without storing it, and the next block's first
// LayerNorm adds both deltas in the same order - the bits of the stream are what two stores per block gave, for 1 KB per
// token and block less traffic. One warp per token, 8 channels per lane.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
add_layernorm_bf16_kernel(float* __restrict__ x, const __nv_bfloat16* __restrict__ delta /*nullable*/,
                          const __nv_bfloat16* __restrict__ delta2 /*nullable, added after delta*/,
                          const float* __restrict__ gamma, const float* __restrict__ beta, __nv_bfloat16* __restrict__ y,
                          int n_tokens, int write_x) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= n_tokens) return;
  float4* xr = reinterpret_cast<float4*>(x + (size_t)warp * kDim) + lane * 2;
  const float4 a = xr[0], b = xr[1];
  float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  if (delta) {
    const uint4 d = reinterpret_cast<const uint4*>(delta + (size_t)warp * kDim)[lane];
    const __nv_bfloat162* dp = reinterpret_cast<const __nv_bfloat162*>(&d);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = __bfloat1622float2(dp[e]);
      v[2 * e] += f.x;
      v[2 * e + 1] += f.y;
    }
    if (delta2) {
      const uint4 d2 = reinterpret_cast<const uint4*>(delta2 + (size_t)warp * kDim)[lane];
      const __nv_bfloat162* dp2 = reinterpret_cast<const __nv_bfloat162*>(&d2);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 f = __bfloat1622float2(dp2[e]);
        v[2 * e] += f.x;
        v[2 * e + 1] += f.y;
      }
    }
    if (write_x) {
      xr[0] = make_float4(v[0], v[1], v[2], v[3]);
      xr[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += v[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s * (1.0f / kDim);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) { v[i] -= mean; q += v[i] * v[i]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = rsqrtf(q * (1.0f / kDim) + 1e-5f);
  const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma) + lane * 2);
  const float4 g1 = __ldg(reinterpret_cast<const float4*>(gamma) + lane * 2 + 1);
  const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta) + lane * 2);
  const float4 b1 = __ldg(reinterpret_cast<const float4*>(beta) + lane * 2 + 1);
  uint4 o;
  o.x = pack_bf16x2(v[0] * rstd * g0.x + b0.x, v[1] * rstd * g0.y + b0.y);
  o.y = pack_bf16x2(v[2] * rstd * g0.z + b0.z, v[3] * rstd * g0.w + b0.w);
  o.z = pack_bf16x2(v[4] * rstd * g1.x + b1.x, v[5] * rstd * g1.y + b1.y);
  o.w = pack_bf16x2(v[6] * rstd * g1.z + b1.z, v[7] * rstd * g1.w + b1.w);
  reinterpret_cast<uint4*>(y + (size_t)warp * kDim)[lane] = o;
}

// x = (x + delta) + delta2 ; xbf = bf16(x): closes the last attention block and feeds the pooling GEMM. 8 channels per thread.
__global__ void __launch_bounds__(256)
add_convert_bf16_kernel(float* __restrict__ x, const __nv_bfloat16* __restrict__ delta /*nullable*/,
                        const __nv_bfloat16* __restrict__ delta2 /*nullable, added after delta*/, __nv_bfloat16* __restrict__ xbf,
                        long long n8) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n8) return;
  float4* xr = reinterpret_cast<float4*>(x) + 2 * i;
  const float4 a = xr[0], b = xr[1];
  float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  if (delta) {
    const uint4 d = reinterpret_cast<const uint4*>(delta)[i];
    const __nv_bfloat162* dp = reinterpret_cast<const __nv_bfloat162*>(&d);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = __bfloat1622float2(dp[e]);
      v[2 * e] += f.x;
      v[2 * e + 1] += f.y;
    }
    if (delta2) {
      const uint4 d2 = reinterpret_cast<const uint4*>(delta2)[i];
      const __nv_bfloat162* dp2 = reinterpret_cast<const __nv_bfloat162*>(&d2);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 f = __bfloat1622float2(dp2[e]);
        v[2 * e] += f.x;
        v[2 * e + 1] += f.y;
      }
    }
    xr[0] = make_float4(v[0], v[1], v[2], v[3]);
    xr[1] = make_float4(v[4], v[5], v[6], v[7]);
  }
  uint4 o;
  o.x = pack_bf16x2(v[0], v[1]); o.y = pack_bf16x2(v[2], v[3]);
  o.z = pack_bf16x2(v[4], v[5]); o.w = pack_bf16x2(v[6], v[7]);
  reinterpret_cast<uint4*>(xbf)[i] = o;
}

// ---------------------------------------------------------------------------------------------
// TemporalConvBlock + residual:  y = x + relu(bn(groupedconv_k(x)))  for k in {3,5,7,11} concatenated.
// Output channel o (branch o/64, group o%64) reads input channels 4*(o%64) .. +3 (model.py:163-169), so the four
// branches of group g share one 4-channel input window. Thread = (group g, 8 consecutive tokens); it produces the
// group's 4 outputs per token (one per branch) with the REAL tap counts 3/5/7/11 = 104 FMAs per token - no padded taps,
// and the input is read once instead of once per branch. Tap-major: per tap the (at most 4) weight vectors of the group
// are read once from shared memory (one float4 = the 4 input channels, BN folded) and one new input row enters an 8-row
// register window: 18 + 26 LDS.128 for 832 FMAs. Tokens of all clips are packed; an 11-bit mask per token says which taps
// stay inside the token's own clip (zero padding of Conv1d(padding=k//2) on a B=1 clip).
//
// A persistent CTA walks tiles of 32 tokens. The 42 rows a tile needs (5 rows of halo either side, rows outside the buffer
// zero-filled by TMA) arrive as ONE 42 KB TMA box in a double-buffered shared-memory tile while the previous tile is
// computed; the producer warp also works out the tile's tap masks; the folded weights are staged once per CTA.
// History: a first version loaded its rows just in time from global memory (4 tokens per thread, weights re-staged per
// 128 tokens): 0.99 ms per 10 000 clips against 0.81 ms now; ncu of both shows an issue-bound kernel (the shared-memory
// port carries 34 %, DRAM 29 %), i.e. what is left is instruction count: the scalar residual loads / stores and addressing.
// ---------------------------------------------------------------------------------------------
constexpr int kTc2Tok = 32;                       // tokens per tile
constexpr int kTc2Rows = kTc2Tok + 10;            // with halo
constexpr int kTc2TileBytes = kTc2Rows * kDim * 4;   // 43 008
constexpr int kTc2Threads = 256 + 32;             // 8 compute warps + the producer warp
constexpr int kTc2SmemBytes = 26 * 64 * 16 + 2 * kTc2TileBytes + 2 * 128 + 64 + 128;

struct TemporalConvParams {
  alignas(64) CUtensorMap tmap_x;   // x [tokens][256] fp32, box 256 columns x 42 rows, no swizzle
  const int* tok_pos;
  const int* tok_len;
  const float* w;      // [4][11][256]
  const float* bias;   // [256]
  float* y;
  int n_tokens;
  int n_tiles;
};

// 8 tokens x 4 branches of one group, one FFMA per multiply-add. kMasked (a token within 5 of an end of its clip is among the
// 8): the input values of a tap outside the clip are ANDed to zero, so the masked path has no branches and gives a token
// with all taps valid exactly the bits the unmasked path gives it - a token's result must not depend on which tokens it
// shares its slice with (weights are finite, so fma(w, 0, acc) = acc).
template <bool kMasked>
__device__ __forceinline__ void temporal_conv_oct(const float* __restrict__ xt /*tile row of the first token's tap 0*/, const float4 (*ws)[64], int g,
                                                  const unsigned (&mask)[8], float (&acc)[8][4]) {
  float4 rows[8];
#pragma unroll
  for (int i = 0; i < 7; ++i) rows[i] = *reinterpret_cast<const float4*>(xt + i * kDim + 4 * g);
#pragma unroll
  for (int tap = 0; tap < 11; ++tap) {
    rows[(tap + 7) & 7] = *reinterpret_cast<const float4*>(xt + (tap + 7) * kDim + 4 * g);
    const float4 w3 = ws[15 + tap][g];
    float4 w2 = w3, w1 = w3, w0 = w3;
    if (tap >= 2 && tap <= 8) w2 = ws[8 + tap - 2][g];
    if (tap >= 3 && tap <= 7) w1 = ws[3 + tap - 3][g];
    if (tap >= 4 && tap <= 6) w0 = ws[tap - 4][g];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      float4 xi = rows[(tap + q) & 7];
      if (kMasked) {   // a tap outside the clip contributes fma(w, 0, acc) = acc: the arithmetic of the valid taps is the same in both paths
        const uint32_t keep = 0u - ((mask[q] >> tap) & 1u);
        xi.x = __uint_as_float(__float_as_uint(xi.x) & keep);
        xi.y = __uint_as_float(__float_as_uint(xi.y) & keep);
        xi.z = __uint_as_float(__float_as_uint(xi.z) & keep);
        xi.w = __uint_as_float(__float_as_uint(xi.w) & keep);
      }
      acc[q][3] = fmaf(w3.w, xi.w, fmaf(w3.z, xi.z, fmaf(w3.y, xi.y, fmaf(w3.x, xi.x, acc[q][3]))));
      if (tap >= 2 && tap <= 8) acc[q][2] = fmaf(w2.w, xi.w, fmaf(w2.z, xi.z, fmaf(w2.y, xi.y, fmaf(w2.x, xi.x, acc[q][2]))));
      if (tap >= 3 && tap <= 7) acc[q][1] = fmaf(w1.w, xi.w, fmaf(w1.z, xi.z, fmaf(w1.y, xi.y, fmaf(w1.x, xi.x, acc[q][1]))));
      if (tap >= 4 && tap <= 6) acc[q][0] = fmaf(w0.w, xi.w, fmaf(w0.z, xi.z, fmaf(w0.y, xi.y, fmaf(w0.x, xi.x, acc[q][0]))));
    }
  }
}

__global__ void __launch_bounds__(kTc2Threads, 2) temporal_conv_tma_kernel(const __grid_constant__ TemporalConvParams p) {
  extern __shared__ uint8_t tc_smem_raw[];
  uint8_t* smem = tc_smem_raw + ((128u - (smem_u32(tc_smem_raw) & 127u)) & 127u);
  float4 (*ws)[64] = reinterpret_cast<float4 (*)[64]>(smem);
  float* tiles = reinterpret_cast<float*>(smem + 26 * 64 * 16);
  unsigned* masks = reinterpret_cast<unsigned*>(smem + 26 * 64 * 16 + 2 * kTc2TileBytes);   // [2][32] valid-tap bits of a tile's tokens
  uint64_t* full = reinterpret_cast<uint64_t*>(masks + 64);                                  // [2] tile rows + masks have landed
  uint64_t* empty = full + 2;                                                               // [2] 8 compute warps are done with the tile
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&p.tmap_x);
    mbar_init(&full[0], 1);
    mbar_init(&full[1], 1);
    mbar_init(&empty[0], 8);
    mbar_init(&empty[1], 8);
    fence_mbar_init();
  }
  for (int idx = threadIdx.x; idx < 26 * 64; idx += kTc2Threads) {
    const int bt = idx >> 6, gg = idx & 63;
    const int j = bt < 3 ? 0 : bt < 8 ? 1 : bt < 15 ? 2 : 3;
    const int tap = j == 0 ? bt + 4 : j == 1 ? bt : j == 2 ? bt - 6 : bt - 15;  // index into the centred 11-tap window
    const int o = j * 64 + gg;
    ws[bt][gg] = make_float4(__ldg(p.w + (0 * 11 + tap) * kDim + o), __ldg(p.w + (1 * 11 + tap) * kDim + o),
                             __ldg(p.w + (2 * 11 + tap) * kDim + o), __ldg(p.w + (3 * 11 + tap) * kDim + o));
  }
  __syncthreads();
  if (warp == 8) {
    // ---- producer: one TMA box per tile; lane i works out which taps of token i stay inside the token's own clip ----
    int it = 0;
    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      const int t = tile * kTc2Tok + lane;
      unsigned m = 0;   // valid taps: 0 <= pos + tap - 5 < len; tokens past the end get an empty mask
      if (t < p.n_tokens) {
        const int pos = __ldg(p.tok_pos + t), len = __ldg(p.tok_len + t);
        const int lo = max(0, 5 - pos), hi = min(10, len + 4 - pos);
        m = hi >= lo ? ((2u << hi) - 1u) & ~((1u << lo) - 1u) : 0u;
      }
      if (it >= 2) mbar_wait(&empty[buf], (uint32_t)(((it >> 1) - 1) & 1));
      masks[buf * 32 + lane] = m;
      __syncwarp();
      if (lane == 0) {
        mbar_arrive_expect_tx(&full[buf], kTc2TileBytes);
        tma_load_2d(&p.tmap_x, &full[buf], reinterpret_cast<uint8_t*>(tiles) + buf * kTc2TileBytes, 0, tile * kTc2Tok - 5);
      }
    }
    return;
  }
  const int g = threadIdx.x & 63;
  const float b[4] = {__ldg(p.bias + g), __ldg(p.bias + 64 + g), __ldg(p.bias + 128 + g), __ldg(p.bias + 192 + g)};
  int it = 0;
  for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++it) {
    const int buf = it & 1;
    // the 8-token slice of the tile rotates over the warp pairs: with clips of equal length the slice that holds a clip boundary
    // (the slower, masked path) would otherwise always fall to the same pair
    const int sub = ((threadIdx.x >> 6) + it) & 3;
    const int t0 = tile * kTc2Tok + sub * 8;
    float acc[8][4];
#pragma unroll
    for (int q = 0; q < 8; ++q)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[q][j] = b[j];
    mbar_wait(&full[buf], (uint32_t)((it >> 1) & 1));
    unsigned mask[8];
    bool all = true;
    {
      const uint4 m0 = *reinterpret_cast<const uint4*>(masks + buf * 32 + sub * 8), m1 = *reinterpret_cast<const uint4*>(masks + buf * 32 + sub * 8 + 4);
      mask[0] = m0.x; mask[1] = m0.y; mask[2] = m0.z; mask[3] = m0.w; mask[4] = m1.x; mask[5] = m1.y; mask[6] = m1.z; mask[7] = m1.w;
#pragma unroll
      for (int q = 0; q < 8; ++q) all = all && mask[q] == 0x7FFu;
    }
    const float* xt = tiles + buf * (kTc2TileBytes / 4) + sub * 8 * kDim;   // row of token t0, tap 0 (= token t0 - 5)
    if (all) temporal_conv_oct<false>(xt, ws, g, mask, acc);                 // warp-uniform: a warp shares its 8 tokens
    else temporal_conv_oct<true>(xt, ws, g, mask, acc);
    float res[8][4];
#pragma unroll
    for (int q = 0; q < 8; ++q)
#pragma unroll
      for (int j = 0; j < 4; ++j) res[q][j] = xt[(q + 5) * kDim + g + 64 * j];
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[buf]);   // this warp has read everything it needs from the tile
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      if (t0 + q < p.n_tokens) {
        float* ys = p.y + (size_t)(t0 + q) * kDim + g;
#pragma unroll
        for (int j = 0; j < 4; ++j) ys[64 * j] = res[q][j] + fmaxf(acc[q][j], 0.0f);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Multi-head self-attention (model.py:143) over PACKED clips, flash-style on the register-fragment tensor path
// (mma.sync m16n8k16 bf16 -> fp32). NOT the production kernel any more: attention_tc_kernel.cuh (tcgen05, scores / P / PV in
// tensor memory) is 1.7x faster and is what vfp_forward launches; this one stays as an independently written twin that the
// boundary test compares it with (vfp_set_tuning(17, 0), tests/test_forward_gpu.py::test_attention_key_block_boundaries).
// (The estimate that kept attention off tcgen05 for a round - a serial chain of ~2 600 cycles of TMEM round trips and
// mbarrier hand-offs per head and key block - was right about the chain and wrong about the conclusion: two CTAs per SM and
// softmax threads that run one step ahead of the PV products hide it.)
//
// A CTA owns one ITEM = 64 consecutive query tokens of ONE clip (the host lists the items: ceil(T / 64) per clip) and walks that
// clip's keys in blocks of 64 tokens from the clip's first token, so what a clip gets never depends on what it is packed next
// to - bit for bit. Per head and key block the Q / K / V slices (64 rows x 64 B each) are staged in shared memory with cp.async
// through a 4-stage ring (three steps of loads in flight per CTA, three CTAs per SM: the kernel moves 2 KB per token and was
// latency-bound with two stages), 80-byte row pitch -> conflict-free ldmatrix, K fragments come from ldmatrix, V fragments
// from ldmatrix.trans (no transposed copy), P goes from the score accumulators straight into the A fragments of the PV
// product. Only the clip's last key block needs a mask.
// (Round 1: one CTA per (clip, head, 64 queries), Q fragments from strided 4-byte global loads, V transposed with scalar
// shared-memory stores: 2.6 ms per 10 000 clips = 64 TFLOP/s.)
// qkv: [tokens][768] bf16 = [Q | K | V], head h = columns 32h .. 32h+31. Softmax in the exp2 domain, fp32.
// ---------------------------------------------------------------------------------------------
constexpr int kAttRows = 64;                          // query tokens per CTA = key tokens per block
constexpr int kAttThreads = 128;                      // 4 warps x 16 query rows
constexpr int kAttPitch = 40;                         // bf16 per shared-memory row: 32 + 8 pad
constexpr int kAttTileElems = kAttRows * kAttPitch;   // one of Q / K / V
constexpr int kAttStageBytes = 3 * kAttTileElems * 2; // 15 360
constexpr int kAttStages = 4;                         // three (head, key block) steps of loads in flight per CTA
constexpr int kAttSmemBytes = kAttStages * kAttStageBytes;   // 61 440: three CTAs per SM

__device__ __forceinline__ void mma_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* smem_row) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(smem_row)));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], const void* smem_row) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(smem_row)));
}
// 16-byte asynchronous copy; src_bytes = 0 zero-fills the destination (rows past the end of the token buffer)
__device__ __forceinline__ void cp_async_16(void* dst, const void* src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ float fast_exp2(float x) {   // one MUFU.EX2; exp2(-inf) = 0
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__global__ void __launch_bounds__(kAttThreads, 3)
attention_fa_kernel(const __nv_bfloat16* __restrict__ qkv, const int4* __restrict__ items /*{first query token, clip start, clip end, 0}*/,
                    __nv_bfloat16* __restrict__ out, int n_tokens) {
  extern __shared__ __align__(16) uint8_t att_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, tig = lane & 3;
  const int4 item = __ldg(items + blockIdx.x);
  const int q0 = item.x, k_begin = item.y, k_end = item.z;
  const int r_lo = q0 + warp * 16 + g, r_hi = r_lo + 8;   // this thread's two query rows (valid below k_end)
  const bool warp_live = q0 + warp * 16 < k_end;          // a warp whose 16 rows lie past the clip only helps with the loads
  const int n_kblocks = (k_end - k_begin + kAttRows - 1) / kAttRows;
  const int n_steps = kHeads * n_kblocks;
  const size_t row_stride = 3 * kDim;

  auto load_stage = [&](int step) {   // step = head * n_kblocks + key block; an empty commit keeps the group count uniform
    if (step < n_steps) {
      const int h = step / n_kblocks, j = step - h * n_kblocks;
      __nv_bfloat16* st = reinterpret_cast<__nv_bfloat16*>(att_smem + (step % kAttStages) * kAttStageBytes);
      const int kbase = k_begin + j * kAttRows;
#pragma unroll
      for (int it = 0; it < 6; ++it) {
        const int idx = threadIdx.x + it * kAttThreads;   // 0 .. 767: tile (0 Q, 1 K, 2 V), row, 16-byte piece
        const int tile = idx >> 8, row = (idx >> 2) & 63, piece = idx & 3;
        const int token = (tile == 0 ? q0 : kbase) + row;
        const bool ok = token < n_tokens;
        const __nv_bfloat16* src = qkv + (size_t)(ok ? token : 0) * row_stride + tile * kDim + h * kHeadDim + piece * 8;
        cp_async_16(st + tile * kAttTileElems + row * kAttPitch + piece * 8, src, ok ? 16 : 0);
      }
    }
    cp_async_commit();
  };

  const float sl2 = 0.17677669529663687f * 1.4426950408889634f;  // 1/sqrt(32) * log2(e)
  float m_lo = -INFINITY, m_hi = -INFINITY, l_lo = 0.f, l_hi = 0.f;
  float o[4][4];
  const int lm = lane >> 3, lr = lane & 7;   // ldmatrix: this lane supplies row lr of matrix lm

#pragma unroll
  for (int pre = 0; pre < kAttStages - 1; ++pre) load_stage(pre);
  for (int step = 0; step < n_steps; ++step) {
    const int h = step / n_kblocks, j = step - h * n_kblocks;
    cp_async_wait<kAttStages - 2>();   // this step's group has landed (the newer ones may still be in flight)
    __syncthreads();                   // ... for every thread's part, and everyone is done with the stage refilled below
    load_stage(step + kAttStages - 1);
    const __nv_bfloat16* Qs = reinterpret_cast<const __nv_bfloat16*>(att_smem + (step % kAttStages) * kAttStageBytes);
    const __nv_bfloat16* Ks = Qs + kAttTileElems;
    const __nv_bfloat16* Vs = Ks + kAttTileElems;
    if (j == 0) {
      m_lo = m_hi = -INFINITY;
      l_lo = l_hi = 0.f;
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) o[a][b] = 0.f;
    }
    const int kbase = k_begin + j * kAttRows;   // first key token of this block
    if (warp_live) {
      // Q fragments of this warp's 16 rows (A operand, two K steps of 16 dims)
      uint32_t qa[2][4];
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) ldmatrix_x4(qa[ks], Qs + (warp * 16 + (lm & 1) * 8 + lr) * kAttPitch + 16 * ks + (lm >> 1) * 8);
      // S = Q K^T for 64 keys: 8 n-tiles of 8 keys
      float s[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        uint32_t kb[4];   // keys 8nt .. 8nt+7; dims 0-7, 8-15, 16-23, 24-31
        ldmatrix_x4(kb, Ks + (nt * 8 + lr) * kAttPitch + lm * 8);
        mma_16816(s[nt], qa[0], kb[0], kb[1]);
        mma_16816(s[nt], qa[1], kb[2], kb[3]);
      }
      // keys past the end of the clip (only in its last block) are masked; block row maxima of the RAW scores - the
      // 1/sqrt(d) log2(e) factor is folded into the exp2
      float mx_lo = -INFINITY, mx_hi = -INFINITY;
      if (kbase + kAttRows <= k_end) {
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          mx_lo = fmaxf(mx_lo, fmaxf(s[nt][0], s[nt][1]));
          mx_hi = fmaxf(mx_hi, fmaxf(s[nt][2], s[nt][3]));
        }
      } else {
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          const int key = kbase + 8 * nt + 2 * tig;
          if (key >= k_end) s[nt][0] = s[nt][2] = -INFINITY;
          if (key + 1 >= k_end) s[nt][1] = s[nt][3] = -INFINITY;
          mx_lo = fmaxf(mx_lo, fmaxf(s[nt][0], s[nt][1]));
          mx_hi = fmaxf(mx_hi, fmaxf(s[nt][2], s[nt][3]));
        }
      }
      mx_lo = fmaxf(mx_lo, __shfl_xor_sync(0xffffffffu, mx_lo, 1));
      mx_lo = fmaxf(mx_lo, __shfl_xor_sync(0xffffffffu, mx_lo, 2));
      mx_hi = fmaxf(mx_hi, __shfl_xor_sync(0xffffffffu, mx_hi, 1));
      mx_hi = fmaxf(mx_hi, __shfl_xor_sync(0xffffffffu, mx_hi, 2));
      // running maxima live in the scaled (log2) domain; every block holds at least one valid key, so they are finite
      const float mn_lo = fmaxf(m_lo, mx_lo * sl2), mn_hi = fmaxf(m_hi, mx_hi * sl2);
      const float ms_lo = mn_lo, ms_hi = mn_hi;
      const float c_lo = fast_exp2(m_lo - ms_lo), c_hi = fast_exp2(m_hi - ms_hi);
      m_lo = mn_lo;
      m_hi = mn_hi;
      l_lo *= c_lo;
      l_hi *= c_hi;
#pragma unroll
      for (int jd = 0; jd < 4; ++jd) {
        o[jd][0] *= c_lo; o[jd][1] *= c_lo; o[jd][2] *= c_hi; o[jd][3] *= c_hi;
      }
      // P = exp2(S - m); O += P V  (P goes from the accumulator registers straight into the A fragments)
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        uint32_t pa[4];
        float p[2][4];
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int nt = 2 * kk + hh;
          p[hh][0] = fast_exp2(fmaf(s[nt][0], sl2, -ms_lo));
          p[hh][1] = fast_exp2(fmaf(s[nt][1], sl2, -ms_lo));
          p[hh][2] = fast_exp2(fmaf(s[nt][2], sl2, -ms_hi));
          p[hh][3] = fast_exp2(fmaf(s[nt][3], sl2, -ms_hi));
          l_lo += p[hh][0] + p[hh][1];
          l_hi += p[hh][2] + p[hh][3];
        }
        pa[0] = pack_bf16x2(p[0][0], p[0][1]);
        pa[1] = pack_bf16x2(p[0][2], p[0][3]);
        pa[2] = pack_bf16x2(p[1][0], p[1][1]);
        pa[3] = pack_bf16x2(p[1][2], p[1][3]);
        // V fragments (B operand, 16 keys x 8 dims per n-tile) through ldmatrix.trans: matrices (keys 0-7 | 8-15) x (dims 8jd | 8jd+8)
#pragma unroll
        for (int jp = 0; jp < 2; ++jp) {
          uint32_t vb[4];
          ldmatrix_x4_trans(vb, Vs + (kk * 16 + (lm & 1) * 8 + lr) * kAttPitch + (2 * jp + (lm >> 1)) * 8);
          mma_16816(o[2 * jp], pa, vb[0], vb[1]);
          mma_16816(o[2 * jp + 1], pa, vb[2], vb[3]);
        }
      }
    }
    if (j == n_kblocks - 1 && warp_live) {   // last key block of this head: normalise and store this head's 32 output columns
      float t_lo = l_lo, t_hi = l_hi;
      t_lo += __shfl_xor_sync(0xffffffffu, t_lo, 1);
      t_lo += __shfl_xor_sync(0xffffffffu, t_lo, 2);
      t_hi += __shfl_xor_sync(0xffffffffu, t_hi, 1);
      t_hi += __shfl_xor_sync(0xffffffffu, t_hi, 2);
      const float i_lo = 1.0f / t_lo, i_hi = 1.0f / t_hi;
      __nv_bfloat16* o_lo = out + (size_t)r_lo * kDim + h * kHeadDim + 2 * tig;
      __nv_bfloat16* o_hi = out + (size_t)r_hi * kDim + h * kHeadDim + 2 * tig;
#pragma unroll
      for (int jd = 0; jd < 4; ++jd) {
        if (r_lo < k_end) *reinterpret_cast<uint32_t*>(o_lo + 8 * jd) = pack_bf16x2(o[jd][0] * i_lo, o[jd][1] * i_lo);
        if (r_hi < k_end) *reinterpret_cast<uint32_t*>(o_hi + 8 * jd) = pack_bf16x2(o[jd][2] * i_hi, o[jd][3] * i_hi);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// adaptive_pooling (model.py:256-270): per clip and channel, mean_T(x), max_T(x) and
// sum_T x * softmax_T(logit) where logit = relu(W_p x + b_p) was produced by the GEMM before.
// One CTA per clip, one thread per channel, single pass with an online softmax.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
temporal_pool_kernel(const float* __restrict__ x, const float* __restrict__ logits, const int* __restrict__ cu,
                     float* __restrict__ pooled /*[clips][768]*/, __nv_bfloat16* __restrict__ pooled_bf /*same, bf16*/) {
  const int clip = blockIdx.x, c = threadIdx.x;
  const int t0 = cu[clip], T = cu[clip + 1] - t0;
  float sum = 0.f, mx = -INFINITY, m = -INFINITY, l = 0.f, ws = 0.f;
  for (int t = 0; t < T; ++t) {
    const float xv = x[(size_t)(t0 + t) * kDim + c];
    const float lg = logits[(size_t)(t0 + t) * kDim + c];
    sum += xv;
    mx = fmaxf(mx, xv);
    const float m_new = fmaxf(m, lg);
    const float corr = __expf(m - m_new);
    const float p = __expf(lg - m_new);
    l = l * corr + p;
    ws = ws * corr + p * xv;
    m = m_new;
  }
  float* o = pooled + (size_t)clip * (3 * kDim);
  __nv_bfloat16* ob = pooled_bf + (size_t)clip * (3 * kDim);
  const float avg = sum / (float)T, wsum = ws / l;
  o[c] = avg;
  o[kDim + c] = mx;
  o[2 * kDim + c] = wsum;
  ob[c] = __float2bfloat16(avg);
  ob[kDim + c] = __float2bfloat16(mx);
  ob[2 * kDim + c] = __float2bfloat16(wsum);
}

// ---------------------------------------------------------------------------------------------
// final_projection (Linear 768->256, ReLU, Linear 256->D) + L2 normalise (model.py:219-224, 292-294),
// fp32 on CUDA cores: 0.5 MFLOP per clip, and the last rounding step before the embedding leaves.
// kClips clips per CTA so the transposed weights are streamed once per CTA, thread = output channel.
// ---------------------------------------------------------------------------------------------
template <int kClips>
__global__ void __launch_bounds__(256)
final_projection_kernel(const float* __restrict__ pooled, const float* __restrict__ w0t /*[768][256]*/,
                        const float* __restrict__ b0, const float* __restrict__ w3t /*[256][D]*/,
                        const float* __restrict__ b3, int D, int n_clips, float* __restrict__ emb /*[clips][D]*/) {
  __shared__ float sp[kClips][3 * kDim];
  __shared__ float sh[kClips][kDim];
  __shared__ float red[kClips][8];
  const int c0 = blockIdx.x * kClips;
  const int tid = threadIdx.x;
  for (int i = tid; i < kClips * 3 * kDim; i += 256) {
    const int v = i / (3 * kDim), k = i - v * 3 * kDim;
    sp[v][k] = (c0 + v < n_clips) ? pooled[(size_t)(c0 + v) * 3 * kDim + k] : 0.f;
  }
  __syncthreads();
  float acc[kClips];
#pragma unroll
  for (int v = 0; v < kClips; ++v) acc[v] = 0.f;
  for (int k = 0; k < 3 * kDim; ++k) {
    const float w = __ldg(w0t + (size_t)k * kDim + tid);
#pragma unroll
    for (int v = 0; v < kClips; ++v) acc[v] += w * sp[v][k];
  }
  const float bb = __ldg(b0 + tid);
#pragma unroll
  for (int v = 0; v < kClips; ++v) sh[v][tid] = fmaxf(acc[v] + bb, 0.f);
  __syncthreads();
  // second layer: D may be smaller/larger than 256 -> loop output channels in strides of 256
  for (int oc = tid; oc < ((D + 255) / 256) * 256; oc += 256) {
    float e[kClips];
#pragma unroll
    for (int v = 0; v < kClips; ++v) e[v] = 0.f;
    if (oc < D) {
      for (int k = 0; k < kDim; ++k) {
        const float w = __ldg(w3t + (size_t)k * D + oc);
#pragma unroll
        for (int v = 0; v < kClips; ++v) e[v] += w * sh[v][k];
      }
      const float b = __ldg(b3 + oc);
#pragma unroll
      for (int v = 0; v < kClips; ++v) e[v] += b;
    }
    // stash un-normalised values in global, accumulate squared norms below
#pragma unroll
    for (int v = 0; v < kClips; ++v) {
      if (oc < D && c0 + v < n_clips) emb[(size_t)(c0 + v) * D + oc] = e[v];
      float q = (oc < D) ? e[v] * e[v] : 0.f;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
      if ((tid & 31) == 0) {
        if (oc < 256) red[v][tid >> 5] = q; else red[v][tid >> 5] += q;
      }
    }
  }
  __syncthreads();
  for (int v = 0; v < kClips; ++v) {
    if (c0 + v >= n_clips) break;
    float n2 = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) n2 += red[v][i];
    const float inv = 1.0f / fmaxf(sqrtf(n2), 1e-12f);
    for (int oc = tid; oc < D; oc += 256) emb[(size_t)(c0 + v) * D + oc] *= inv;
  }
}

// fp32 -> bf16 row copy (pooling GEMM input, join operands)
__global__ void f32_to_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, long long n8) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n8) return;
  const float4 a = reinterpret_cast<const float4*>(in)[2 * i];
  const float4 b = reinterpret_cast<const float4*>(in)[2 * i + 1];
  uint4 o;
  o.x = pack_bf16x2(a.x, a.y); o.y = pack_bf16x2(a.z, a.w);
  o.z = pack_bf16x2(b.x, b.y); o.w = pack_bf16x2(b.z, b.w);
  reinterpret_cast<uint4*>(out)[i] = o;
}

}  // namespace vfp
