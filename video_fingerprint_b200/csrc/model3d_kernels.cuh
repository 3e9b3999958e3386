// VideoFingerprint3D forward (/root/reference/model.py:406-512), the reference's second model behind create_model("3d").
// Four Conv3d + BatchNorm3d + ReLU blocks, spatial average pool, a temporal Conv1d, attention + average pooling over time,
// a two-layer projector and L2 normalisation. Every Conv3d runs as   im2col (this file)  ->  tcgen05 GEMM (gemm_sm100.cuh,
// bias + ReLU + bf16 TMA-store epilogue)   on bf16 operands with fp32 accumulation; the GEMM output [positions][C_out] IS the
// channels-last activation tensor the next layer's im2col reads. The small tail (pooling, Conv1d, softmax, projector,
// normalise: < 0.2 MFLOP per clip) is one fp32 CTA per clip.
// First version of this model: correct and on the tensor cores, but the explicit im2col costs ~6x the input in HBM traffic;
// an implicit-GEMM loader like the attention model's stem is the obvious next step (DESIGN.md section 7).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "conv1_kernel.cuh"   // FrameDtype

namespace vfp {

// Every kernel below works on a PACKED pass: clips of any lengths back to back, each activation the concatenation of the
// clips' own activations in clip order (layer 1: sum G * 1024 rows, layer 2: sum G * 256, layer 3: sum T3 * 64, layer 4:
// sum T3 * 16, with G = ceil(T / fs) and T3 = (G - 1) / 2 + 1 per clip). A row or CTA finds its clip through a small table the
// host builds per pass; the arithmetic is the same as for the clip alone, so packed results equal B = 1 results bit for bit.
// An equal-length batch is the special case of uniform clip lengths.

// Layer 1: Conv3d(3 -> 16, kernel (fs, 5, 5), stride (fs, 2, 2), padding (0, 2, 2)) + folded BatchNorm3d + ReLU over frames
// of any accepted type: planar (T, 3, 64, 64) u8 / bf16 / fp32 or decoder-layout (T, 64, 64, 3) u8; each clip's T is
// zero-padded to a multiple of fs like model.py:468-471.
// C_in = 3 makes this the same problem as the attention model's conv1 (6-byte pixels are not TMA / UMMA addressable), with
// the same answer: the register-fragment tensor path. Per (kt, kh) the 5 x 3 (kw, c) taps of an output position are 15
// CONSECUTIVE bf16 of a pixel-interleaved (HWC) copy of the input row (+ 1 don't-care with zero weight), so one A register of
// mma.sync m16n8k16 is one aligned 32-bit shared load: K = 16 * 5 * fs, k = (kt*5 + kh)*16 + kw*3 + c.
// One CTA per (global group, oh) = 32 output positions x 16 channels. groups[global group] = {device address of the group's
// first frame, frames of its clip from there on}: frames at or past the clip's own end read as zero, never as whatever lies
// next in memory, so clips may sit anywhere (separate allocations, overlapping windows of one buffer, one view listed twice).
// The 5 input rows x fs frames a CTA needs are staged in shared memory (68 pixels: zero halo of 2 on both sides; rows outside
// the image and frames past the clip end are zero), the four warps split the 5*fs K runs, partial sums meet in shared memory,
// bias + ReLU, bf16 channels-last output [position][32] (channels 16..31 zero: the 32-column box of the next layer's GEMM).
// An earlier version materialised the im2col matrix (2.6 GB written and read back per 256 clips): 1.05 ms per 256 clips
// against 0.1 ms here.
// wpack: [5*fs runs][2 n-tiles][32 lanes] x uint2 = the B fragments of the folded weights; bias [16].
struct __align__(16) L1Group {
  const void* frames;   // first frame of the group; 16-byte aligned (8/16-byte vector loads)
  int left;             // frames of the clip from this one on (>= 1)
  int pad;
};
__global__ void __launch_bounds__(128) conv3d_l1_kernel(int frame_dtype, const L1Group* __restrict__ groups, int fs,
                                                        const uint2* __restrict__ wpack, const float* __restrict__ bias,
                                                        __nv_bfloat16* __restrict__ out) {
  extern __shared__ __align__(16) uint8_t smem3d[];
  __nv_bfloat16* tile = reinterpret_cast<__nv_bfloat16*>(smem3d);   // [fs*5 runs][68 pixels][3 channels] (+ 2 pad elements)
  const int runs = fs * 5;
  float* part = reinterpret_cast<float*>(smem3d + (((size_t)runs * 204 * 2 + 4 + 15) & ~size_t(15)));   // [4 warps][16][32 lanes]
  const int oh = blockIdx.x & 31;
  const unsigned gg = blockIdx.x >> 5;
  const L1Group grp = groups[gg];
  const uint8_t* fbase = static_cast<const uint8_t*>(grp.frames);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // halo pixels (x = -2, -1, 64, 65) of every run
  for (int i = tid; i < runs * 12; i += 128) {
    const int run = i / 12, r = i - run * 12;
    const int x = r < 6 ? r / 3 : 66 + (r - 6) / 3, c = r % 3;
    tile[(run * 68 + x) * 3 + c] = __float2bfloat16(0.0f);
  }
  if (tid < 2) tile[runs * 204 + tid] = __float2bfloat16(0.0f);   // the don't-care element after the very last run
  if (frame_dtype == kFrameU8HWC) {
    // decoder layout: an input row (run, ih) is 192 contiguous bytes already in the tile's pixel-interleaved order, so byte b
    // goes to element run*204 + 6 + b. One item = 16 bytes: one 16-byte load, eight 4-byte bf16x2 stores (even element offset).
    // Same value as the planar u8 path, (float)u8 * (1/255) rounded to bf16, so both layouts give the same bits.
    for (int i = tid; i < runs * 12; i += 128) {
      const int q = i % 12, run = i / 12;
      const int kh = run % 5, kt = run / 5;
      const int ih = 2 * oh + kh - 2;
      uint4 d = make_uint4(0u, 0u, 0u, 0u);
      if (kt < grp.left && ih >= 0 && ih < 64) d = *reinterpret_cast<const uint4*>(fbase + (size_t)kt * 12288 + ih * 192 + q * 16);
      const uint32_t w[4] = {d.x, d.y, d.z, d.w};
      __nv_bfloat162* dst = reinterpret_cast<__nv_bfloat162*>(tile + run * 204 + 6 + q * 16);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const uint32_t b = w[j >> 1] >> (16 * (j & 1));
        dst[j] = __floats2bfloat162_rn((float)(b & 0xFF) * (1.0f / 255.0f), (float)((b >> 8) & 0xFF) * (1.0f / 255.0f));
      }
    }
  } else {
    // planar: one item = 8 consecutive pixels of one (run, plane) row: a 16-byte (bf16) / 8-byte (u8) / 32-byte (fp32) load
    for (int i = tid; i < runs * 24; i += 128) {
      const int x0 = (i & 7) * 8, c = (i >> 3) % 3, run = i / 24;
      const int kh = run % 5, kt = run / 5;
      const int ih = 2 * oh + kh - 2;
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.0f;
      if (kt < grp.left && ih >= 0 && ih < 64) {
        const size_t idx = (((size_t)kt * 3 + c) * 64 + ih) * 64 + x0;
        if (frame_dtype == kFrameBF16) {
          const uint4 q = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(fbase) + idx);
          const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            v[2 * j] = __uint_as_float(w[j] << 16);
            v[2 * j + 1] = __uint_as_float(w[j] & 0xFFFF0000u);
          }
        } else if (frame_dtype == kFrameU8) {
          const uint2 q = *reinterpret_cast<const uint2*>(fbase + idx);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            v[j] = (float)((q.x >> (8 * j)) & 0xFF) * (1.0f / 255.0f);
            v[4 + j] = (float)((q.y >> (8 * j)) & 0xFF) * (1.0f / 255.0f);
          }
        } else {
          const float4 a = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(fbase) + idx);
          const float4 d = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(fbase) + idx + 4);
          v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = d.x; v[5] = d.y; v[6] = d.z; v[7] = d.w;
        }
      }
      __nv_bfloat16* dst = tile + (run * 68 + x0 + 2) * 3 + c;
#pragma unroll
      for (int j = 0; j < 8; ++j) dst[3 * j] = __float2bfloat16(v[j]);
    }
  }
  __syncthreads();
  // ---- this warp's share of the K runs: 2 m-tiles (positions 0-15, 16-31) x 2 n-tiles (channels 0-7, 8-15) ----
  const int g = lane >> 2, tig = lane & 3;
  const uint32_t* tile32 = reinterpret_cast<const uint32_t*>(tile);
  float acc[2][2][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[mt][nt][i] = 0.0f;
  for (int run = warp; run < runs; run += 4) {
    const uint2 b0 = __ldg(wpack + (run * 2 + 0) * 32 + lane), b1 = __ldg(wpack + (run * 2 + 1) * 32 + lane);
    const uint32_t bf0[2] = {b0.x, b0.y}, bf1[2] = {b1.x, b1.y};
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      // element (run*68 + 2*ow)*3 + k of the tile = word run*102 + 3*ow + k/2; fragment rows are positions ow = 16*mt + g, + 8
      const uint32_t* base = tile32 + run * 102 + 3 * (16 * mt + g) + tig;
      uint32_t a[4];
      a[0] = base[0];
      a[1] = base[24];
      a[2] = base[4];
      a[3] = base[28];
      mma_bf16_16816(acc[mt][0], a, bf0);
      mma_bf16_16816(acc[mt][1], a, bf1);
    }
  }
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) part[(warp * 16 + (mt * 2 + nt) * 4 + i) * 32 + lane] = acc[mt][nt][i];
  __syncthreads();
  // ---- reduce the four partial sums, bias + ReLU, channels-last bf16 rows of 32 (16 real channels + 16 zeros) ----
  __nv_bfloat16* orow = out + ((size_t)gg * 1024 + (size_t)oh * 32) * 32;
  for (int o = tid; o < 32 * 8; o += 128) {         // one item = channel pair (2 * cp, 2 * cp + 1) of one position
    const int ow = o >> 3, cp = o & 7;
    // fragment coordinates of (position ow, channels 2cp, 2cp+1): mt = ow / 16, row r = ow % 16 -> g = r % 8, upper = r / 8;
    // nt = cp / 4, tig = cp % 4 -> accumulator elements i = 2 * upper, 2 * upper + 1 of lane g * 4 + tig
    const int mt = ow >> 4, r = ow & 15, gg = r & 7, upper = r >> 3, nt = cp >> 2, tg = cp & 3;
    const int ln = gg * 4 + tg, e0 = (mt * 2 + nt) * 4 + 2 * upper;
    float s0 = bias[2 * cp], s1 = bias[2 * cp + 1];
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      s0 += part[(w * 16 + e0) * 32 + ln];
      s1 += part[(w * 16 + e0 + 1) * 32 + ln];
    }
    *reinterpret_cast<__nv_bfloat162*>(orow + ow * 32 + 2 * cp) = __floats2bfloat162_rn(fmaxf(s0, 0.0f), fmaxf(s1, 0.0f));
  }
  for (int o = tid; o < 32 * 2; o += 128)           // channels 16..31 = 0
    *reinterpret_cast<uint4*>(orow + (o >> 1) * 32 + 16 + (o & 1) * 8) = make_uint4(0u, 0u, 0u, 0u);
}

// Layers 2-4: Conv3d(C -> *, kernel 3x3x3, stride (st, 2, 2), padding 1) over a packed channels-last activation
// [sum Ti][Hi][Wi][C] (C a multiple of 8). Row = (output slot, oh, ow), column k = ((kt*3 + kh)*3 + kw)*C + c; one thread
// moves 8 channels (16 bytes). slots[output slot] = {first input slot of the clip, the clip's input positions Ti, first input
// position of the window (to * st - 1, clip-local), 0}: the temporal zero padding and the stride stop at the clip's own ends.
__global__ void im2col3d_ndhwc_kernel(const __nv_bfloat16* __restrict__ in, const int4* __restrict__ slots, long long n_slots, int Hi,
                                      int Wi, int C, int Ho, int Wo, int kp, __nv_bfloat16* __restrict__ out) {
  const int k8n = kp / 8;
  const long long rows = n_slots * Ho * Wo;
  const long long total = rows * k8n;
  const int kreal = 27 * C;
  for (long long it = (long long)blockIdx.x * blockDim.x + threadIdx.x; it < total; it += (long long)gridDim.x * blockDim.x) {
    const long long row = it / k8n;
    const int k0 = (int)(it - row * k8n) * 8;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (k0 < kreal) {
      const int tap = k0 / C, c0 = k0 - tap * C;
      const int kw = tap % 3, kh = (tap / 3) % 3, kt = tap / 9;
      long long r = row;
      const int ow = (int)(r % Wo); r /= Wo;
      const int oh = (int)(r % Ho); r /= Ho;
      const int4 s = __ldg(slots + r);
      const int t = s.z + kt, ih = 2 * oh + kh - 1, iw = 2 * ow + kw - 1;
      if (t >= 0 && t < s.y && ih >= 0 && ih < Hi && iw >= 0 && iw < Wi)
        v = *reinterpret_cast<const uint4*>(in + ((((size_t)s.x + t) * Hi + ih) * Wi + iw) * C + c0);
    }
    *reinterpret_cast<uint4*>(out + row * kp + k0) = v;
  }
}

struct Head3dParams {
  const __nv_bfloat16* act;   // packed layer-4 output [sum T3][16][128]
  const int2* clips;          // per clip {first temporal slot in act, T3}
  const float *tc_w, *tc_b;   // temporal_conv (128, 128, 3), (128)
  const float *ta_w, *ta_b;   // temporal_attention (1, 128, 1), (1)
  const float *p0_w, *p0_b;   // projector.0 (128, 128)
  const float *p3_w, *p3_b;   // projector.3 (D, 128)
  int D;
  float* out;                 // [clips][D]
};
constexpr int kHead3dMaxT = 32;   // temporal positions after the two temporal strides (clips of up to 32 * 2 * fs frames)

// model.py:476-509 for one clip per CTA (128 threads = one per channel); pooling, Conv1d padding and softmax see only that clip
__global__ void __launch_bounds__(128) head3d_kernel(const Head3dParams p) {
  __shared__ float feat[kHead3dMaxT + 2][128];   // spatial means, rows 0 and T3+1 are the Conv1d zero padding
  __shared__ float tc[kHead3dMaxT][128];
  __shared__ float prob[kHead3dMaxT];
  __shared__ float vec[128], hid[128];
  __shared__ float red[4];
  const int b = blockIdx.x, c = threadIdx.x;
  const int2 clip = p.clips[b];
  const int T3 = clip.y;
  const __nv_bfloat16* a = p.act + (size_t)clip.x * 16 * 128;
  feat[0][c] = 0.0f;
  feat[T3 + 1][c] = 0.0f;
  for (int t = 0; t < T3; ++t) {
    float s = 0.0f;
    for (int px = 0; px < 16; ++px) s += __bfloat162float(a[((size_t)t * 16 + px) * 128 + c]);
    feat[t + 1][c] = s * (1.0f / 16.0f);   // AdaptiveAvgPool3d((None, 1, 1))
  }
  __syncthreads();
  for (int t = 0; t < T3; ++t) {           // temporal_conv: Conv1d(128, 128, 3, padding 1)
    float s = p.tc_b[c];
    const float* w = p.tc_w + (size_t)c * 128 * 3;
    for (int ci = 0; ci < 128; ++ci)
      s += w[ci * 3] * feat[t][ci] + w[ci * 3 + 1] * feat[t + 1][ci] + w[ci * 3 + 2] * feat[t + 2][ci];
    tc[t][c] = s;
  }
  __syncthreads();
  for (int t = c; t < T3; t += 128) {      // temporal_attention logits
    float s = p.ta_b[0];
    for (int ci = 0; ci < 128; ++ci) s += p.ta_w[ci] * tc[t][ci];
    prob[t] = s;
  }
  __syncthreads();
  if (c == 0) {                             // softmax over time (T3 <= 64)
    float mx = -INFINITY, den = 0.0f;
    for (int t = 0; t < T3; ++t) mx = fmaxf(mx, prob[t]);
    for (int t = 0; t < T3; ++t) { prob[t] = expf(prob[t] - mx); den += prob[t]; }
    for (int t = 0; t < T3; ++t) prob[t] /= den;
  }
  __syncthreads();
  {
    float wsum = 0.0f, avg = 0.0f;
    for (int t = 0; t < T3; ++t) { wsum += tc[t][c] * prob[t]; avg += tc[t][c]; }
    vec[c] = wsum + avg / (float)T3;        // weighted + average pooling
  }
  __syncthreads();
  {
    float s = p.p0_b[c];
    const float* w = p.p0_w + (size_t)c * 128;
    for (int ci = 0; ci < 128; ++ci) s += w[ci] * vec[ci];
    hid[c] = fmaxf(s, 0.0f);
  }
  __syncthreads();
  float e[4];   // D <= 512
  float sq = 0.0f;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int d = c + 128 * j;
    e[j] = 0.0f;
    if (d < p.D) {
      float s = p.p3_b[d];
      const float* w = p.p3_w + (size_t)d * 128;
      for (int ci = 0; ci < 128; ++ci) s += w[ci] * hid[ci];
      e[j] = s;
      sq += s * s;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  if ((c & 31) == 0) red[c >> 5] = sq;
  __syncthreads();
  const float nrm = fmaxf(sqrtf(red[0] + red[1] + red[2] + red[3]), 1e-12f);   // F.normalize eps
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int d = c + 128 * j;
    if (d < p.D) p.out[(size_t)b * p.D + d] = e[j] / nrm;
  }
}

}  // namespace vfp
