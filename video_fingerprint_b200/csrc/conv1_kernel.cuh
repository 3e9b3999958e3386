// Frame-encoder stem: Conv2d(3->32, k5, s2, p2) + folded BatchNorm + ReLU, planar CHW frames in
// (u8 / bf16 / fp32), bf16 out in space-to-depth NHWC: [frame][16][16][(oh%2*2 + ow%2)*32 + c].
//
// C_in = 3 gives 6-byte pixels, which neither the TMA im2col box nor a UMMA smem descriptor can address,
// so this layer runs on the register-fragment tensor path (mma.sync m16n8k16, bf16 -> fp32): every thread
// builds its A fragments straight from an HWC copy of the frame in shared memory. The GEMM view is
//   M = 1024 output pixels, N = 32, K = 5 (kh) x 16 (15 = 5 kw x 3 c, +1 zero-weight pad).
// For output pixel (oh, ow) and filter row kh the 15 taps are 15 CONSECUTIVE bf16 values of the padded HWC
// frame, so each A register (two consecutive k) is one aligned 32-bit shared load.
#pragma once
#include "sm100_primitives.cuh"

namespace vfp {

constexpr int kC1Threads = 128;   // 4 warps; small CTAs so ~5 frames are in flight per SM
constexpr int kC1PadW = 68;   // columns -2 .. 65
constexpr int kC1PadH = 67;   // rows    -2 .. 64
constexpr int kC1SmemElems = kC1PadH * kC1PadW * 3 + 8;
constexpr int kC1CellPitch = 272;                 // 256 B cell + 16 B pad: conflict-free fragment stores
constexpr int kC1StageBytes = 8 * kC1CellPitch;   // per warp: 8 cells

enum FrameDtype : int { kFrameU8 = 0, kFrameBF16 = 1, kFrameF32 = 2, kFrameU8HWC = 3 };

__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// Copy the frame at `frame` into the padded HWC bf16 tile (interior cells only; the halo stays zero). Any of the accepted
// frame formats: planar CHW uint8 / bf16 / fp32 (what _preprocess_frames returns, fingerprint.py:210-214) or decoder-layout
// HWC uint8. uint8 values are divided by 255 like the reference does.
__device__ __forceinline__ void stage_frame_hwc(const void* __restrict__ frame, int frame_dtype,
                                                __nv_bfloat16* __restrict__ tile, int tid, int nthreads) {
  if (frame_dtype == kFrameU8) {
    const uint32_t* src = reinterpret_cast<const uint32_t*>(frame);
#pragma unroll 4
    for (int i = tid; i < 3072; i += nthreads) {
      const uint32_t q = __ldg(src + i);
      const int e = i * 4;
      const int c = e >> 12, h = (e >> 6) & 63, w = e & 63;
      __nv_bfloat16* d = tile + ((h + 2) * kC1PadW + (w + 2)) * 3 + c;
      d[0] = __float2bfloat16((float)(q & 0xFF) / 255.0f);
      d[3] = __float2bfloat16((float)((q >> 8) & 0xFF) / 255.0f);
      d[6] = __float2bfloat16((float)((q >> 16) & 0xFF) / 255.0f);
      d[9] = __float2bfloat16((float)(q >> 24) / 255.0f);
    }
  } else if (frame_dtype == kFrameU8HWC) {
    // decoder layout (H, W, 3) uint8, i.e. what _preprocess_frames sees before its permute (fingerprint.py:210-212):
    // a frame row is 192 contiguous bytes = 192 contiguous elements of the padded HWC tile
    const uint32_t* src = reinterpret_cast<const uint32_t*>(frame);
#pragma unroll 4
    for (int i = tid; i < 3072; i += nthreads) {
      const uint32_t q = __ldg(src + i);
      const int h = i / 48, k = (i - h * 48) * 4;
      __nv_bfloat162* d = reinterpret_cast<__nv_bfloat162*>(tile + ((h + 2) * kC1PadW + 2) * 3 + k);
      d[0] = __floats2bfloat162_rn((float)(q & 0xFF) / 255.0f, (float)((q >> 8) & 0xFF) / 255.0f);
      d[1] = __floats2bfloat162_rn((float)((q >> 16) & 0xFF) / 255.0f, (float)(q >> 24) / 255.0f);
    }
  } else if (frame_dtype == kFrameBF16) {
    const uint2* src = reinterpret_cast<const uint2*>(frame);
#pragma unroll 4
    for (int i = tid; i < 3072; i += nthreads) {
      const uint2 q = __ldg(src + i);
      const int e = i * 4;
      const int c = e >> 12, h = (e >> 6) & 63, w = e & 63;
      __nv_bfloat16* d = tile + ((h + 2) * kC1PadW + (w + 2)) * 3 + c;
      const __nv_bfloat162 lo = *reinterpret_cast<const __nv_bfloat162*>(&q.x);
      const __nv_bfloat162 hi = *reinterpret_cast<const __nv_bfloat162*>(&q.y);
      d[0] = lo.x; d[3] = lo.y; d[6] = hi.x; d[9] = hi.y;
    }
  } else {
    const float4* src = reinterpret_cast<const float4*>(frame);
#pragma unroll 4
    for (int i = tid; i < 3072; i += nthreads) {
      const float4 q = __ldg(src + i);
      const int e = i * 4;
      const int c = e >> 12, h = (e >> 6) & 63, w = e & 63;
      __nv_bfloat16* d = tile + ((h + 2) * kC1PadW + (w + 2)) * 3 + c;
      d[0] = __float2bfloat16(q.x); d[3] = __float2bfloat16(q.y);
      d[6] = __float2bfloat16(q.z); d[9] = __float2bfloat16(q.w);
    }
  }
}

// frame_addr: [n_frames] device address of each frame (token_map_kernel); wpack: [5 kh][4 n-tiles][32 lanes][2] packed
// bf16x2 B fragments, bias: [32] fp32 (BN folded)
__global__ void __launch_bounds__(kC1Threads)
conv1_stem_kernel(const unsigned long long* __restrict__ frame_addr, int frame_dtype, long long n_frames,
                  const uint32_t* __restrict__ wpack, const float* __restrict__ bias,
                  __nv_bfloat16* __restrict__ out) {
  __shared__ __align__(16) __nv_bfloat16 tile[kC1SmemElems];
  __shared__ __align__(16) uint8_t stage[(kC1Threads / 32) * kC1StageBytes];
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, tig = lane & 3;

  // B fragments and bias stay in registers for the whole kernel.
  uint32_t bfrag[5][4][2];
#pragma unroll
  for (int kh = 0; kh < 5; ++kh)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const uint2 w = __ldg(reinterpret_cast<const uint2*>(wpack) + (kh * 4 + nt) * 32 + lane);
      bfrag[kh][nt][0] = w.x;
      bfrag[kh][nt][1] = w.y;
    }
  float bia[4][2];
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) {
    bia[nt][0] = __ldg(bias + nt * 8 + 2 * tig);
    bia[nt][1] = __ldg(bias + nt * 8 + 2 * tig + 1);
  }

  // zero the halo once: interior cells are rewritten for every frame, halo cells never are.
  for (int i = tid; i < kC1SmemElems; i += kC1Threads) tile[i] = __float2bfloat16(0.0f);
  __syncthreads();

  for (long long f = blockIdx.x; f < n_frames; f += gridDim.x) {
    stage_frame_hwc(reinterpret_cast<const void*>(__ldg(frame_addr + f)), frame_dtype, tile, tid, kC1Threads);
    __syncthreads();

    // ---- 64 m-tiles of 16 pixels, processed as 32 vertical PAIRS (output rows 2j, 2j+1; same 16 columns): in the
    //      space-to-depth output a pair covers 8 whole cells = 2 KB of contiguous global memory. The fragments are
    //      re-assembled through a padded per-warp staging tile so that the global stores are full 512-byte lines
    //      (direct fragment stores put 8 different lines into every store instruction: ncu showed the LSU, not HBM or
    //      the tensor pipe, as the limiter of this kernel). ----
    const uint32_t* tile32 = reinterpret_cast<const uint32_t*>(tile);
    __nv_bfloat16* out_f = out + f * (1024 * 32);
    uint8_t* my_stage = stage + warp * kC1StageBytes;
#pragma unroll 1
    for (int pair = warp; pair < 32; pair += kC1Threads / 32) {
      const int j = pair >> 1;            // output rows 2j, 2j+1 = cell row j
      const int ow0 = (pair & 1) * 16;
#pragma unroll
      for (int sh = 0; sh < 2; ++sh) {
        const int oh = 2 * j + sh;
        float acc[4][4];
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
          for (int i = 0; i < 4; ++i) acc[nt][i] = 0.0f;
#pragma unroll
        for (int kh = 0; kh < 5; ++kh) {
          // element offset of (pixel ow, k) = ((2*oh+kh)*PadW + 2*ow)*3 + k ; all terms even -> word aligned
          const int base_lo = (((2 * oh + kh) * kC1PadW + 2 * (ow0 + g)) * 3) >> 1;
          const int base_hi = base_lo + 24;  // pixel +8 -> +16 columns -> +48 elements -> +24 words
          uint32_t a[4];
          a[0] = tile32[base_lo + tig];
          a[1] = tile32[base_hi + tig];
          a[2] = tile32[base_lo + tig + 4];
          a[3] = tile32[base_hi + tig + 4];
#pragma unroll
          for (int nt = 0; nt < 4; ++nt) mma_bf16_16816(acc[nt], a, bfrag[kh][nt]);
        }
        // pixel ow0+g -> cell g/2, sub-position sh*2 + g%2; pixel +8 -> cell +4. Cells are 272 B apart in staging.
        uint8_t* p_lo = my_stage + (g >> 1) * kC1CellPitch + (sh * 2 + (g & 1)) * 64 + 4 * tig;
        uint8_t* p_hi = p_lo + 4 * kC1CellPitch;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          const float v0 = fmaxf(acc[nt][0] + bia[nt][0], 0.0f);
          const float v1 = fmaxf(acc[nt][1] + bia[nt][1], 0.0f);
          const float v2 = fmaxf(acc[nt][2] + bia[nt][0], 0.0f);
          const float v3 = fmaxf(acc[nt][3] + bia[nt][1], 0.0f);
          *reinterpret_cast<__nv_bfloat162*>(p_lo + nt * 16) = __floats2bfloat162_rn(v0, v1);
          *reinterpret_cast<__nv_bfloat162*>(p_hi + nt * 16) = __floats2bfloat162_rn(v2, v3);
        }
      }
      __syncwarp();
      // 8 cells x 256 B = 128 chunks of 16 B, contiguous in global memory
      uint4* dst = reinterpret_cast<uint4*>(out_f + ((size_t)j * 16 + (ow0 >> 1)) * 128);
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        const int q = it * 32 + lane;
        dst[q] = *reinterpret_cast<const uint4*>(my_stage + (q >> 4) * kC1CellPitch + (q & 15) * 16);
      }
      __syncwarp();
    }
    __syncthreads();  // before the next frame overwrites the tile
  }
}

}  // namespace vfp
