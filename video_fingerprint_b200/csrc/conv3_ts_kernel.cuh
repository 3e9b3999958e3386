// conv3 (64 -> 128 channels, 3x3 stride 2, 16x16 -> 8x8, model.py:107-109) with the FILTERS IN TENSOR MEMORY.
//
// The generic GEMM kernel ran this layer with the channels on M and four frames' pixels on N: every UMMA then streamed
// 4 KB of filters and 8 KB of pixels from shared memory, and every K block was refilled by TMA with 16 KB of filters + 32 KB of
// pixels: 96 B/clk of operand reads + 96 B/clk of fill against a 128 B/clk shared-memory port - the layer sat at 54 % tensor
// utilisation (ncu) with the port as the wall (multicasting the filter tile across a CTA pair did not help: the bytes still
// land in every CTA's shared memory). The filters are only 128 x 576 bf16 = 288 TMEM columns, so here they are written to
// tensor memory ONCE per CTA (tcgen05.st, lane = output channel) and every UMMA takes its A operand from there (TS mode, as
// conv1 of the stem does): shared memory only carries the pixels, 6 KB of operand reads per UMMA + 24 KB of fill per K block.
// What is left of the 512 columns holds ONE accumulator of 192 columns = three frames' 8 x 8 output pixels, so the
// accumulator cannot be double buffered: the UMMAs of the next tile start when the epilogue warps have pulled the previous
// one into registers (96 values per thread), the bias / ReLU / transposed staging / TMA store then overlap the next tile.
//
//   warp 0      TMA producer: per tile nine 4-D boxes (one per filter tap) of 3 frames x 8 x 8 pixels x 64 channels, stride 2,
//               halo zero-filled by the TMA unit, through a ring of 24 KB stages
//   warp 1      TMEM allocation + UMMA issuer: 9 x 4 UMMAs M128 N192 K16 per tile
//   warps 2-9   filter preload (once), then epilogue: TMEM lane quarter = warp % 4 (32 channels), pixel half = (warp - 2) / 4
#pragma once
#include "epilogues.cuh"
#include "stem_ts_kernel.cuh"

namespace vfp {

constexpr int kC3Frames = 3;                       // frames per tile
constexpr int kC3Pixels = kC3Frames * 64;          // accumulator columns
constexpr int kC3StageBytes = kC3Pixels * 128;     // 24 KB: 192 pixel rows x 64 channels
constexpr int kC3ColW = 0, kC3ColAcc = 288;        // TMEM: filters 9 taps x 32 columns | accumulator 192 columns
constexpr int kC3Threads = 64 + 256;

template <int STAGES>
struct Conv3Smem {
  static constexpr int kRing = 0;
  static constexpr int kStage = STAGES * kC3StageBytes;      // epilogue staging: 8 warps x 2 x 2 KB
  static constexpr int kBars = kStage + 8 * 2 * 2048;
  static constexpr int kTotal = kBars + 256 + 1024;
};

struct Conv3Params {
  alignas(64) CUtensorMap tmap_in;    // c2 [frames][16][16][64] bf16: box 64 ch x 8 (stride 2) x 8 (stride 2) x 3 frames, SWIZZLE_128B
  alignas(64) CUtensorMap tmap_out;   // c3 [frames * 64 pixels][128] bf16, box 32 channels x 32 pixels, SWIZZLE_64B
  const __nv_bfloat16* w;             // [128][576] bf16, K = (kh * 3 + kw) * 64 + c, BatchNorm folded
  const float* bias;                  // [128]
  int n_tiles;                        // ceil(frames / 3)
};

template <int STAGES>
__global__ void __launch_bounds__(kC3Threads, 1) conv3_ts_kernel(const __grid_constant__ Conv3Params p) {
  using L = Conv3Smem<STAGES>;
  static_assert(L::kTotal <= 232448, "conv3 kernel shared memory");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* ring = smem + L::kRing;
  uint8_t* stagebuf = smem + L::kStage;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kBars);
  uint64_t* full = bars;                 // [STAGES]
  uint64_t* empty = bars + STAGES;       // [STAGES]
  uint64_t* acc_full = bars + 2 * STAGES;
  uint64_t* acc_empty = acc_full + 1;    // 8 arrivals: every epilogue warp holds its part of the accumulator in registers
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmap_in);
    tma_prefetch_desc(&p.tmap_out);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 8);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // ---- filters -> tensor memory: lane (= accumulator row) c holds output channel c; a K step of 16 is 8 columns ----
  if (warp >= 2 && warp < 6) {
    const int ch = (warp & 3) * 32 + lane;
    const uint4* src = reinterpret_cast<const uint4*>(p.w + (size_t)ch * 576);
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>((warp & 3) * 32) << 16) + kC3ColW;
#pragma unroll 1
    for (int tap = 0; tap < 9; ++tap) {
      uint32_t v[32];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint4 q = __ldg(src + tap * 8 + i);
        v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
      }
      tmem_st_32x32(lane_base + tap * 32, v);
    }
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      int stage = 0;
      uint32_t ph = 0;
      for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
        for (int tap = 0; tap < 9; ++tap) {
          mbar_wait(&empty[stage], ph ^ 1);
          mbar_arrive_expect_tx(&full[stage], kC3StageBytes);
          tma_load_4d(&p.tmap_in, &full[stage], ring + stage * kC3StageBytes, 0, tap % 3 - 1, tap / 3 - 1, t * kC3Frames);
          if (++stage == STAGES) { stage = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ UMMA issuer (A = filters in TMEM) ------------------------------
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(128, kC3Pixels);
      int stage = 0;
      uint32_t ph = 0, e_ph = 0;
      const uint32_t d_acc = tmem_base + kC3ColAcc;
      for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
        mbar_wait(acc_empty, e_ph ^ 1);
        e_ph ^= 1;
        tc_fence_after();
        for (int tap = 0; tap < 9; ++tap) {
          mbar_wait(&full[stage], ph);
          tc_fence_after();
          const uint32_t b_lo = desc_lo_sw128(smem_u32(ring + stage * kC3StageBytes));
          const uint32_t a_col = tmem_base + kC3ColW + tap * 32;
          if (tap == 0) umma_ts_lo<false>(d_acc, a_col, b_lo, idesc); else umma_ts_lo<true>(d_acc, a_col, b_lo, idesc);
#pragma unroll
          for (int k = 1; k < 4; ++k) umma_ts_lo<true>(d_acc, a_col + 8 * k, b_lo + 2 * k, idesc);
          umma_commit(&empty[stage]);
          if (++stage == STAGES) { stage = 0; ph ^= 1; }
        }
        umma_commit(acc_full);
      }
    }
  } else {
    // ------------------------------ epilogue: bias + ReLU, transposed to [pixel][channel], TMA store ------------------------------
    const int q = warp & 3;                // lane quarter = channels 32q ..
    const int half = (warp - 2) >> 2;      // pixels 96 half .. of the tile
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + kC3ColAcc + half * 96;
    const float b = __ldg(p.bias + q * 32 + lane);
    uint8_t* stage2 = stagebuf + (warp - 2) * 4096;
    uint32_t f_ph = 0;
    int buf = 0;
    const int chunk = lane >> 3;
    for (int t = blockIdx.x; t < p.n_tiles; t += gridDim.x) {
      mbar_wait(acc_full, f_ph);
      f_ph ^= 1;
      tc_fence_after();
      uint32_t v[3][32];
#pragma unroll
      for (int c = 0; c < 3; ++c) tmem_ld_32x32(taddr + c * 32, v[c]);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty);   // the accumulator is in registers: the next tile's UMMAs may start
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        uint8_t* dst = stage2 + buf * 2048;
        if (lane == 0) tma_store_wait_read<1>();   // the store that last used this buffer has read it
        __syncwarp();
        uint8_t* col = dst + (lane & 7) * 2;
#pragma unroll
        for (int i = 0; i < 32; ++i) {   // element (pixel i, channel lane) of a 32 x 32 tile with 64-byte rows, SWIZZLE_64B
          const float y = fmaxf(__uint_as_float(v[c][i]) + b, 0.0f);
          *reinterpret_cast<__nv_bfloat16*>(col + i * 64 + ((chunk ^ ((i >> 1) & 3)) << 4)) = __float2bfloat16(y);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&p.tmap_out, dst, q * 32, t * kC3Pixels + half * 96 + c * 32);   // rows past the last frame are clipped
          tma_store_commit();
        }
        buf ^= 1;
      }
    }
    if (lane == 0) tma_store_wait_read<0>();
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace vfp
