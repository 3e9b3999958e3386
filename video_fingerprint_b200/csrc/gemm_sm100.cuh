// Persistent, warp-specialised tcgen05 GEMM skeleton for sm_100a.
//
//   D[128 x BLOCK_N] (fp32, TMEM) = A[128 x K] (bf16, K-major) * B[BLOCK_N x K]^T (bf16, K-major)
//
//   warp 0      : TMA producer (one lane)            global -> swizzled smem ring, mbarrier complete_tx
//   warp 1      : TMEM allocator + UMMA issuer (one lane), tcgen05.commit releases smem stages
//   warps 2..5(9): epilogue; each warp owns one 32-lane quarter of the 128 accumulator rows (x half the columns) and
//                 drains them with tcgen05.ld while the issuer already fills the other accumulator
//                 buffer (two BLOCK_N-column buffers in TMEM).
//
// The A operand is fetched either as a plain 2-D row tile or as a strided 4-D box over an NHWC
// activation tensor (one 3x3/stride-2 filter tap per K block = implicit-GEMM convolution with the
// im2col done by the TMA unit, padding supplied by its out-of-bounds zero fill).
#pragma once
#include "sm100_primitives.cuh"

namespace vfp {

constexpr int kBlockM = 128;

// Epilogues that only do column-local work let two or four warps share one TMEM lane quarter (each takes a slice of
// the BLOCK_N columns); row-reducing epilogues keep one thread per row.
template <int BLOCK_N, class Epilogue>
constexpr int gemm_column_split() {
  return (Epilogue::kColumnSplit >= 4 && BLOCK_N >= 128) ? 4 : (Epilogue::kColumnSplit >= 2 && BLOCK_N >= 64) ? 2 : 1;
}
template <int BLOCK_N, class Epilogue>
constexpr int gemm_threads() { return 64 + 128 * gemm_column_split<BLOCK_N, Epilogue>(); }

struct GemmShape {
  int m_tiles;     // number of 128-row tiles
  int n_tiles;     // number of BLOCK_N column tiles
  int k_blocks;    // K / BLOCK_K
  int group_m;     // rasterisation: tiles are walked in groups of `group_m` row tiles (L2 reuse)
  // schedule 1 ("row-block resident", used by the top-k search): a work item is one 128-row tile x one of
  // `n_segments` contiguous column ranges; a CTA walks the item's column tiles in ascending order so a
  // row-reducing epilogue can keep per-row state across them. Concurrent CTAs stream the same columns -> L2 reuse.
  int row_resident;
  int n_segments;
  // A operand addressing
  int a_conv;           // 0: rows are GEMM rows; 1: 4-D box (C, W, H, frame) over an NHWC activation tensor
  int tiles_per_frame;  // conv: row tiles per frame (>=1) ...
  int frames_per_tile;  //       ... or frames per row tile (>=1)
  int tile_out_rows;    // conv: output rows (H) covered by one tile inside a frame
  int h_mul;            // conv: H coordinate of a tile = h_mul * first_output_row + tap_h[kb]
  // conv: per-K-block box origin (channel offset, W offset, H offset). One K block = one filter tap
  // (or a channel slice of it); the -1 entries address the zero halo the TMA unit fills in.
  signed char tap_c_blk[18];  // channel offset in units of BLOCK_K
  signed char tap_w[18];
  signed char tap_h[18];
};

__device__ __forceinline__ void tile_coords(const GemmShape& s, int t, int& mt, int& nt) {
  const int group_size = s.group_m * s.n_tiles;
  const int g = t / group_size;
  const int r = t - g * group_size;
  const int m_first = g * s.group_m;
  const int gm = min(s.group_m, s.m_tiles - m_first);
  mt = m_first + (r % gm);
  nt = r / gm;
}

// The tile sequence of one CTA; all three warp roles instantiate it and therefore see identical sequences.
struct TileWalk {
  const GemmShape& s;
  int cur, stride, limit;       // schedule 0: tile index; schedule 1: work-item index
  int nt, nt_end, mt, seg;      // schedule 1: position inside the item
  __device__ TileWalk(const GemmShape& shape, int cta, int n_cta)
      : s(shape), cur(cta), stride(n_cta), limit(shape.row_resident ? shape.m_tiles * shape.n_segments : shape.m_tiles * shape.n_tiles),
        nt(0), nt_end(0), mt(0), seg(0) {}
  // returns false when the CTA is done; first/last flag the first/last column tile of a work item
  __device__ bool next(int& out_mt, int& out_nt, bool& first, bool& last) {
    if (!s.row_resident) {
      if (cur >= limit) return false;
      tile_coords(s, cur, out_mt, out_nt);
      cur += stride;
      first = last = true;
      return true;
    }
    if (nt >= nt_end) {
      if (cur >= limit) return false;
      mt = cur / s.n_segments;
      seg = cur - mt * s.n_segments;
      const int per = (s.n_tiles + s.n_segments - 1) / s.n_segments;
      nt = seg * per;
      nt_end = min(nt + per, s.n_tiles);
      cur += stride;
      first = true;
      if (nt >= nt_end) { nt_end = nt + 1; }  // degenerate empty segment: still one (fully out-of-range) tile
    } else {
      first = false;
    }
    out_mt = mt;
    out_nt = nt;
    ++nt;
    last = nt >= nt_end;
    return true;
  }
};

template <int BLOCK_N, int BLOCK_K, int STAGES, int MT = 1>
struct GemmSmemLayout {
  static constexpr int kRowBytes = BLOCK_K * 2;
  static constexpr int kABytes = kBlockM * kRowBytes;      // one 128-row sub-tile of A
  static constexpr int kAStage = MT * kABytes;
  static constexpr int kBBytes = BLOCK_N * kRowBytes;
  static constexpr int kStageBytes = kAStage + kBBytes;
  static constexpr int kBarrierBytes = 256;
  static constexpr int kCore = STAGES * kStageBytes + kBarrierBytes;
  static constexpr int kCoreAligned = (kCore + 1023) / 1024 * 1024;  // epilogue staging starts 1024-aligned
  static constexpr int kTotal = kCoreAligned + 1024 /*alignment slack*/;
};

// MT > 1: one CTA tile = MT consecutive 128-row sub-tiles sharing the B tile, each with its own TMEM accumulator.
// UMMAs that accumulate into the SAME TMEM tile issue back to back only every ~180 cycles (measured: 24 dependent
// M128 N64 K16 instructions take 4300 cycles), which starves narrow tiles (N=64: 32 cycles of work per
// instruction). Round-robin over MT independent accumulators hides that latency.
template <int BLOCK_N, int BLOCK_K, int STAGES, class Epilogue, int MT = 1>
__global__ void __launch_bounds__(gemm_threads<BLOCK_N, Epilogue>(), 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                    const GemmShape shape_in, const __grid_constant__ typename Epilogue::Params ep) {
  using L = GemmSmemLayout<BLOCK_N, BLOCK_K, STAGES, MT>;
  static_assert(BLOCK_N % 32 == 0 && BLOCK_N >= 32 && BLOCK_N <= 256, "BLOCK_N");
  static_assert(BLOCK_K == 64 || BLOCK_K == 32 || BLOCK_K == 16, "BLOCK_K");
  static_assert(2 * MT * BLOCK_N <= 512, "TMEM: two accumulator buffers");
  constexpr int kAccCols = MT * BLOCK_N;  // columns of one accumulator buffer
  constexpr uint32_t kTmemCols = (2 * kAccCols <= 32) ? 32 : (2 * kAccCols <= 64) ? 64 : (2 * kAccCols <= 128) ? 128
                                 : (2 * kAccCols <= 256) ? 256 : 512;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + STAGES * L::kAStage;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * L::kStageBytes);
  uint64_t* full_bar = bars;                  // [STAGES]
  uint64_t* empty_bar = bars + STAGES;        // [STAGES]
  uint64_t* acc_full = bars + 2 * STAGES;     // [2]
  uint64_t* acc_empty = bars + 2 * STAGES + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // the tile walk runs over super-tiles of MT row tiles
  GemmShape shape = shape_in;
  const int m_tiles_real = shape_in.m_tiles;
  shape.m_tiles = (shape_in.m_tiles + MT - 1) / MT;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 4 * gemm_column_split<BLOCK_N, Epilogue>());  // one arrive per epilogue warp
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      TileWalk walk(shape, blockIdx.x, gridDim.x);
      int mts, nt;
      bool first, last;
      while (walk.next(mts, nt, first, last)) {
        int frame0[MT], oh0[MT];
#pragma unroll
        for (int sub = 0; sub < MT; ++sub) {
          const int mt = mts * MT + sub;
          frame0[sub] = 0;
          oh0[sub] = 0;
          if (shape.a_conv) {
            if (shape.tiles_per_frame > 1) {
              frame0[sub] = mt / shape.tiles_per_frame;
              oh0[sub] = (mt - frame0[sub] * shape.tiles_per_frame) * shape.tile_out_rows;
            } else {
              frame0[sub] = mt * shape.frames_per_tile;
            }
          }
        }
        for (int kb = 0; kb < shape.k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[stage], L::kStageBytes);
#pragma unroll
          for (int sub = 0; sub < MT; ++sub) {
            uint8_t* dst = smem_a + stage * L::kAStage + sub * L::kABytes;
            if (shape.a_conv) {
              tma_load_4d(&tmap_a, &full_bar[stage], dst, shape.tap_c_blk[kb] * BLOCK_K, shape.tap_w[kb],
                          shape.h_mul * oh0[sub] + shape.tap_h[kb], frame0[sub]);
            } else {
              tma_load_2d(&tmap_a, &full_bar[stage], dst, kb * BLOCK_K, (mts * MT + sub) * kBlockM);
            }
          }
          tma_load_2d(&tmap_b, &full_bar[stage], smem_b + stage * L::kBBytes, kb * BLOCK_K, nt * BLOCK_N);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ UMMA issuer ------------------------------
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(kBlockM, BLOCK_N);
      int stage = 0;
      uint32_t phase = 0;
      int local = 0;
      TileWalk walk(shape, blockIdx.x, gridDim.x);
      int mts, nt;
      bool first, last;
      for (; walk.next(mts, nt, first, last); ++local) {
        const int acc = local & 1;
        const uint32_t acc_phase = (local >> 1) & 1;
        mbar_wait(&acc_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * kAccCols;
        for (int kb = 0; kb < shape.k_blocks; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t bdesc = umma_smem_desc_kmajor<L::kRowBytes>(smem_u32(smem_b + stage * L::kBBytes));
          const uint32_t a_base = smem_u32(smem_a + stage * L::kAStage);
#pragma unroll
          for (int k = 0; k < BLOCK_K / 16; ++k) {
            // advancing 16 bf16 along K = 32 bytes = 2 units of the (addr >> 4) field
#pragma unroll
            for (int sub = 0; sub < MT; ++sub) {
              const uint64_t adesc = umma_smem_desc_kmajor<L::kRowBytes>(a_base + sub * L::kABytes);
              umma_bf16(d_tmem + sub * BLOCK_N, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            }
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&acc_full[acc]);
      }
    }
  } else {
    // ------------------------------ epilogue ------------------------------
    constexpr int kSplit = gemm_column_split<BLOCK_N, Epilogue>();
    constexpr int kColsPerWarp = BLOCK_N / kSplit;
    const int quarter = warp & 3;  // TMEM lane quarter this warp may touch
    const int row = quarter * 32 + lane;
    const int col_begin = ((warp - 2) >> 2) * kColsPerWarp;
    int local = 0;
    TileWalk walk(shape, blockIdx.x, gridDim.x);
    int mts, nt;
    bool first, last;
    Epilogue epi;
    uint8_t* extra_smem = smem + L::kCoreAligned;
    epi.setup(ep, extra_smem, warp - 2, lane);
    epi.set_block_n(BLOCK_N);
    for (; walk.next(mts, nt, first, last); ++local) {
      const int acc = local & 1;
      const uint32_t acc_phase = (local >> 1) & 1;
      if (first) epi.item_begin(ep, mts, walk.seg, row, extra_smem);
      mbar_wait(&acc_full[acc], acc_phase);
      tc_fence_after();
#pragma unroll 1
      for (int sub = 0; sub < MT; ++sub) {
        const int mt = mts * MT + sub;
        if (mt >= m_tiles_real) break;  // warp-uniform
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * kAccCols + sub * BLOCK_N;
        epi.begin(ep, mt, nt, row);
#pragma unroll 1
        for (int pass = 0; pass < Epilogue::kPasses; ++pass) {  // row-wise reductions re-read the accumulator
#pragma unroll 1
          for (int c = col_begin; c < col_begin + kColsPerWarp; c += 32) {
            uint32_t v[32];
            tmem_ld_32x32(taddr + c, v);
            tmem_ld_wait();
            epi.chunk(ep, mt, nt * BLOCK_N + c, row, v, pass);
          }
        }
        epi.end(ep, mt, nt, row);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[acc]);
      if (last) epi.item_end(ep, mts, walk.seg, row, extra_smem);
    }
    epi.finish(ep, lane);
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// =================================================================================================
// B-resident variant. The profiles of the kernel above show it is bound by operand fill (L2 -> SMEM through
// TMA, ~40-48 B/clk/SM), not by the MMA pipe: every 128-row tile re-fetches its whole B tile. Here the B operand
// of the current column tile (all KB K-blocks: conv filters, a 256x256 weight block, a database tile of the join)
// stays in shared memory while the CTA sweeps a CONTIGUOUS run of row tiles, so only A streams through the ring.
// Tiles are numbered column-tile-major (u = nt * m_tiles + mt) and each CTA takes one contiguous range, hence
// B is (re)loaded only when the range crosses into the next column tile.
// =================================================================================================
template <int BLOCK_N, int BLOCK_K, int STAGES, int KB>
struct GemmBresSmemLayout {
  static constexpr int kRowBytes = BLOCK_K * 2;
  static constexpr int kABytes = kBlockM * kRowBytes;
  static constexpr int kBBytes = BLOCK_N * kRowBytes;  // one K block of B
  static constexpr int kCore = STAGES * kABytes + KB * kBBytes + 256;
  static constexpr int kCoreAligned = (kCore + 1023) / 1024 * 1024;
  static constexpr int kTotal = kCoreAligned + 1024;
};

template <int BLOCK_N, int BLOCK_K, int STAGES, int KB, class Epilogue>
__global__ void __launch_bounds__(gemm_threads<BLOCK_N, Epilogue>(), 1)
gemm_bres_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                         const GemmShape shape, const __grid_constant__ typename Epilogue::Params ep) {
  using L = GemmBresSmemLayout<BLOCK_N, BLOCK_K, STAGES, KB>;
  constexpr uint32_t kTmemCols = (2 * BLOCK_N <= 32) ? 32 : (2 * BLOCK_N <= 64) ? 64 : (2 * BLOCK_N <= 128) ? 128
                                 : (2 * BLOCK_N <= 256) ? 256 : 512;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + STAGES * L::kABytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * L::kABytes + KB * L::kBBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + STAGES;
  uint64_t* acc_full = bars + 2 * STAGES;
  uint64_t* acc_empty = bars + 2 * STAGES + 2;
  uint64_t* b_full = bars + 2 * STAGES + 4;
  uint64_t* b_empty = bars + 2 * STAGES + 5;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 6);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const long long total = (long long)shape.m_tiles * shape.n_tiles;
  const long long per = (total + gridDim.x - 1) / gridDim.x;
  const long long u0 = (long long)blockIdx.x * per;
  const long long u1 = min(total, u0 + per);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 4 * gemm_column_split<BLOCK_N, Epilogue>());
    }
    mbar_init(b_full, 1);
    mbar_init(b_empty, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0, cur_nt = -1;
      uint32_t phase = 0, b_phase = 0;
      for (long long u = u0; u < u1; ++u) {
        const int nt = (int)(u / shape.m_tiles);
        const int mt = (int)(u - (long long)nt * shape.m_tiles);
        if (nt != cur_nt) {
          if (cur_nt >= 0) {  // the MMAs of the previous column tile must have drained before B is overwritten
            mbar_wait(b_empty, b_phase);
            b_phase ^= 1;
          }
          mbar_arrive_expect_tx(b_full, KB * L::kBBytes);
          for (int kb = 0; kb < KB; ++kb)
            tma_load_2d(&tmap_b, b_full, smem_b + kb * L::kBBytes, kb * BLOCK_K, nt * BLOCK_N);
          cur_nt = nt;
        }
        int frame0 = 0, oh0 = 0;
        if (shape.a_conv) {
          if (shape.tiles_per_frame > 1) {
            frame0 = mt / shape.tiles_per_frame;
            oh0 = (mt - frame0 * shape.tiles_per_frame) * shape.tile_out_rows;
          } else {
            frame0 = mt * shape.frames_per_tile;
          }
        }
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[stage], L::kABytes);
          if (shape.a_conv) {
            tma_load_4d(&tmap_a, &full_bar[stage], smem_a + stage * L::kABytes, shape.tap_c_blk[kb] * BLOCK_K,
                        shape.tap_w[kb], shape.h_mul * oh0 + shape.tap_h[kb], frame0);
          } else {
            tma_load_2d(&tmap_a, &full_bar[stage], smem_a + stage * L::kABytes, kb * BLOCK_K, mt * kBlockM);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(kBlockM, BLOCK_N);
      int stage = 0, cur_nt = -1, local = 0;
      uint32_t phase = 0, b_phase = 0;
      for (long long u = u0; u < u1; ++u, ++local) {
        const int nt = (int)(u / shape.m_tiles);
        if (nt != cur_nt) {
          mbar_wait(b_full, b_phase);
          b_phase ^= 1;
          cur_nt = nt;
        }
        const int acc = local & 1;
        const uint32_t acc_phase = (local >> 1) & 1;
        mbar_wait(&acc_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
#pragma unroll 1
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t adesc = umma_smem_desc_kmajor<L::kRowBytes>(smem_u32(smem_a + stage * L::kABytes));
          const uint64_t bdesc = umma_smem_desc_kmajor<L::kRowBytes>(smem_u32(smem_b + kb * L::kBBytes));
#pragma unroll
          for (int k = 0; k < BLOCK_K / 16; ++k) umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&acc_full[acc]);
        if (u + 1 < u1 && (int)((u + 1) / shape.m_tiles) != nt) umma_commit(b_empty);
      }
    }
  } else {
    constexpr int kSplit = gemm_column_split<BLOCK_N, Epilogue>();
    constexpr int kColsPerWarp = BLOCK_N / kSplit;
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int col_begin = ((warp - 2) >> 2) * kColsPerWarp;
    int local = 0;
    Epilogue epi;
    epi.setup(ep, smem + L::kCoreAligned, warp - 2, lane);
    epi.set_block_n(BLOCK_N);
    for (long long u = u0; u < u1; ++u, ++local) {
      const int nt = (int)(u / shape.m_tiles);
      const int mt = (int)(u - (long long)nt * shape.m_tiles);
      const int acc = local & 1;
      const uint32_t acc_phase = (local >> 1) & 1;
      mbar_wait(&acc_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BLOCK_N;
      epi.begin(ep, mt, nt, row);
#pragma unroll 1
      for (int pass = 0; pass < Epilogue::kPasses; ++pass) {
#pragma unroll 1
        for (int c = col_begin; c < col_begin + kColsPerWarp; c += 32) {
          uint32_t v[32];
          tmem_ld_32x32(taddr + c, v);
          tmem_ld_wait();
          epi.chunk(ep, mt, nt * BLOCK_N + c, row, v, pass);
        }
      }
      epi.end(ep, mt, nt, row);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[acc]);
    }
    epi.finish(ep, lane);
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// =================================================================================================
// A-resident, panel-major schedule of the all-pairs similarity join (vfp_join_threshold).
// The plain kernel above re-fetches BOTH operands for every 128 x 256 tile: 192 KB per 2 048 MMA cycles = 94 B/clk per SM,
// above what L2 -> SM delivers, so the join ran at 0.59-0.75 of the tensor peak. Here a work item is
//      (a super-tile of kAresMT x 128 query rows) x (one PANEL of database column tiles),
// the query super-tile (all K blocks) is loaded ONCE per item and stays in shared memory, and only the database streams
// through the ring in blocks of 64 columns.
// Items are numbered PANEL-MAJOR and dealt round-robin, so at any time all CTAs work inside the same one or two panels:
// a panel (<= 65 536 database rows = 32 MB of bf16) is read from HBM once and then served from L2 however far the CTAs
// drift apart; a row-major order would let 148 CTAs stream 148 different parts of a database that does not fit L2.
// `tri` (self joins): S is symmetric, so column tiles that lie entirely below the diagonal of the item's rows are
// skipped; the epilogue keeps j >= i and the re-score kernel emits the mirrored pair.
// =================================================================================================
// KB (template parameter of the kernel) = resident K blocks of 64 columns, ceil(dim / 64): 4 for the 256-wide embeddings the
// models produce by default. Columns past dim in the last block are zero-filled by the TMA unit and add +0 to every score.
constexpr int kAresMT = 2;

struct AresShape {
  int m_super;        // super-tiles of kAresMT * 128 query rows
  int n_tiles;        // database column tiles of block_n rows
  int panel_tiles;    // column tiles per panel
  int n_panels;
  int tri;            // 1: skip column tiles strictly below the diagonal
  long long q_row0;   // global index of query row 0 (position of the diagonal)
  int block_n;        // database rows per column tile (kAres2BlockN)
};

struct AresWalk {
  const AresShape& s;
  long long cur, stride, limit;
  __device__ AresWalk(const AresShape& shape, int cta, int n_cta)
      : s(shape), cur(cta), stride(n_cta), limit((long long)shape.m_super * shape.n_panels) {}
  // next non-empty item of this CTA: super-tile index and its column tile range [nt0, nt1)
  __device__ bool next(int& mts, int& nt0, int& nt1) {
    while (cur < limit) {
      const int p = (int)(cur / s.m_super);
      mts = (int)(cur - (long long)p * s.m_super);
      cur += stride;
      nt0 = p * s.panel_tiles;
      nt1 = min(s.n_tiles, nt0 + s.panel_tiles);
      if (s.tri) nt0 = max(nt0, (int)((s.q_row0 + (long long)mts * (kAresMT * kBlockM)) / s.block_n));
      if (nt0 < nt1) return true;
    }
    return false;
  }
};

// =================================================================================================
// CTA-pair version of the A-resident join kernel (tcgen05 cta_group::2). An SS-mode UMMA streams both operands from shared
// memory: (128 + N) rows x 32 B per instruction, i.e. 128 B/clk at M128 N128 - the whole shared-memory port, with the TMA
// fill (32 B/clk) on top; that is what held a single-CTA version of this schedule (M128 N128 UMMAs, 256 resident query
// rows) at 0.74 of the tensor peak. A pair of CTAs issues
// ONE UMMA of M = 256, N = 256: each SM computes its 128 query rows against all 256 database rows but keeps only 128 of
// them (16 KB per K block) in its own shared memory and reads the peer's half over the pair link: 64 B/clk of operand
// reads + 32 B/clk of fill per SM.
//   work item = (256 query rows: 128 per CTA, resident) x (one panel of 256-row database tiles), panel-major as above
//   leader CTA (cluster rank 0): its warp 1 issues every UMMA and commits to BOTH CTAs' barriers (multicast commit);
//   both producers load their own query rows and their half of each database tile, the byte counts land on the LEADER's
//   full barriers; both CTAs' epilogue warps drain their own TMEM and arrive on the LEADER's acc_empty barrier.
// =================================================================================================
constexpr int kAres2BlockN = 256;

template <int STAGES, int KB>
struct Ares2SmemLayout {
  static constexpr int kABytes = kBlockM * 128;                   // one K block of this CTA's 128 query rows
  static constexpr int kAResident = KB * kABytes;                 // 16 KB per K block (64 KB at KB = 4)
  static constexpr int kBBytes = (kAres2BlockN / 2) * 128;        // this CTA's half of one K block of a database tile
  static constexpr int kCore = kAResident + STAGES * kBBytes + 256;
  static constexpr int kCoreAligned = (kCore + 1023) / 1024 * 1024;
  static constexpr int kTotal = kCoreAligned + 1024;
};

template <int STAGES, int KB, class Epilogue>
__global__ void __launch_bounds__(gemm_threads<kAres2BlockN, Epilogue>(), 1)
gemm_ares2_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                          const AresShape shape, const __grid_constant__ typename Epilogue::Params ep) {
  using L = Ares2SmemLayout<STAGES, KB>;
  constexpr int kEpiWarps = 4 * gemm_column_split<kAres2BlockN, Epilogue>();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + L::kAResident;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kAResident + STAGES * L::kBBytes);
  uint64_t* full_bar = bars;                       // leader's are used (bytes of both CTAs)
  uint64_t* empty_bar = bars + STAGES;             // per CTA, fed by the leader's multicast commits
  uint64_t* acc_full = bars + 2 * STAGES;          // per CTA (multicast commit)
  uint64_t* acc_empty = bars + 2 * STAGES + 2;     // leader's: 2 x kEpiWarps arrivals
  uint64_t* a_full = bars + 2 * STAGES + 4;        // leader's
  uint64_t* a_empty = bars + 2 * STAGES + 5;       // per CTA (multicast commit)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 6);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 2 * kEpiWarps);
    }
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc_2cta(tmem_slot, 512);
    tmem_relinquish_2cta();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // both CTAs' barriers and TMEM exist before any cross-CTA traffic
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;

  if (warp == 0) {
    // ------------------------------ TMA producer (both CTAs) ------------------------------
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0, a_phase = 0;
      AresWalk walk(shape, pair, n_pairs);
      int mts, nt0, nt1;
      const uint32_t a_full_leader = mapa_u32(a_full, 0);
      while (walk.next(mts, nt0, nt1)) {
        mbar_wait(a_empty, a_phase ^ 1);
        a_phase ^= 1;
        if (leader) mbar_arrive_expect_tx(a_full, 2 * L::kAResident);
#pragma unroll
        for (int kb = 0; kb < KB; ++kb)
          tma_load_2d_2cta(&tmap_a, a_full_leader, smem_a + kb * L::kABytes, kb * 64, (mts * 2 + (int)crank) * kBlockM);
        for (int nt = nt0; nt < nt1; ++nt) {
#pragma unroll
          for (int kb = 0; kb < KB; ++kb) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * L::kBBytes);
            tma_load_2d_2cta(&tmap_b, mapa_u32(&full_bar[stage], 0), smem_b + stage * L::kBBytes, kb * 64,
                             nt * kAres2BlockN + (int)crank * (kAres2BlockN / 2));
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ UMMA issuer (leader CTA only) ------------------------------
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = umma_idesc_bf16(2 * kBlockM, kAres2BlockN);
      int stage = 0, local = 0;
      uint32_t phase = 0, a_phase = 0;
      AresWalk walk(shape, pair, n_pairs);
      int mts, nt0, nt1;
      const uint32_t a_base = smem_u32(smem_a);
      while (walk.next(mts, nt0, nt1)) {
        mbar_wait(a_full, a_phase);
        a_phase ^= 1;
        tc_fence_after();
        for (int nt = nt0; nt < nt1; ++nt, ++local) {
          const int acc = local & 1;
          mbar_wait(&acc_empty[acc], ((local >> 1) & 1) ^ 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * kAres2BlockN;
#pragma unroll
          for (int kb = 0; kb < KB; ++kb) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint64_t adesc = umma_smem_desc_kmajor<128>(a_base + kb * L::kABytes);
            const uint64_t bdesc = umma_smem_desc_kmajor<128>(smem_u32(smem_b + stage * L::kBBytes));
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16_2cta(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            umma_commit_2cta(&empty_bar[stage], 3);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
          umma_commit_2cta(&acc_full[acc], 3);
        }
        umma_commit_2cta(a_empty, 3);
      }
    }
  } else {
    // ------------------------------ epilogue (both CTAs, own TMEM half) ------------------------------
    constexpr int kSplit = gemm_column_split<kAres2BlockN, Epilogue>();
    constexpr int kColsPerWarp = kAres2BlockN / kSplit;
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int col_begin = ((warp - 2) >> 2) * kColsPerWarp;
    int local = 0;
    AresWalk walk(shape, pair, n_pairs);
    int mts, nt0, nt1;
    Epilogue epi;
    epi.setup(ep, smem + L::kCoreAligned, warp - 2, lane);
    const uint32_t acc_empty_leader[2] = {mapa_u32(&acc_empty[0], 0), mapa_u32(&acc_empty[1], 0)};
    while (walk.next(mts, nt0, nt1)) {
      const int mt = mts * 2 + (int)crank;   // this CTA's 128-row tile
      for (int nt = nt0; nt < nt1; ++nt, ++local) {
        const int acc = local & 1;
        mbar_wait(&acc_full[acc], (local >> 1) & 1);
        tc_fence_after();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * kAres2BlockN;
        epi.begin(ep, mt, nt, row);
#pragma unroll 1
        for (int c = col_begin; c < col_begin + kColsPerWarp; c += 32) {
          uint32_t v[32];
          tmem_ld_32x32(taddr + c, v);
          tmem_ld_wait();
          epi.chunk(ep, mt, nt * kAres2BlockN + c, row, v, 0);
        }
        epi.end(ep, mt, nt, row);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(acc_empty_leader[acc]);
      }
    }
    epi.finish(ep, lane);
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2cta(tmem_base, 512);
  }
}

// =================================================================================================
// CTA-pair version of the generic kernel (tcgen05 cta_group::2): one UMMA of M = 256, N = 256 per K step for a PAIR of
// neighbouring 128-row tiles. Each CTA loads its own A tile and HALF of the B tile (128 of the 256 rows) per K block, so a
// stage is 32 KB instead of 48 KB, the shared-memory port carries 64 B/clk of operand reads instead of 96 B/clk, and six
// stages fit where four did. Same roles and schedule as gemm_tcgen05_kernel (plain tile order, A as rows or as a 4-D
// convolution box); the leader CTA (cluster rank 0) issues, commits are multicast, both producers report their bytes to
// the leader's full barriers, both CTAs' epilogue warps drain their own TMEM and arrive on the leader's acc_empty.
// =================================================================================================
template <int BLOCK_K, int STAGES>
struct GemmPairSmemLayout {
  static constexpr int kRowBytes = BLOCK_K * 2;
  static constexpr int kABytes = kBlockM * kRowBytes;
  static constexpr int kBBytes = 128 * kRowBytes;          // this CTA's half of the 256-row B tile
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kCore = STAGES * kStageBytes + 256;
  static constexpr int kCoreAligned = (kCore + 1023) / 1024 * 1024;
  static constexpr int kTotal = kCoreAligned + 1024;
};

template <int BLOCK_K, int STAGES, class Epilogue>
__global__ void __launch_bounds__(gemm_threads<256, Epilogue>(), 1)
gemm_pair_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                         const GemmShape shape_in, const __grid_constant__ typename Epilogue::Params ep) {
  constexpr int BLOCK_N = 256;
  using L = GemmPairSmemLayout<BLOCK_K, STAGES>;
  constexpr int kEpiWarps = 4 * gemm_column_split<BLOCK_N, Epilogue>();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + STAGES * L::kABytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * L::kStageBytes);
  uint64_t* full_bar = bars;                     // leader's are used (bytes of both CTAs)
  uint64_t* empty_bar = bars + STAGES;           // per CTA (multicast commit)
  uint64_t* acc_full = bars + 2 * STAGES;        // per CTA (multicast commit)
  uint64_t* acc_empty = bars + 2 * STAGES + 2;   // leader's: 2 x kEpiWarps arrivals
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  GemmShape shape = shape_in;
  const int m_tiles_real = shape_in.m_tiles;
  shape.m_tiles = (shape_in.m_tiles + 1) / 2;   // the walk runs over pairs of row tiles
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 2 * kEpiWarps);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc_2cta(tmem_slot, 512);
    tmem_relinquish_2cta();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------ TMA producer (both CTAs) ------------------------------
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      TileWalk walk(shape, pair, n_pairs);
      int mp, nt;
      bool first, last;
      while (walk.next(mp, nt, first, last)) {
        const int mt = mp * 2 + (int)crank;
        int frame0 = 0, oh0 = 0;
        if (shape.a_conv) {
          if (shape.tiles_per_frame > 1) {
            frame0 = mt / shape.tiles_per_frame;
            oh0 = (mt - frame0 * shape.tiles_per_frame) * shape.tile_out_rows;
          } else {
            frame0 = mt * shape.frames_per_tile;
          }
        }
        for (int kb = 0; kb < shape.k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * L::kStageBytes);
          const uint32_t full_leader = mapa_u32(&full_bar[stage], 0);
          uint8_t* dst = smem_a + stage * L::kABytes;
          if (shape.a_conv) {
            tma_load_4d_2cta(&tmap_a, full_leader, dst, shape.tap_c_blk[kb] * BLOCK_K, shape.tap_w[kb],
                             shape.h_mul * oh0 + shape.tap_h[kb], frame0);
          } else {
            tma_load_2d_2cta(&tmap_a, full_leader, dst, kb * BLOCK_K, mt * kBlockM);
          }
          tma_load_2d_2cta(&tmap_b, full_leader, smem_b + stage * L::kBBytes, kb * BLOCK_K, nt * BLOCK_N + (int)crank * 128);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ UMMA issuer (leader CTA only) ------------------------------
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = umma_idesc_bf16(2 * kBlockM, BLOCK_N);
      int stage = 0;
      uint32_t phase = 0;
      int local = 0;
      TileWalk walk(shape, pair, n_pairs);
      int mp, nt;
      bool first, last;
      for (; walk.next(mp, nt, first, last); ++local) {
        const int acc = local & 1;
        mbar_wait(&acc_empty[acc], ((local >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
        for (int kb = 0; kb < shape.k_blocks; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint64_t adesc = umma_smem_desc_kmajor<L::kRowBytes>(smem_u32(smem_a + stage * L::kABytes));
          const uint64_t bdesc = umma_smem_desc_kmajor<L::kRowBytes>(smem_u32(smem_b + stage * L::kBBytes));
#pragma unroll
          for (int k = 0; k < BLOCK_K / 16; ++k) umma_bf16_2cta(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit_2cta(&empty_bar[stage], 3);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit_2cta(&acc_full[acc], 3);
      }
    }
  } else {
    // ------------------------------ epilogue (both CTAs, own 128 rows) ------------------------------
    constexpr int kSplit = gemm_column_split<BLOCK_N, Epilogue>();
    constexpr int kColsPerWarp = BLOCK_N / kSplit;
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int col_begin = ((warp - 2) >> 2) * kColsPerWarp;
    int local = 0;
    TileWalk walk(shape, pair, n_pairs);
    int mp, nt;
    bool first, last;
    Epilogue epi;
    uint8_t* extra_smem = smem + L::kCoreAligned;
    epi.setup(ep, extra_smem, warp - 2, lane);
    epi.set_block_n(BLOCK_N);
    const uint32_t acc_empty_leader[2] = {mapa_u32(&acc_empty[0], 0), mapa_u32(&acc_empty[1], 0)};
    for (; walk.next(mp, nt, first, last); ++local) {
      const int mt = mp * 2 + (int)crank;
      const int acc = local & 1;
      mbar_wait(&acc_full[acc], (local >> 1) & 1);
      tc_fence_after();
      if (mt < m_tiles_real) {   // the odd tile out of the last pair has no rows: nothing to write (warp-uniform, whole CTA)
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BLOCK_N;
        epi.begin(ep, mt, nt, row);
#pragma unroll 1
        for (int pass = 0; pass < Epilogue::kPasses; ++pass) {
#pragma unroll 1
          for (int c = col_begin; c < col_begin + kColsPerWarp; c += 32) {
            uint32_t v[32];
            tmem_ld_32x32(taddr + c, v);
            tmem_ld_wait();
            epi.chunk(ep, mt, nt * BLOCK_N + c, row, v, pass);
          }
        }
        epi.end(ep, mt, nt, row);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(acc_empty_leader[acc]);
    }
    epi.finish(ep, lane);
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2cta(tmem_base, 512);
  }
}

}  // namespace vfp
