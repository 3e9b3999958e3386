// Fused frame-encoder stem, all-tcgen05 version: conv1 (3->32, k5 s2) runs on the 5th-gen tensor cores too, as a
// "TS" UMMA whose A operand (the im2col rows) lives in TENSOR MEMORY. The round-1 kernel computed conv1 with
// mma.sync: 1360 HMMA.16816 per frame keep the legacy tensor path busy for ~2750 cycles per frame (8.1 cycles per HMMA and
// SM sub-partition, profiles/r01_microbench_tensor_pipe.txt), during which conv2's UMMAs cannot run (and vice versa).
//
// conv1 as a GEMM the tensor core likes. C_in = 3 means an im2col row of one output pixel is 5 x 15 values that no
// TMA box / UMMA smem descriptor can address, and N = 32 output channels would leave a 128 x N x 16 UMMA at its ~46-cycle
// floor. So: (1) an A row is built IN REGISTERS by the thread that owns the row (aligned 8-byte shared loads from the
// zero-haloed HWC copy of the frame) and written to TMEM with tcgen05.st; (2) a row is a horizontal PAIR of output pixels
// (ow = 2cx, 2cx+1): the 7-pixel input window they share is read once and the weights of the two pixels are stacked
// along N (Toeplitz trick): N = 2 x 32 = 64. Per filter row kh a row holds 24 consecutive bf16 of the HWC tile starting
// at pixel 4cx-3 channel 1 (8-byte aligned): 2 don't-care values, the 7 x 3 window, 1 don't-care; K = 5 x 24 = 120 -> 128,
// the weight matrix is zero wherever a row value is not a tap of that output pixel. (3) K columns 120 / 121 of every row
// hold 1.0 and the matching weight rows hold the folded BatchNorm bias split into two bf16 (hi + lo, ~16 bits), so the
// accumulator already contains the bias and the epilogue is ReLU + pack + store.
//   GEMM per tile: M = 128 rows = 4 cell rows x 16 cells x 2 sub-rows (sh), N = 64 = (sw, 32 channels), K = 128
//   -> 8 UMMAs (M128 N64 K16, TS) of ~49 cycles; 4 tiles per frame = 1570 cycles instead of 2750.
// The accumulator row of thread (cell, sh) is exactly the 2 x 64 bytes conv2's A-operand buffers AL0 / AL1 need from it
// (see stem_common.cuh for those buffers and conv2's UMMA schedule).
//
// What bounds this kernel is the serial instruction stream of each role, not a pipe (scripts/dev_knockout.py, and
// tests/cuda/microbench_handoff.cu: an mbarrier hand-off costs 100-250 cycles): with every load, store and UMMA removed
// the barrier skeleton of the first version still took 2 us per frame. Hence two UMMA issuer warps (a unit's conv2 must not
// wait behind the next tiles' conv1 hand-offs and vice versa), descriptors built once, every TMEM buffer double buffered (conv2's two unshifted accumulators merged to make room), and
// no per-element work that the tensor core can do instead (the bias).
//
// One CTA per SM, persistent over frames, 24 warps:
//   WG0   warp 0        bulk-copy issuer (raw frame planes -> smem ring, L2 prefetch two frames ahead; each frame's address
//                       comes from the pass's frame address table), weights once (TMA)
//         warp 1        TMEM allocation + conv1 UMMA issuer (TS mode)
//         warp 2        transposer (raw planes -> HWC bf16 tile), with WG5
//         warp 3        conv2 UMMA issuer
//   WG1-2 warps 4-11    conv2 epilogue (TMEM -> bias, shifted-tap add, ReLU -> bf16 -> staging -> TMA store)
//   WG3   warps 12-15   conv1 generators: HWC tile -> registers -> TMEM A operand
//   WG4   warps 16-19   conv1 epilogue: TMEM D -> ReLU, bf16 -> conv2's A buffers (16-byte conflict-free stores)
//   WG5   warps 20-23   transposers
// TMEM (512 columns), everything double buffered: conv2 accumulators 2 x 128 (columns 0-63: all unshifted taps, kw = 1 and
// kw = 2, summed by the tensor core; 64-127: the kw = 0 taps the epilogue shifts by one cell), conv1 A 2 x 64, conv1 D 2 x 64.
#pragma once
#include "stem_common.cuh"

namespace vfp {

constexpr int kTsGenWarp0 = 12, kTsGenWarps = 4;
constexpr int kTsEpiWarp0 = 16, kTsEpiWarps = 4;
constexpr int kTsRawSlots = 3;
constexpr int kTsXposeWarp1 = 20, kTsXposeWarps = 5;         // warp 2 + WG5
constexpr int kTsABufs = 2;
constexpr int kTsColAcc = 0, kTsColA = 256, kTsColD = 384;  // TMEM column map: conv2 acc 2 x 128 | conv1 A 2 x 64 | conv1 D 2 x 64
// development knock-out mask (compile time, -DVFP_STEM_KNOCKOUT=mask): 1 no output store, 2 no transposition, 4 no frame
// copies, 8 no conv2 UMMAs, 16 no conv1 UMMAs, 32 no conv1-epilogue stores, 64 no generator loads, 128 no conv2-epilogue
// work, 256 no conv1-epilogue TMEM loads, 512 no generator TMEM stores (1023 = the bare barrier skeleton)
// development experiment (-DVFP_STEM_HALFB=1, wrong results): every UMMA of the stem reads half of its weight operand, which is what a CTA pair would read
#ifndef VFP_STEM_HALFB
#define VFP_STEM_HALFB 0
#endif
#ifndef VFP_STEM_KNOCKOUT
#define VFP_STEM_KNOCKOUT 0
#endif
constexpr int kTsKnock = VFP_STEM_KNOCKOUT;

struct StemTsSmem {
  static constexpr int kC1 = 0;                                          // 2 units of AL0 | AL1
  static constexpr int kW2 = kC1 + 2 * kStemUnitBytes;                   // conv2: 5 weight tiles of 64 rows x 128 B
  static constexpr int kW1 = kW2 + kStemWBlocks * 8192;                  // conv1: 2 weight tiles of 64 rows x 128 B
  static constexpr int kStage = kW1 + 2 * 8192;                          // 8 conv2-epilogue warps x 2 KB
  static constexpr int kRaw = kStage + kStemEpiWarps * 2048;             // raw frame planes
  static constexpr int kTile = kRaw + kTsRawSlots * kStemRawSlotBytes;   // 2 HWC tiles
  static constexpr int kBars = kTile + 2 * kStemTileBytes;
  static constexpr int kBias = kBars + 512;              // conv2 bias (64 floats): no L1 is left beside 225 KB of shared memory,
  static constexpr int kTotal = kBias + 256 + 1024;      // so a __ldg in the epilogue loop is an L2 round trip every time
};
static_assert(StemTsSmem::kTotal <= 232448, "stem TS kernel shared memory");
static_assert(StemTsSmem::kW2 % 1024 == 0 && StemTsSmem::kW1 % 1024 == 0 && StemTsSmem::kStage % 1024 == 0 && StemTsSmem::kRaw % 1024 == 0,
              "alignment");

struct StemTsParams {
  alignas(64) CUtensorMap tmap_w2;   // conv2 weights [64][320] bf16 (fused K order), box 64 x 64, SWIZZLE_128B
  alignas(64) CUtensorMap tmap_w1;   // conv1 stacked weights + bias rows [64][128] bf16, box 64 x 64, SWIZZLE_128B
  alignas(64) CUtensorMap tmap_out;  // conv2 output [frames*256][64] bf16, box 32 x 32, SWIZZLE_64B
  const unsigned long long* frame_addr;   // [n_frames] device address of each frame (16-byte aligned; token_map_kernel)
  int frame_dtype;
  long long n_frames;
  const float* c2_bias;  // [64]
};

// The upper word of every SWIZZLE_128B K-major descriptor of this kernel is the same constant; the lower word is
// (address >> 4) | LBO, so descriptors are advanced with one 32-bit add.
constexpr uint32_t kDescHiSw128 = (uint32_t)(((8ull * 128) >> 4) | (1ull << 14) | (2ull << 29));
__device__ __forceinline__ uint32_t desc_lo_sw128(uint32_t smem_addr) { return ((smem_addr & 0x3FFFFu) >> 4) | (1u << 16); }

// D[tmem] (+)= A[smem] * B[smem], descriptors given as 32-bit lower words (see kDescHiSw128); ACC is a compile-time flag
template <bool ACC>
__device__ __forceinline__ void umma_ss_lo(uint32_t tmem_d, uint32_t adesc_lo, uint32_t bdesc_lo, uint32_t idesc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 da, {%1, %4};\n\t"
      "mov.b64 db, {%2, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(adesc_lo), "r"(bdesc_lo), "r"(idesc), "r"(kDescHiSw128), "r"(ACC ? 1u : 0u)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]: the A rows come from tensor memory (lane = row, 2 bf16 per 32-bit column)
template <bool ACC>
__device__ __forceinline__ void umma_ts_lo(uint32_t tmem_d, uint32_t tmem_a, uint32_t bdesc_lo, uint32_t idesc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 db, {%2, %4};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "r"(bdesc_lo), "r"(idesc), "r"(kDescHiSw128), "r"(ACC ? 1u : 0u)
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
      "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]),
      "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]),
      "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__global__ void __launch_bounds__(kStemThreads, 1) stem_ts_kernel(const __grid_constant__ StemTsParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* c1buf = smem + StemTsSmem::kC1;
  uint8_t* w2buf = smem + StemTsSmem::kW2;
  uint8_t* w1buf = smem + StemTsSmem::kW1;
  uint8_t* stagebuf = smem + StemTsSmem::kStage;
  uint8_t* rawbuf = smem + StemTsSmem::kRaw;
  uint8_t* tilebuf = smem + StemTsSmem::kTile;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + StemTsSmem::kBars);
  uint64_t* w_full = bars;            // [1]
  uint64_t* c1_full = bars + 1;       // [2] conv1 epilogue -> conv2 issuer (unit buffer written)
  uint64_t* c1_empty = bars + 3;      // [2] conv2 issuer -> conv1 epilogue (conv2 of the unit has read the buffer)
  uint64_t* acc_full = bars + 28;     // [2] conv2 issuer -> conv2 epilogue
  uint64_t* acc_empty = bars + 30;    // [2] conv2 epilogue -> conv2 issuer
  uint64_t* tile_full = bars + 7;     // [2] transposers -> generators
  uint64_t* tile_empty = bars + 9;    // [2] generators -> transposers
  uint64_t* a_full = bars + 11;       // [3] generators -> conv1 issuer
  uint64_t* a_empty = bars + 14;      // [3] conv1 issuer -> generators
  uint64_t* d_full = bars + 17;       // [2] conv1 issuer -> conv1 epilogue
  uint64_t* d_empty = bars + 19;      // [2] conv1 epilogue -> conv1 issuer
  uint64_t* raw_full = bars + 32;     // [5] bulk copy -> transposers
  uint64_t* raw_empty = bars + 37;    // [5] transposers -> bulk copy issuer
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 42);
  float* c2_bias_s = reinterpret_cast<float*>(smem + StemTsSmem::kBias);

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  pdl_launch_dependents();
  // a conv pass is at most 16384 frames, so 32-bit counters are enough everywhere below
  const int n_local = (p.n_frames > blockIdx.x) ? (int)((p.n_frames - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;
  const int n_tiles = 4 * n_local, n_units = 2 * n_local;

  for (int i = tid; i < (2 * kStemUnitBytes) / 16; i += kStemThreads) reinterpret_cast<uint4*>(c1buf)[i] = make_uint4(0, 0, 0, 0);
  for (int i = tid; i < (2 * kStemTileBytes) / 16; i += kStemThreads) reinterpret_cast<uint4*>(tilebuf)[i] = make_uint4(0, 0, 0, 0);
  if (tid < 64) c2_bias_s[tid] = __ldg(p.c2_bias + tid);
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmap_w2);
    tma_prefetch_desc(&p.tmap_w1);
    tma_prefetch_desc(&p.tmap_out);
    mbar_init(w_full, 1);
    mbar_init(&c1_full[0], 2 * kTsEpiWarps);       // two tiles
    mbar_init(&c1_full[1], 2 * kTsEpiWarps + 1);   // + the halo cell row written by the warp that owns cell row 7
    for (int i = 0; i < 2; ++i) {
      mbar_init(&c1_empty[i], 1);
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], kStemEpiWarps);
      mbar_init(&tile_full[i], kTsXposeWarps);
      mbar_init(&tile_empty[i], kTsGenWarps);
      mbar_init(&d_full[i], 1);
      mbar_init(&d_empty[i], kTsEpiWarps);
    }
    for (int i = 0; i < kTsABufs; ++i) {
      mbar_init(&a_full[i], kTsGenWarps);
      mbar_init(&a_empty[i], 1);
    }
    for (int i = 0; i < kTsRawSlots; ++i) {
      mbar_init(&raw_full[i], 1);
      mbar_init(&raw_empty[i], kTsXposeWarps);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t plane_bytes = p.frame_dtype == kFrameBF16 ? 8192u : 4096u;
  pdl_wait();   // the previous conv pass (conv3 still reads the c2 buffer this kernel overwrites) must have completed

  // ------------------------------ transposers: raw planes -> HWC tile (warp 2 and WG5, ltid 0 .. 159) ------------------------------
  auto transposer_role = [&](int ltid) {
    int slot0 = 0;
    uint32_t n0 = 0;
    for (int li = 0; li < n_local; ++li) {
      const int t = li & 1;
      uint8_t* tile = tilebuf + t * kStemTileBytes;
      mbar_wait_lazy(&tile_empty[t], (uint32_t)(((li >> 1) & 1) ^ 1));
      const uint8_t* pl[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const uint32_t n = n0 + c;
        const int s = (slot0 + c) % kTsRawSlots;
        mbar_wait_lazy(&raw_full[s], (n / kTsRawSlots) & 1u);
        pl[c] = rawbuf + s * kStemRawSlotBytes;
      }
      if (!(kTsKnock & 2)) stem_transpose_frame(pl, tile, p.frame_dtype, ltid, kTsXposeWarps * 32);
      __syncwarp();
      if (lane == 0) {
#pragma unroll
        for (int c = 0; c < 3; ++c) mbar_arrive(&raw_empty[(slot0 + c) % kTsRawSlots]);
        mbar_arrive(&tile_full[t]);
      }
      slot0 = (slot0 + 3) % kTsRawSlots;
      n0 += 3;
    }
  };

  // register budget (768 threads x 80): WG0-2 56, WG3 112, WG4 96, WG5 56 -> 4*56 + 112 + 96 = 432 <= 480
  if (warp < kStemEpiWarp0) {
    setmaxnreg_dec<56>();
    if (warp == 0) {
      // ------------------------------ weights once, then the raw-plane ring ------------------------------
      if (lane == 0) {
        mbar_arrive_expect_tx(w_full, (kStemWBlocks + 2) * 8192);
        for (int kb = 0; kb < kStemWBlocks; ++kb) tma_load_2d(&p.tmap_w2, w_full, w2buf + kb * 8192, kb * 64, 0);
        for (int kb = 0; kb < 2; ++kb) tma_load_2d(&p.tmap_w1, w_full, w1buf + kb * 8192, kb * 64, 0);
        const unsigned long long* addr = p.frame_addr + blockIdx.x;   // this CTA's frames: addr[li * gridDim.x]
        int slot = 0;
        uint32_t ph = 0;
        for (int li = 0; li < n_local; ++li) {
          // one 8-byte load per frame: frames may sit anywhere (clip views, separate allocations), each one contiguous
          const uint8_t* src = reinterpret_cast<const uint8_t*>(__ldg(addr + (size_t)li * gridDim.x));
          // the ring only holds one frame, so a copy is issued about one frame time before its data is needed: pull the
          // frame after next into L2 now and the copy only pays the L2 latency
          if (li + 2 < n_local && !(kTsKnock & 4))
            bulk_prefetch_l2(reinterpret_cast<const uint8_t*>(__ldg(addr + (size_t)(li + 2) * gridDim.x)), 3 * plane_bytes);
          for (int c = 0; c < 3; ++c) {
            mbar_wait_lazy(&raw_empty[slot], ph ^ 1);
            if (kTsKnock & 4) {
              mbar_arrive(&raw_full[slot]);
            } else {
              mbar_arrive_expect_tx(&raw_full[slot], plane_bytes);
              bulk_copy_g2s(rawbuf + slot * kStemRawSlotBytes, src + c * plane_bytes, plane_bytes, &raw_full[slot]);
            }
            if (++slot == kTsRawSlots) { slot = 0; ph ^= 1; }
          }
        }
      }
    } else if (warp == 1) {
      // ------------------------------ conv1 UMMA issuer (TS mode) ------------------------------
      // the whole warp waits (a converged try_wait wakes up faster than a single-lane one), lane 0 issues
      constexpr uint32_t idesc64 = umma_idesc_bf16(128, VFP_STEM_HALFB ? 32 : 64);
      mbar_wait_relaxed(w_full, 0);
      const uint32_t w1_lo = desc_lo_sw128(smem_u32(w1buf));
      int ab = 0;
      uint32_t aph = 0;
      for (int g = 0; g < n_tiles; ++g) {
        const int b = g & 1;
        const uint32_t ph = (uint32_t)((g >> 1) & 1);
        mbar_wait_relaxed(&a_full[ab], aph);
        mbar_wait_relaxed(&d_empty[b], ph ^ 1);
        tc_fence_after();
        if (lane == 0) {
          const uint32_t a_col = tmem_base + kTsColA + ab * 64, d_col = tmem_base + kTsColD + b * 64;
          if (!(kTsKnock & 16)) {
            umma_ts_lo<false>(d_col, a_col, w1_lo, idesc64);
#pragma unroll
            for (int s = 1; s < 8; ++s) umma_ts_lo<true>(d_col, a_col + 8 * s, w1_lo + (s >> 2) * 512 + 2 * (s & 3), idesc64);
          }
          umma_commit(&a_empty[ab]);
          umma_commit(&d_full[b]);
        }
        __syncwarp();
        if (++ab == kTsABufs) { ab = 0; aph ^= 1; }
      }
    } else if (warp == 3) {
      // ------------------------------ conv2 UMMA issuer ------------------------------
      constexpr uint32_t idesc64 = umma_idesc_bf16(128, VFP_STEM_HALFB ? 32 : 64);
      constexpr uint32_t idesc128 = umma_idesc_bf16(128, VFP_STEM_HALFB ? 64 : 128);
      mbar_wait_relaxed(w_full, 0);
      const uint32_t w2_lo = desc_lo_sw128(smem_u32(w2buf));
      const uint32_t c1_lo = desc_lo_sw128(smem_u32(c1buf));
      for (int u = 0; u < n_units; ++u) {
        const int b = u & 1;
        const uint32_t ph = (uint32_t)((u >> 1) & 1);
        mbar_wait_relaxed(&acc_empty[b], ph ^ 1);
        mbar_wait_relaxed(&c1_full[b], ph);
        tc_fence_after();
        if (lane == 0) {
          // the four tap groups of stem_common.cuh, the unshifted ones sharing an accumulator: columns 0-63 collect the
          // kw = 1 taps (N = 64 UMMAs on AL0) AND the kw = 2 taps (first half of the stacked N = 128 UMMAs on AL1), columns
          // 64-127 the kw = 0 taps. Descriptor arithmetic in 16-byte units: K step 2, buffer cell row 128, weight block 512
          const uint32_t d_acc = tmem_base + kTsColAcc + b * 128;
          const uint32_t al0 = c1_lo + b * (kStemUnitBytes >> 4), al1 = al0 + (kStemABuf >> 4);
          if (!(kTsKnock & 8)) {
            umma_ss_lo<false>(d_acc, al1 + 128, w2_lo + 512, idesc128);               // G_BC k = 0 initialises all 128 columns
            umma_ss_lo<true>(d_acc, al0 + 128, w2_lo, idesc64);                       // G_A  k = 0
#pragma unroll
            for (int k = 1; k < 4; ++k) {
              umma_ss_lo<true>(d_acc, al0 + 128 + 2 * k, w2_lo + 2 * k, idesc64);            // G_A
              umma_ss_lo<true>(d_acc, al1 + 128 + 2 * k, w2_lo + 512 + 2 * k, idesc128);     // G_BC
            }
#pragma unroll
            for (int k = 0; k < 2; ++k) {
              umma_ss_lo<true>(d_acc, al0 + 2 * (2 + k), w2_lo + 3 * 512 + 2 * (2 + k), idesc64);   // G_D
              umma_ss_lo<true>(d_acc, al1 + 2 * k, w2_lo + 3 * 512 + 2 * k, idesc128);              // G_EF
            }
          }
          umma_commit(&c1_empty[b]);
          umma_commit(&acc_full[b]);
        }
        __syncwarp();
      }
    } else {
      transposer_role(lane);
    }
  } else if (warp < kTsGenWarp0) {
    // ------------------------------ conv2 epilogue ------------------------------
    setmaxnreg_dec<56>();
    const int quarter = warp & 3;
    const int col_half = (warp - kStemEpiWarp0) >> 2;
    const float keep = (lane & 15) == 0 ? 0.0f : 1.0f;
    const float2 keep2 = make_float2(keep, keep);
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + kTsColAcc + col_half * 32;
    // Output: bf16 rows staged in shared memory (swizzled, conflict-free 16-byte stores) and written by the TMA unit.
    // (Direct 16-byte global stores from the row-per-thread layout touch 32 lines per instruction: measured 25 % slower.)
    uint8_t* dst = stagebuf + (warp - kStemEpiWarp0) * 2048;
    uint8_t* r0 = dst + lane * 64;
    const int sw = (lane >> 1) & 3;
    int out_row = (int)blockIdx.x * 256 + quarter * 32;   // conv2 output row (pixel) of this warp's 32 rows, unit 0
    for (int u = 0; u < n_units; ++u) {
      const int b = u & 1;
      mbar_wait_relaxed(&acc_full[b], (uint32_t)((u >> 1) & 1));
      tc_fence_after();
      if (lane == 0) tma_store_wait_read<0>();
      __syncwarp();
      // software pipelined over the four 8-column chunks: the TMEM loads of chunk c+1 are in flight while chunk c is
      // shuffled, summed and stored (v0: kw = 1 and kw = 2 taps, v2: kw = 0 taps of the cell to the left)
      if (kTsKnock & 128) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[b]);
        continue;
      }
      uint32_t va[2][8], vb[2][8];
      tmem_ld_32x8(taddr + b * 128, va[0]);
      tmem_ld_32x8(taddr + b * 128 + 64, vb[0]);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint32_t(&v0)[8] = va[c & 1];
        uint32_t(&v2)[8] = vb[c & 1];
        tmem_ld_wait();
        if (c < 3) {
          tmem_ld_32x8(taddr + b * 128 + 8 * (c + 1), va[(c + 1) & 1]);
          tmem_ld_32x8(taddr + b * 128 + 64 + 8 * (c + 1), vb[(c + 1) & 1]);
        } else {  // everything this warp needs has left TMEM
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_empty[b]);
        }
        // y = v0 + bias + keep * shuffled(v2), two channels per instruction (FADD2 / FFMA2); keep = 0 for cell column 0, whose
        // left neighbour is the zero padding (the shuffle hands it cell 15 of the previous cell row)
        uint32_t q[4];
#pragma unroll
        for (int i = 0; i < 8; i += 4) {
          const float4 bb = *reinterpret_cast<const float4*>(c2_bias_s + col_half * 32 + 8 * c + i);
          const float s0 = __shfl_up_sync(0xffffffffu, __uint_as_float(v2[i]), 1), s1 = __shfl_up_sync(0xffffffffu, __uint_as_float(v2[i + 1]), 1);
          const float s2 = __shfl_up_sync(0xffffffffu, __uint_as_float(v2[i + 2]), 1), s3 = __shfl_up_sync(0xffffffffu, __uint_as_float(v2[i + 3]), 1);
          const float2 y01 = ffma2(make_float2(s0, s1), keep2, fadd2(make_float2(__uint_as_float(v0[i]), __uint_as_float(v0[i + 1])), make_float2(bb.x, bb.y)));
          const float2 y23 = ffma2(make_float2(s2, s3), keep2, fadd2(make_float2(__uint_as_float(v0[i + 2]), __uint_as_float(v0[i + 3])), make_float2(bb.z, bb.w)));
          q[i / 2] = relu_pack_bf16x2(y01.x, y01.y);
          q[i / 2 + 1] = relu_pack_bf16x2(y23.x, y23.y);
        }
        *reinterpret_cast<uint4*>(r0 + ((c ^ sw) << 4)) = make_uint4(q[0], q[1], q[2], q[3]);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0 && !(kTsKnock & 1)) {
        tma_store_2d(&p.tmap_out, dst, col_half * 32, out_row + (u & 1) * 128);
        tma_store_commit();
      }
      if (u & 1) out_row += (int)gridDim.x * 256;
    }
    if (lane == 0) tma_store_wait_read<0>();
  } else if (warp < kTsEpiWarp0) {
    // ------------------------------ conv1 generators ------------------------------
    setmaxnreg_inc<112>();
    const int q = warp & 3;            // TMEM lane quarter = cell row within the tile
    const int cx = lane & 15, sh = lane >> 4;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + kTsColA;
    // row (cell (cy, cx), sh) of tile t: cy = 4t + q, output row oh = 2cy + sh reads tile rows 2*oh + kh = 4cy + 2sh + kh;
    // 12 words from word 6cx + 8 of each (pixel 4cx-3 channel 1 .. pixel 4cx+5 channel 0)
    const uint8_t* lane_src = tilebuf + ((4 * q + 2 * sh) * 108 + 6 * cx + 8) * 4;
    int ab = 0;
    uint32_t aph = 0;
    for (int li = 0; li < n_local; ++li) {
      mbar_wait_relaxed(&tile_full[li & 1], (uint32_t)((li >> 1) & 1));
#pragma unroll 1
      for (int t = 0; t < 4; ++t) {
        const uint2* src = reinterpret_cast<const uint2*>(lane_src + (li & 1) * kStemTileBytes + t * (16 * 108 * 4));
        uint32_t v[64];
#pragma unroll
        for (int kh = 0; kh < 5; ++kh)
#pragma unroll
          for (int j = 0; j < 6; ++j) {
            const uint2 w = (kTsKnock & 64) ? make_uint2(0u, 0u) : src[kh * 54 + j];
            v[kh * 12 + 2 * j] = w.x;
            v[kh * 12 + 2 * j + 1] = w.y;
          }
        v[60] = 0x3F803F80u;   // K = 120, 121: 1.0 x (bias hi, bias lo)
        v[61] = 0u; v[62] = 0u; v[63] = 0u;
        if (t == 3) {  // this warp has read everything it needs from the frame's tile
          __syncwarp();
          if (lane == 0) mbar_arrive(&tile_empty[li & 1]);
        }
        mbar_wait_relaxed(&a_empty[ab], aph ^ 1);
        tc_fence_after();
        if (!(kTsKnock & 512)) {
          tmem_st_32x32(lane_base + ab * 64, v);
          tmem_st_32x32(lane_base + ab * 64 + 32, v + 32);
          tmem_st_wait();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&a_full[ab]);
        if (++ab == kTsABufs) { ab = 0; aph ^= 1; }
      }
    }
  } else if (warp < kTsEpiWarp0 + kTsEpiWarps) {
    // ------------------------------ conv1 epilogue ------------------------------
    setmaxnreg_inc<96>();
    const int q = warp & 3;
    const int cx = lane & 15, sh = lane >> 4;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + kTsColD;
    const uint32_t phase = (uint32_t)(cx & 7);   // swizzle phase of a buffer row = its cell column (row blocks are 16 rows)
    // byte offset of the four 16-byte chunks of sub-column sw inside a buffer row: logical chunk (sh ^ sw)*4 + j, swizzled
    uint32_t chunk_off[2][4];
#pragma unroll
    for (int sw = 0; sw < 2; ++sw)
#pragma unroll
      for (int j = 0; j < 4; ++j) chunk_off[sw][j] = (((uint32_t)((sh ^ sw) * 4 + j)) ^ phase) << 4;
    for (int g = 0; g < n_tiles; ++g) {
      const int li = g >> 2;
      const int b = g & 1;
      const int hf = (g >> 1) & 1;
      const int cyu = 4 * (g & 1) + q;   // cell row within the unit
      mbar_wait_relaxed(&d_full[b], (uint32_t)((g >> 1) & 1));
      tc_fence_after();
      uint32_t packed[2][16];
#pragma unroll
      for (int sw = 0; sw < 2; ++sw) {
        if (kTsKnock & 256) break;
        uint32_t d[32];
        tmem_ld_32x32(lane_base + b * 64 + sw * 32, d);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 16; ++j) packed[sw][j] = relu_pack_bf16x2(__uint_as_float(d[2 * j]), __uint_as_float(d[2 * j + 1]));
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&d_empty[b]);
      // unit buffer: AL0 (sw = 0, K order [sh=0 | sh=1]) and AL1 (sw = 1, K order [sh=1 | sh=0]); row block 0 is the halo
      mbar_wait_relaxed(&c1_empty[hf], (uint32_t)((li & 1) ^ 1));
      uint8_t* row = c1buf + hf * kStemUnitBytes + ((cyu + 1) * 16 + cx) * 128;
      if (!(kTsKnock & 32)) {
#pragma unroll
        for (int sw = 0; sw < 2; ++sw)
#pragma unroll
          for (int j = 0; j < 4; ++j)
            *reinterpret_cast<uint4*>(row + sw * kStemABuf + chunk_off[sw][j]) =
                make_uint4(packed[sw][4 * j], packed[sw][4 * j + 1], packed[sw][4 * j + 2], packed[sw][4 * j + 3]);
      }
      const bool halo = hf == 0 && cyu == 7;   // cell row 7 is also the halo row block of the frame's second unit
      if (halo) {
        mbar_wait_relaxed(&c1_empty[1], (uint32_t)((li & 1) ^ 1));
        uint8_t* hrow = c1buf + kStemUnitBytes + cx * 128;
#pragma unroll
        for (int sw = 0; sw < 2; ++sw)
#pragma unroll
          for (int j = 0; j < 4; ++j)
            *reinterpret_cast<uint4*>(hrow + sw * kStemABuf + chunk_off[sw][j]) =
                make_uint4(packed[sw][4 * j], packed[sw][4 * j + 1], packed[sw][4 * j + 2], packed[sw][4 * j + 3]);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&c1_full[hf]);
        if (halo) mbar_arrive(&c1_full[1]);
      }
    }
  } else {
    setmaxnreg_dec<56>();
    transposer_role((1 + warp - kTsXposeWarp1) * 32 + lane);
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
