// Multi-head self-attention (model.py:143) over PACKED clips on the 5th-generation tensor cores: QK^T as SS-mode UMMAs into
// tensor memory, softmax by one thread per score row straight out of TMEM (no shuffles: a thread owns its whole row), P written
// back to TMEM as bf16 and used from there as the A operand of the PV UMMA (TS mode), V taken MN-major from the very tile the
// TMA unit delivered (no transposed copy).
//
// head_dim is 32 and a clip of the benchmark has 64 tokens, so one (clip, head) problem is 64 x 64 x 32 - half a UMMA tile in
// M. Two heads share a tile: a UNIT is (64 query tokens of one clip, a PAIR of heads). The TMA box is 64 tokens x the pair's
// 64 columns of Q, K or V (128-byte rows, SWIZZLE_128B). The Q box is loaded twice, back to back, so the A operand has 128
// rows = the same 64 queries twice; the first K step pair (columns 0-31 = head 2hp) accumulates into TMEM columns 0-63 and the
// second (columns 32-63 = head 2hp+1) into columns 64-127, so accumulator rows 0-63 read "their" scores from the first half
// and rows 64-127 from the second: every one of the 128 softmax threads has a full score row of ONE head. P (128 rows x 64
// keys) times the V box (64 keys x 64 columns, both heads side by side) gives a 128 x 64 block of which rows 0-63 keep columns
// 0-31 and rows 64-127 columns 32-63. Half of each product is thrown away; the tensor pipe has the room (the stage is 0.7 % of
// the forward's FLOPs), the point is that nothing but TMA, UMMA and TMEM loads touch the operands.
//
// Keys are walked in blocks of 64 from the clip's first token (online softmax, raw-score maxima, scale folded into the exp2
// argument; the running output is rescaled in registers, 32 floats per thread, so TMEM holds no state between key blocks);
// only a clip's last key block needs a mask, and what a clip gets never depends on what it is packed next to - bit for bit.
//
//   warp 0      TMA producer: per step Q box (twice) + K box + V box = 32 KB into a 3-stage ring
//   warp 1      TMEM allocation (256 columns: S 128 | P 2 x 32 | O 64) + UMMA issuer; S of the next step is issued as soon as the
//               softmax threads have pulled the current S into registers, i.e. it overlaps their exponentials
//   warps 2-5   softmax / output: TMEM lane quarter = warp % 4. They run one step ahead of the PV products: P of step t is
//               written before the product of step t - 1 is collected, so the PV UMMAs and both hand-offs hide behind the
//               exponentials (P is double buffered for that)
// Two CTAs per SM (2 x 256 TMEM columns, 2 x 97 KB of shared memory) cover each other's TMEM and mbarrier round trips.
#pragma once
#include "stem_ts_kernel.cuh"
#include "token_kernels.cuh"

namespace vfp {

constexpr int kAtcThreads = 192;
constexpr int kAtcStages = 3;
constexpr int kAtcStageBytes = 32768;                          // Q twice 16 KB | K 8 KB | V 8 KB
constexpr int kAtcColS = 0, kAtcColP = 128, kAtcColO = 192;    // TMEM column map: S 128 | P 2 x 32 | O 64
constexpr int kAtcTmemCols = 256;
constexpr int kAtcSmemBytes = kAtcStages * kAtcStageBytes + 256 + 1024;

struct AttnTcParams {
  alignas(64) CUtensorMap tmap_qkv;   // [tokens][768] bf16 = [Q | K | V], box 64 columns x 64 tokens, SWIZZLE_128B
  const int4* items;                  // {first query token, clip start, clip end, 0} per 64 query tokens of one clip
  __nv_bfloat16* out;                 // [tokens][256] bf16
  int n_units;                        // 4 head pairs per item
};

__global__ void __launch_bounds__(kAtcThreads, 2) attention_tc_kernel(const __grid_constant__ AttnTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* ring = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kAtcStages * kAtcStageBytes);
  uint64_t* full = bars;                    // [stages] TMA -> issuer
  uint64_t* empty = bars + kAtcStages;      // [stages] PV UMMAs done -> producer
  uint64_t* s_full = bars + 2 * kAtcStages; // scores in TMEM
  uint64_t* s_empty = s_full + 1;           // scores in registers (4 warps)
  uint64_t* p_full = s_full + 2;            // P in TMEM (4 warps)
  uint64_t* o_full = s_full + 3;            // PV product in TMEM
  uint64_t* o_empty = s_full + 4;           // PV product in registers (4 warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s_full + 5);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmap_qkv);
    for (int i = 0; i < kAtcStages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(s_empty, 4);
    mbar_init(p_full, 4);
    mbar_init(o_full, 1);
    mbar_init(o_empty, 4);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, kAtcTmemCols);
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
      uint32_t ph = 0;
      for (int u = blockIdx.x; u < p.n_units; u += gridDim.x) {
        const int4 it = __ldg(p.items + (u >> 2));
        const int col = (u & 3) * 64;
        const int n_kb = (it.z - it.y + 63) >> 6;
        for (int kb = 0; kb < n_kb; ++kb) {
          mbar_wait(&empty[stage], ph ^ 1);
          mbar_arrive_expect_tx(&full[stage], kAtcStageBytes);
          uint8_t* dst = ring + stage * kAtcStageBytes;
          tma_load_2d(&p.tmap_qkv, &full[stage], dst, col, it.x);
          tma_load_2d(&p.tmap_qkv, &full[stage], dst + 8192, col, it.x);
          tma_load_2d(&p.tmap_qkv, &full[stage], dst + 16384, 256 + col, it.y + kb * 64);
          tma_load_2d(&p.tmap_qkv, &full[stage], dst + 24576, 512 + col, it.y + kb * 64);
          if (++stage == kAtcStages) { stage = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ UMMA issuer ------------------------------
    if (lane == 0) {
      constexpr uint32_t idesc_s = umma_idesc_bf16(128, 64);
      constexpr uint32_t idesc_pv = umma_idesc_bf16(128, 64) | (1u << 16);   // B (= V) is MN-major: [key][column]
      const uint32_t ring_lo = desc_lo_sw128(smem_u32(ring));
      // scores of one step: two heads x two K steps of 16 columns, M128 N64
      auto issue_s = [&](int stage) {
        const uint32_t a_lo = ring_lo + ((stage * kAtcStageBytes) >> 4), b_lo = a_lo + (16384 >> 4);
        umma_ss_lo<false>(tmem_base + kAtcColS, a_lo, b_lo, idesc_s);
        umma_ss_lo<true>(tmem_base + kAtcColS, a_lo + 2, b_lo + 2, idesc_s);
        umma_ss_lo<false>(tmem_base + kAtcColS + 64, a_lo + 4, b_lo + 4, idesc_s);
        umma_ss_lo<true>(tmem_base + kAtcColS + 64, a_lo + 6, b_lo + 6, idesc_s);
      };
      // P (TMEM, 8 columns per 16 keys) x V (16 keys = 2 KB per K step)
      auto issue_pv = [&](int stage, uint32_t t) {
        const uint32_t v_lo = ring_lo + ((stage * kAtcStageBytes + 24576) >> 4);
        const uint32_t p_col = tmem_base + kAtcColP + (t & 1) * 32;
        umma_ts_lo<false>(tmem_base + kAtcColO, p_col, v_lo, idesc_pv);
#pragma unroll
        for (int k = 1; k < 4; ++k) umma_ts_lo<true>(tmem_base + kAtcColO, p_col + 8 * k, v_lo + 128 * k, idesc_pv);
      };
      // the steps of this CTA, flattened: (unit, key block)
      int u = blockIdx.x, kb = 0, n_kb = 0;
      auto load_unit = [&]() {
        const int4 it = __ldg(p.items + (u >> 2));
        n_kb = (it.z - it.y + 63) >> 6;
      };
      if (u < p.n_units) {
        load_unit();
        int s_stage = 0, pv_stage = 0;
        uint32_t s_ph = 0;
        uint32_t t = 0;
        mbar_wait(&full[0], 0);
        tc_fence_after();
        issue_s(0);
        umma_commit(s_full);
        if (++s_stage == kAtcStages) { s_stage = 0; s_ph ^= 1; }
        for (;;) {
          // is there a step t + 1?
          bool more = true;
          if (++kb == n_kb) {
            kb = 0;
            u += gridDim.x;
            if (u < p.n_units) load_unit(); else more = false;
          }
          if (more) {
            mbar_wait(&full[s_stage], s_ph);
            mbar_wait(s_empty, t & 1);           // the softmax threads hold step t's scores in registers
            tc_fence_after();
            issue_s(s_stage);
            umma_commit(s_full);
            if (++s_stage == kAtcStages) { s_stage = 0; s_ph ^= 1; }
          }
          mbar_wait(p_full, t & 1);
          if (t > 0) mbar_wait(o_empty, (t - 1) & 1);
          tc_fence_after();
          issue_pv(pv_stage, t);
          umma_commit(o_full);
          umma_commit(&empty[pv_stage]);
          if (++pv_stage == kAtcStages) pv_stage = 0;
          ++t;
          if (!more) break;
        }
      }
    }
  } else {
    // ------------------------------ softmax + output: one thread per score row ------------------------------
    // Software-pipelined by one step: the thread writes P of step t, and only then collects the PV product of step t - 1 (whose
    // UMMAs ran while it was busy with the exponentials of step t), so it never waits for the tensor pipe or its hand-offs.
    const int q = warp & 3;
    const int r = q * 32 + lane;            // accumulator row
    const int hsel = r >> 6;                // rows 0-63: first head of the pair, 64-127: second
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t s_addr = lane_base + kAtcColS + hsel * 64, p_addr = lane_base + kAtcColP, o_addr = lane_base + kAtcColO + hsel * 32;
    const float sl2 = 0.17677669529663687f * 1.4426950408889634f;   // 1/sqrt(32) * log2(e)
    float acc[32];                          // running output of the unit whose PV products are being collected
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = 0.0f;
    // the step whose PV product is still to be collected
    bool pend = false, pend_last = false;
    float pend_alpha = 0.0f, pend_inv = 0.0f;
    __nv_bfloat16* pend_dst = nullptr;      // nullptr: a query row past the end of its clip
    auto collect = [&](uint32_t tp) {
      mbar_wait(o_full, tp & 1);
      tc_fence_after();
      uint32_t o[32];
      tmem_ld_32x32(o_addr, o);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(o_empty);
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[i] = fmaf(acc[i], pend_alpha, __uint_as_float(o[i]));   // first key block: alpha = 0
      if (pend_last && pend_dst != nullptr) {
        const float inv = pend_inv;
        uint4* dst = reinterpret_cast<uint4*>(pend_dst);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          dst[i] = make_uint4(pack_bf16x2(acc[8 * i] * inv, acc[8 * i + 1] * inv), pack_bf16x2(acc[8 * i + 2] * inv, acc[8 * i + 3] * inv),
                              pack_bf16x2(acc[8 * i + 4] * inv, acc[8 * i + 5] * inv), pack_bf16x2(acc[8 * i + 6] * inv, acc[8 * i + 7] * inv));
      }
    };
    uint32_t t = 0;
    for (int u = blockIdx.x; u < p.n_units; u += gridDim.x) {
      const int4 it = __ldg(p.items + (u >> 2));
      const int head = (u & 3) * 2 + hsel;
      const int len = it.z - it.y;
      const int n_kb = (len + 63) >> 6;
      const int token = it.x + (r & 63);
      float m = -INFINITY, l = 0.0f;
      for (int kb = 0; kb < n_kb; ++kb, ++t) {
        mbar_wait(s_full, t & 1);
        tc_fence_after();
        uint32_t s0[32], s1[32];
        tmem_ld_32x32(s_addr, s0);
        tmem_ld_32x32(s_addr + 32, s1);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(s_empty);
        const int valid = len - kb * 64;
        if (valid < 64) {   // the clip's last key block: rows past its end belong to the next clip (or are TMA zero fill)
#pragma unroll
          for (int c = 0; c < 32; ++c) {
            if (c >= valid) s0[c] = 0xff800000u;
            if (c + 32 >= valid) s1[c] = 0xff800000u;
          }
        }
        float mx = __uint_as_float(s0[0]);
#pragma unroll
        for (int c = 1; c < 32; ++c) mx = fmaxf(mx, __uint_as_float(s0[c]));
#pragma unroll
        for (int c = 0; c < 32; ++c) mx = fmaxf(mx, __uint_as_float(s1[c]));
        const float m_new = fmaxf(m, mx);
        const float alpha = fast_exp2((m - m_new) * sl2);   // 0 in a unit's first key block (m = -inf)
        const float msl = m_new * sl2;
        m = m_new;
        float sum = 0.0f;
        uint32_t pk[32];
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          const float a = fast_exp2(fmaf(__uint_as_float(s0[2 * c]), sl2, -msl));
          const float b = fast_exp2(fmaf(__uint_as_float(s0[2 * c + 1]), sl2, -msl));
          sum += a + b;
          pk[c] = pack_bf16x2(a, b);
        }
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          const float a = fast_exp2(fmaf(__uint_as_float(s1[2 * c]), sl2, -msl));
          const float b = fast_exp2(fmaf(__uint_as_float(s1[2 * c + 1]), sl2, -msl));
          sum += a + b;
          pk[16 + c] = pack_bf16x2(a, b);
        }
        l = l * alpha + sum;
        tmem_st_32x32(p_addr + (t & 1) * 32, pk);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full);
        if (pend) collect(t - 1);
        pend = true;
        pend_alpha = alpha;
        pend_last = kb == n_kb - 1;
        pend_inv = 1.0f / l;
        pend_dst = token < it.z ? p.out + (size_t)token * kDim + head * 32 : nullptr;
      }
    }
    if (pend) collect(t - 1);
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kAtcTmemCols);
  }
}

}  // namespace vfp
