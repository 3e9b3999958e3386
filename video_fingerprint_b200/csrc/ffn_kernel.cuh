// Fused feed-forward of a TemporalAttentionBlock (model.py:147-150): delta = W2 * GELU(W1 * xn + b1) + b2, with the
// 1024-wide hidden activation never leaving the SM, on CTA PAIRS (tcgen05 cta_group::2).
//
// As two GEMM launches the MLP moves 5 KB per token through HBM (xn in - four times, once per column tile -, h out; h in,
// delta out) and is bound by that: 3.3 ms per 10 000 x 64-frame clips for 2.7 TFLOP. Here a pair of CTAs owns 256 tokens
// (128 per CTA) and produces / consumes the hidden activation in four chunks of 256 columns:
//      GEMM1_c : D1 (256 TMEM columns)   = xn_tile * W1[256c .. 256c+256, :]^T                 16 UMMAs M256 N256 K16
//      act_c   : H (shared memory, bf16, K-major SWIZZLE_128B = the layout of an A operand) = GELU(D1 + b1)
//      GEMM2_c : D2 (256 TMEM columns)  += H * W2[:, 256c .. 256c+256]^T                        16 UMMAs M256 N256 K16
// so HBM sees 512 B in and 512 B out per token.
//
// Why pairs. An SS-mode UMMA streams BOTH operands from shared memory, (128 + N) rows x 32 B per instruction per SM: 96 B/clk
// at N = 256, 128 B/clk - the whole shared-memory port - at N = 128, and the weight stream of this kernel (1 MB per 128
// tokens) adds 64 B/clk of TMA fill. The first, single-CTA version of this kernel (N = 128 UMMAs, eight 128-column chunks)
// ran at 40 % tensor-pipe utilisation (ncu: the issuer never waited, the pipe itself was starved by the port) and was no
// faster than the two GEMMs. With cta_group::2 each SM keeps only HALF of every weight block (128 of its 256 rows) and
// reads the other half from its peer: 64 B/clk of operand reads + 32 B/clk of fill + 16 B/clk of hidden-chunk writes.
//
//   warp 0      TMA producer (both CTAs): own xn tile (4 K blocks) and own half of every weight block through a ring of
//               16 KB slots, in exactly the order the issuer consumes them; byte counts land on the LEADER's barriers
//   warp 1      TMEM allocation (512 columns: D1 256 | D2 256); in the leader CTA (cluster rank 0) also the UMMA issuer,
//               whose commits are multicast to both CTAs' barriers
//   warps 2-17  activation / output warps (both CTAs): TMEM lane quarter = warp % 4, column quarter = (warp - 2) / 4.
//               Sixteen of them: the activation phase is bound by the MUFU pipe (one tanh per element, 2 048 cycles per chunk)
//               and the FMA pipe (~2 300), with eight warps it took 4 000 cycles (cycle trace) and set the kernel's pace
// D1 and H are single buffers: the issuer's order G1(n+1), G2(n) puts a whole GEMM between a buffer's last read and its next
// write, which is when the activation warps drain D1 / refill H.
#pragma once
#include "epilogues.cuh"
#include "sm100_primitives.cuh"

namespace vfp {

constexpr int kFfnHidden = 1024;
constexpr int kFfnChunk = 256;
constexpr int kFfnChunks = kFfnHidden / kFfnChunk;
constexpr int kFfnActWarps = 16;                     // four per TMEM lane quarter: 64 hidden / 64 output columns each
constexpr int kFfnThreads = 64 + 32 * kFfnActWarps;

// development trace (-DVFP_FFN_TRACE): block 0 records (tag, clock) pairs of its producer, issuer and first activation warp
#ifdef VFP_FFN_TRACE
__device__ long long g_ffn_trace[8192];   // [role 0: issuer, role 1: activation warp 2][2048 slots][tag, clock]... two values per slot
__device__ unsigned int g_ffn_trace_n = 0;
// plain stores into a slot the calling thread counts itself: no atomics, nothing to wait for (an atomicAdd per point cost ~800 cycles)
#define FFN_TRACE_DECL(role) int trace_i = 0; const int trace_role = (role); (void)trace_i; (void)trace_role
#define FFN_TRACE(tag) do { if (blockIdx.x == 0 && trace_i < 1024) { g_ffn_trace[(trace_role * 1024 + trace_i) * 2] = (tag); g_ffn_trace[(trace_role * 1024 + trace_i) * 2 + 1] = clock64(); ++trace_i; } } while (0)
#else
#define FFN_TRACE_DECL(role)
#define FFN_TRACE(tag)
#endif

template <int SLOTS>
struct FfnSmem {
  static constexpr int kA0 = 0;                          // xn tile: 4 K blocks of 128 rows x 128 B
  static constexpr int kRing = kA0 + 4 * 16384;          // weight blocks: this CTA's 128 rows x 128 B each
  static constexpr int kH = kRing + SLOTS * 16384;       // hidden chunk: 4 K blocks of 128 rows x 128 B
  static constexpr int kBias = kH + 4 * 16384;           // b1 (1024 floats) | b2 (256 floats): see below
  static constexpr int kBars = kBias + 5 * 1024;
  static constexpr int kTotal = kBars + 512 + 1024;
};

struct FfnParams {
  alignas(64) CUtensorMap tmap_x;    // xn [M][256] bf16, box 128 rows x 64 cols, SWIZZLE_128B
  alignas(64) CUtensorMap tmap_w1;   // W1 [1024][256] bf16 K-major, box 128 rows x 64 cols
  alignas(64) CUtensorMap tmap_w2;   // W2 [256][1024] bf16 K-major, box 128 rows x 64 cols
  alignas(64) CUtensorMap tmap_out;  // delta [M][256] bf16, box 32 x 32, SWIZZLE_64B
  const float* b1;                   // [1024]
  const float* b2;                   // [256]
  int M;
  int pair_tiles;                    // ceil(M / 256)
};

template <int SLOTS>
__global__ void __launch_bounds__(kFfnThreads, 1) ffn_pair_kernel(const __grid_constant__ FfnParams p) {
  using L = FfnSmem<SLOTS>;
  static_assert(L::kTotal <= 232448, "ffn kernel shared memory");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* a0 = smem + L::kA0;
  uint8_t* ring = smem + L::kRing;
  uint8_t* hbuf = smem + L::kH;
  // The biases live in shared memory: with ~225 KB of the SM's 228 KB carved out as shared memory there is no L1 left, so every
  // __ldg of a bias vector is an L2 round trip (300+ cycles) in the middle of the activation phase.
  float* sbias = reinterpret_cast<float*>(smem + L::kBias);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::kBars);
  uint64_t* full = bars;                    // [SLOTS] leader's: bytes of both CTAs
  uint64_t* empty = bars + SLOTS;           // [SLOTS] per CTA (multicast commit)
  uint64_t* a0_full = bars + 2 * SLOTS;     // leader's
  uint64_t* a0_empty = a0_full + 1;         // per CTA: GEMM1 of the tile's last chunk has read the xn tile
  uint64_t* d1_full = a0_full + 2;          // per CTA
  uint64_t* d1_empty = a0_full + 3;         // leader's, 16 arrivals: both CTAs' activation warps have drained D1
  uint64_t* h_full = a0_full + 4;           // leader's, 16 arrivals: both CTAs' hidden chunks are written
  uint64_t* h_empty = a0_full + 5;          // per CTA: GEMM2 has read the hidden chunk
  uint64_t* d2_full = a0_full + 6;          // per CTA
  uint64_t* d2_empty = a0_full + 7;         // leader's, 16 arrivals
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a0_full + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const bool leader = crank == 0;
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int my_tiles = p.pair_tiles > pair ? (p.pair_tiles - pair + n_pairs - 1) / n_pairs : 0;
  const int n_chunks = my_tiles * kFfnChunks;   // global chunk sequence of this pair

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmap_x);
    tma_prefetch_desc(&p.tmap_w1);
    tma_prefetch_desc(&p.tmap_w2);
    tma_prefetch_desc(&p.tmap_out);
    for (int i = 0; i < SLOTS; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(a0_full, 1);
    mbar_init(a0_empty, 1);
    mbar_init(d1_full, 1);
    mbar_init(d1_empty, 2 * kFfnActWarps);
    mbar_init(h_full, 2 * kFfnActWarps);
    mbar_init(h_empty, 1);
    mbar_init(d2_full, 1);
    mbar_init(d2_empty, 2 * kFfnActWarps);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc_2cta(tmem_slot, 512);
    tmem_relinquish_2cta();
  }
  // b1 as f16x2 pairs (the activation adds it after converting the accumulator to f16x2), b2 as fp32
  uint32_t* sbias_h = reinterpret_cast<uint32_t*>(sbias);
  for (int i = threadIdx.x; i < kFfnHidden / 2; i += kFfnThreads) {
    const __half2 h = __floats2half2_rn(__ldg(p.b1 + 2 * i), __ldg(p.b1 + 2 * i + 1));
    sbias_h[i] = *reinterpret_cast<const uint32_t*>(&h);
  }
  for (int i = threadIdx.x; i < 256; i += kFfnThreads) sbias[kFfnHidden + i] = __ldg(p.b2 + i);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------ TMA producer (both CTAs) ------------------------------
    if (lane == 0) {
      int slot = 0;
      uint32_t ph = 0, a_ph = 0;
      const uint32_t a0_full_leader = mapa_u32(a0_full, 0);
      auto load_w = [&](const CUtensorMap* map, int k_col, int row0) {
        mbar_wait(&empty[slot], ph ^ 1);
        if (leader) mbar_arrive_expect_tx(&full[slot], 2 * 16384);
        tma_load_2d_2cta(map, mapa_u32(&full[slot], 0), ring + slot * 16384, k_col, row0 + (int)crank * 128);
        if (++slot == SLOTS) { slot = 0; ph ^= 1; }
      };
      auto load_g1 = [&](int n) {   // operands of GEMM1 of global chunk n: the xn tile at a tile's first chunk, W1 rows 256c ..
        const int c = n % kFfnChunks;
        if (c == 0) {
          const int tile = pair + (n / kFfnChunks) * n_pairs;
          mbar_wait(a0_empty, a_ph ^ 1);
          a_ph ^= 1;
          if (leader) mbar_arrive_expect_tx(a0_full, 2 * 4 * 16384);
          for (int kb = 0; kb < 4; ++kb) tma_load_2d_2cta(&p.tmap_x, a0_full_leader, a0 + kb * 16384, kb * 64, (tile * 2 + (int)crank) * 128);
        }
        for (int kb = 0; kb < 4; ++kb) load_w(&p.tmap_w1, kb * 64, c * kFfnChunk);
      };
      auto load_g2 = [&](int n) {   // W2: all 256 output rows (128 per CTA), K columns 256c + 64kb
        const int c = n % kFfnChunks;
        for (int kb = 0; kb < 4; ++kb) load_w(&p.tmap_w2, c * kFfnChunk + kb * 64, 0);
      };
      if (n_chunks > 0) load_g1(0);
      for (int n = 0; n < n_chunks; ++n) {
        if (n + 1 < n_chunks) load_g1(n + 1);
        load_g2(n);
      }
    }
  } else if (warp == 1) {
    // ------------------------------ UMMA issuer (leader CTA only) ------------------------------
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = umma_idesc_bf16(256, 256);
      FFN_TRACE_DECL(0);
      int slot = 0;
      uint32_t ph = 0, a_ph = 0, d1e_ph = 0, hf_ph = 0, d2e_ph = 0;
      const uint32_t a0_addr = smem_u32(a0), h_addr = smem_u32(hbuf);
      auto commit_slot = [&]() {
        umma_commit_2cta(&empty[slot], 3);
        if (++slot == SLOTS) { slot = 0; ph ^= 1; }
      };
      auto gemm1 = [&](int n) {
        const int c = n % kFfnChunks;
        if (c == 0) {
          mbar_wait(a0_full, a_ph);
          a_ph ^= 1;
        }
        FFN_TRACE(100);
        mbar_wait(d1_empty, d1e_ph ^ 1);   // both CTAs' activation warps hold the previous chunk in registers
        d1e_ph ^= 1;
        tc_fence_after();
        FFN_TRACE(101);
        for (int kb = 0; kb < 4; ++kb) {
          mbar_wait(&full[slot], ph);
          tc_fence_after();
          const uint64_t adesc = umma_smem_desc_kmajor<128>(a0_addr + kb * 16384);
          const uint64_t bdesc = umma_smem_desc_kmajor<128>(smem_u32(ring + slot * 16384));
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16_2cta(tmem_base, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          commit_slot();
        }
        umma_commit_2cta(d1_full, 3);
        FFN_TRACE(102);
        if (c == kFfnChunks - 1) umma_commit_2cta(a0_empty, 3);   // last GEMM1 of the tile: the xn tiles may be replaced
      };
      auto gemm2 = [&](int n) {
        const int c = n % kFfnChunks;
        if (c == 0) {   // the output warps of both CTAs have drained D2 of the previous tile
          mbar_wait(d2_empty, d2e_ph ^ 1);
          d2e_ph ^= 1;
        }
        FFN_TRACE(110);
        mbar_wait(h_full, hf_ph);
        hf_ph ^= 1;
        tc_fence_after();
        FFN_TRACE(111);
        for (int kb = 0; kb < 4; ++kb) {
          mbar_wait(&full[slot], ph);
          tc_fence_after();
          const uint64_t adesc = umma_smem_desc_kmajor<128>(h_addr + kb * 16384);
          const uint64_t bdesc = umma_smem_desc_kmajor<128>(smem_u32(ring + slot * 16384));
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16_2cta(tmem_base + 256, adesc + 2 * k, bdesc + 2 * k, idesc, (c | kb | k) != 0 ? 1u : 0u);
          commit_slot();
        }
        umma_commit_2cta(h_empty, 3);
        FFN_TRACE(112);
        if (c == kFfnChunks - 1) umma_commit_2cta(d2_full, 3);
      };
      if (n_chunks > 0) gemm1(0);
      for (int n = 0; n < n_chunks; ++n) {
        if (n + 1 < n_chunks) gemm1(n + 1);
        gemm2(n);
      }
    }
  } else {
    // ------------------------------ activation + output warps (both CTAs) ------------------------------
    const int q = warp & 3;                 // TMEM lane quarter
    const int cq = (warp - 2) >> 2;         // column quarter: hidden columns 64 cq .. of the chunk / output columns 64 cq ..
    const int row = q * 32 + lane;          // token row inside this CTA's tile
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    uint32_t d1f_ph = 0, he_ph = 0, d2f_ph = 0;
    FFN_TRACE_DECL(1);
    const uint32_t d1_empty_leader = mapa_u32(d1_empty, 0), h_full_leader = mapa_u32(h_full, 0), d2_empty_leader = mapa_u32(d2_empty, 0);
    // hidden chunk layout (A operand of GEMM2): K block = 64 hidden columns = one 128-byte row per token, 16-byte pieces
    // XOR-swizzled with the row index (SWIZZLE_128B); this warp's 64 columns are K block cq
    uint8_t* h_row = hbuf + cq * 16384 + row * 128;
    const uint32_t sw = (uint32_t)(row & 7);
    // output staging: once GEMM2 of a tile's last chunk has completed the hidden buffer is free; every warp stages its
    // 32 rows x 64 columns there (two 2 KB chunks of 32 x 32 bf16, SWIZZLE_64B) and hands them to the TMA unit
    uint8_t* stage = hbuf + (warp - 2) * 4096;

    auto output_tile = [&](int tile) {   // delta = D2 + b2 -> bf16 -> staging -> TMA store
      mbar_wait(d2_full, d2f_ph);
      d2f_ph ^= 1;
      tc_fence_after();
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t v[32];
        tmem_ld_32x32(lane_addr + 256 + cq * 64 + c * 32, v);
        tmem_ld_wait();
        const float* bias = sbias + kFfnHidden + cq * 64 + c * 32;
        uint8_t* r0 = stage + c * 2048 + lane * 64;
        const int s64 = (lane >> 1) & 3;
#pragma unroll
        for (int piece = 0; piece < 4; ++piece) {
          const float4 ba = *reinterpret_cast<const float4*>(bias + 8 * piece);
          const float4 bc = *reinterpret_cast<const float4*>(bias + 8 * piece + 4);
          uint4 o;
          o.x = pack_bf16x2(__uint_as_float(v[8 * piece + 0]) + ba.x, __uint_as_float(v[8 * piece + 1]) + ba.y);
          o.y = pack_bf16x2(__uint_as_float(v[8 * piece + 2]) + ba.z, __uint_as_float(v[8 * piece + 3]) + ba.w);
          o.z = pack_bf16x2(__uint_as_float(v[8 * piece + 4]) + bc.x, __uint_as_float(v[8 * piece + 5]) + bc.y);
          o.w = pack_bf16x2(__uint_as_float(v[8 * piece + 6]) + bc.z, __uint_as_float(v[8 * piece + 7]) + bc.w);
          *reinterpret_cast<uint4*>(r0 + ((piece ^ s64) << 4)) = o;
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(d2_empty_leader);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        const int grow0 = (tile * 2 + (int)crank) * 128 + q * 32;
        tma_store_2d(&p.tmap_out, stage, cq * 64, grow0);          // rows past M are clipped by the tensor map
        tma_store_2d(&p.tmap_out, stage + 2048, cq * 64 + 32, grow0);
        tma_store_commit();
        tma_store_wait_read<0>();   // the staging bytes are about to be overwritten by the next hidden chunk
      }
      // every warp's stores must have been read before ANY warp writes the hidden buffer again
      asm volatile("bar.sync 1, %0;" ::"n"(32 * kFfnActWarps) : "memory");
    };

    for (int n = 0; n < n_chunks; ++n) {
      const int c = n % kFfnChunks;
      if (warp == 2 && lane == 0) FFN_TRACE(200);
      mbar_wait(d1_full, d1f_ph);
      d1f_ph ^= 1;
      tc_fence_after();
      if (warp == 2 && lane == 0) FFN_TRACE(201);
      uint32_t packed[32];
      {
        uint32_t va[32], vb[32];
        tmem_ld_32x32(lane_addr + cq * 64, va);
        tmem_ld_32x32(lane_addr + cq * 64 + 32, vb);
        tmem_ld_wait();
        if (warp == 2 && lane == 0) FFN_TRACE(203);
        tc_fence_before();   // D1 is in registers: GEMM1 of the next chunk may overwrite it
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(d1_empty_leader);
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          uint32_t(&v)[32] = cc ? vb : va;
          const uint32_t* bias = sbias_h + (c * kFfnChunk + cq * 64 + cc * 32) / 2;
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            const uint4 bb = *reinterpret_cast<const uint4*>(bias + i / 2);
            packed[cc * 16 + i / 2] = gelu_bias_bf16x2(make_float2(__uint_as_float(v[i]), __uint_as_float(v[i + 1])), bb.x);
            packed[cc * 16 + i / 2 + 1] = gelu_bias_bf16x2(make_float2(__uint_as_float(v[i + 2]), __uint_as_float(v[i + 3])), bb.y);
            packed[cc * 16 + i / 2 + 2] = gelu_bias_bf16x2(make_float2(__uint_as_float(v[i + 4]), __uint_as_float(v[i + 5])), bb.z);
            packed[cc * 16 + i / 2 + 3] = gelu_bias_bf16x2(make_float2(__uint_as_float(v[i + 6]), __uint_as_float(v[i + 7])), bb.w);
          }
        }
      }
      // the previous tile's output goes out between the activation's register phase and its shared-memory phase: its
      // accumulator completes (GEMM2 of the last chunk) while the registers above are being filled
      if (warp == 2 && lane == 0) FFN_TRACE(204);
      if (c == 0 && n > 0) output_tile(pair + (n / kFfnChunks - 1) * n_pairs);
      if (warp == 2 && lane == 0) FFN_TRACE(205);
      mbar_wait(h_empty, he_ph ^ 1);   // GEMM2 of the previous chunk has read the hidden buffer
      he_ph ^= 1;
      if (warp == 2 && lane == 0) FFN_TRACE(206);
#pragma unroll
      for (int piece = 0; piece < 8; ++piece)
        *reinterpret_cast<uint4*>(h_row + ((piece ^ sw) << 4)) =
            make_uint4(packed[4 * piece], packed[4 * piece + 1], packed[4 * piece + 2], packed[4 * piece + 3]);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(h_full_leader);
      if (warp == 2 && lane == 0) FFN_TRACE(207);
    }
    if (n_chunks > 0) output_tile(pair + (my_tiles - 1) * n_pairs);
    if (lane == 0) tma_store_wait_read<0>();
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
