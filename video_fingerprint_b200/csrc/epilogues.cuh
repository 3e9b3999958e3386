// Epilogue functors for gemm_tcgen05_kernel. Each epilogue thread owns ONE accumulator row of the
// 128-row tile and receives it in chunks of 32 consecutive fp32 columns straight from TMEM.
#pragma once
#include "sm100_primitives.cuh"

namespace vfp {

// GELU of the MLP up-projection (nn.GELU() default = erf form, model.py:136). The epilogue evaluates 2.6e9 of these per
// 10k clips and is issue-bound on them (the erf form costs ~18 instructions and two MUFU ops per value), so the
// value is computed as 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3))) with the hardware tanh (one MUFU op, six
// instructions). |difference to the erf form| <= 4.8e-4 (+ 2^-11 relative from tanh.approx), below the bf16 rounding
// the stored activation gets anyway for |x| > 0.1; measured end to end on the fp32 oracle the embeddings move by
// 1 - cos = 2e-9 (tests/test_oracle.py::test_tanh_gelu_is_harmless).
__device__ __forceinline__ float gelu_erf(float x) {
  const float u = x * fmaf(x * x, 0.0356774081f, 0.7978845608f);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  const float hx = 0.5f * x;
  return fmaf(hx, t, hx);
}

// Two values at once, in half precision. The MLP evaluates 2.6e9 GELUs per 10 000 clips; in fp32 (even as packed FMUL2 / FFMA2)
// that is ~12 FMA-pipe cycles per element and warp, which made the activation phase - not the tensor pipe - the pace of the
// fused feed-forward kernel (cycle trace: 4 800 cycles of GELU per 128 x 256 chunk against 4 096 cycles of UMMAs). The result
// is stored as bf16 (8 mantissa bits), so the polynomial, the tanh and the blend run as fp16x2 instructions (11 bits, one
// instruction per PAIR): x -> f16x2, u = x (c0 + c1 x^2), t = tanh.approx.f16x2(u), y = 0.5 x t + 0.5 x. Large |x| overflow x^2
// to inf, which tanh maps to +-1 - the right limit. |fp16 form - fp32 form| < 2^-10 |y| + 2^-11 |x|, below the bf16 rounding of
// the stored value.
__device__ __forceinline__ uint32_t gelu_erf2_f16(float2 x) {
  uint32_t xh, y;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(xh) : "f"(x.y), "f"(x.x));
  asm("{\n\t"
      ".reg .b32 x2, p, u, t, hx;\n\t"
      "mul.rn.f16x2 x2, %1, %1;\n\t"
      "fma.rn.f16x2 p, x2, %2, %3;\n\t"
      "mul.rn.f16x2 u, %1, p;\n\t"
      "tanh.approx.f16x2 t, u;\n\t"
      "mul.rn.f16x2 hx, %1, %4;\n\t"
      "fma.rn.f16x2 %0, hx, t, hx;\n\t"
      "}"
      : "=r"(y)
      : "r"(xh), "r"(0x28912891u) /* 0.0356774 */, "r"(0x3A623A62u) /* 0.7978846 */, "r"(0x38003800u) /* 0.5 */);
  return y;
}
// accumulator pair + bias pair (already f16x2) -> GELU -> bf16x2: the bias joins after the conversion to f16x2 (the packed fp32
// add it replaces, FADD2, costs about four times an HADD2 in issue slots: ncu source page of the fused MLP kernel)
__device__ __forceinline__ uint32_t gelu_bias_bf16x2(float2 acc, uint32_t bias_h2) {
  uint32_t xh, y;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(xh) : "f"(acc.y), "f"(acc.x));
  asm("{\n\t"
      ".reg .b32 x, x2, p, u, t, hx;\n\t"
      "add.rn.f16x2 x, %1, %5;\n\t"
      "mul.rn.f16x2 x2, x, x;\n\t"
      "fma.rn.f16x2 p, x2, %2, %3;\n\t"
      "mul.rn.f16x2 u, x, p;\n\t"
      "tanh.approx.f16x2 t, u;\n\t"
      "mul.rn.f16x2 hx, x, %4;\n\t"
      "fma.rn.f16x2 %0, hx, t, hx;\n\t"
      "}"
      : "=r"(y)
      : "r"(xh), "r"(0x28912891u) /* 0.0356774 */, "r"(0x3A623A62u) /* 0.7978846 */, "r"(0x38003800u) /* 0.5 */, "r"(bias_h2));
  float lo, hi;
  asm("{\n\t.reg .b16 l, h;\n\tmov.b32 {l, h}, %2;\n\tcvt.f32.f16 %0, l;\n\tcvt.f32.f16 %1, h;\n\t}" : "=f"(lo), "=f"(hi) : "r"(y));
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// fp32 pair in, fp32 pair out (callers that keep working in fp32)
__device__ __forceinline__ float2 gelu_erf2(float2 x) {
  const uint32_t y = gelu_erf2_f16(x);
  float2 r;
  asm("{\n\t.reg .b16 lo, hi;\n\tmov.b32 {lo, hi}, %2;\n\tcvt.f32.f16 %0, lo;\n\tcvt.f32.f16 %1, hi;\n\t}" : "=f"(r.x), "=f"(r.y) : "r"(y));
  return r;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}

// Defaults shared by the epilogues: one sweep over the accumulator, no state across tiles, no extra smem.
struct EpiDefaults {
  static constexpr int kPasses = 1;
  static constexpr int kColumnSplit = 2;
  static constexpr int kExtraSmemBytes = 0;
  int block_n_ = 0;   // column tile width of the kernel that runs this epilogue (set once by the kernel)
  __device__ __forceinline__ void set_block_n(int n) { block_n_ = n; }
  template <class P> __device__ __forceinline__ void setup(const P&, uint8_t*, int, int) {}
  template <class P> __device__ __forceinline__ void finish(const P&, int) {}
  template <class P> __device__ __forceinline__ void item_begin(const P&, int, int, int, uint8_t*) {}
  template <class P> __device__ __forceinline__ void item_end(const P&, int, int, int, uint8_t*) {}
};

// -------------------------------------------------------------------------------------------
// y = act(acc + bias [+ pe[pos[row]]]) [+ residual]  -> fp32 and/or bf16 row-major outputs
// -------------------------------------------------------------------------------------------
struct EpiBiasAct : EpiDefaults {
  struct Params {
    const float* bias;       // [N] or null
    const float* residual;   // [M][ld_res] fp32 or null (added after the activation)
    const float* pe;         // [max_len][N] positional table or null
    const int* token_pos;    // [M] position of each row inside its clip (with pe)
    float* out_f32;          // [M][ld_out] or null
    __nv_bfloat16* out_bf16; // [M][ld_out] or null
    int ld_res, ld_out;
    int M, N;
    int act;  // 0 none, 1 relu, 2 gelu(erf)
  };
  __device__ __forceinline__ void begin(const Params&, int, int, int) {}
  __device__ __forceinline__ void end(const Params&, int, int, int) {}
  __device__ __forceinline__ void chunk(const Params& p, int mt, int col0, int row, uint32_t (&v)[32], int /*pass*/) {
    const long long grow = (long long)mt * kBlockMRows + row;
    if (grow >= p.M || col0 >= p.N) return;
    float x[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) x[i] = __uint_as_float(v[i]);
    if (p.bias) {
#pragma unroll
      for (int i = 0; i < 32; i += 4) {
        const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + i));
        x[i] += b.x; x[i + 1] += b.y; x[i + 2] += b.z; x[i + 3] += b.w;
      }
    }
    if (p.pe) {
      const float* pr = p.pe + (long long)p.token_pos[grow] * p.N + col0;
#pragma unroll
      for (int i = 0; i < 32; i += 4) {
        const float4 b = __ldg(reinterpret_cast<const float4*>(pr + i));
        x[i] += b.x; x[i + 1] += b.y; x[i + 2] += b.z; x[i + 3] += b.w;
      }
    }
    if (p.act == 1) {
#pragma unroll
      for (int i = 0; i < 32; ++i) x[i] = fmaxf(x[i], 0.0f);
    } else if (p.act == 2) {
#pragma unroll
      for (int i = 0; i < 32; ++i) x[i] = gelu_erf(x[i]);
    }
    if (p.residual) {
      const float* rr = p.residual + grow * p.ld_res + col0;
#pragma unroll
      for (int i = 0; i < 32; i += 4) {
        const float4 b = *reinterpret_cast<const float4*>(rr + i);
        x[i] += b.x; x[i + 1] += b.y; x[i + 2] += b.z; x[i + 3] += b.w;
      }
    }
    if (p.out_f32) {
      float* o = p.out_f32 + grow * p.ld_out + col0;
#pragma unroll
      for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(o + i) = make_float4(x[i], x[i + 1], x[i + 2], x[i + 3]);
    }
    if (p.out_bf16) {
      __nv_bfloat16* o = p.out_bf16 + grow * p.ld_out + col0;
#pragma unroll
      for (int i = 0; i < 32; i += 8) {
        uint4 q;
        q.x = pack_bf16x2(x[i], x[i + 1]);
        q.y = pack_bf16x2(x[i + 2], x[i + 3]);
        q.z = pack_bf16x2(x[i + 4], x[i + 5]);
        q.w = pack_bf16x2(x[i + 6], x[i + 7]);
        *reinterpret_cast<uint4*>(o + i) = q;
      }
    }
  }
  static constexpr int kBlockMRows = 128;
};

// -------------------------------------------------------------------------------------------
// Bias of the current column tile in shared memory. These kernels carve ~225 KB of the SM's 228 KB out as shared memory,
// which leaves no L1: a __ldg of the bias inside the chunk loop is an L2 round trip (300+ cycles) on the epilogue's critical
// path, eight of them per 32 x 32 chunk (measured on the fused feed-forward kernel: 4.0 -> 3.06 ms when its biases moved
// to shared memory). All epilogue threads call load() from begin() with the same tile sequence; the tile's <= 256 bias
// values are (re)loaded only when the column tile changes, between two named barriers of the epilogue threads.
// -------------------------------------------------------------------------------------------
struct BiasTileCache {
  float* s = nullptr;
  int nt = -1;
  __device__ __forceinline__ void init(uint8_t* smem_1kb) { s = reinterpret_cast<float*>(smem_1kb); nt = -1; }
  __device__ __forceinline__ void load(const float* bias, int N, int tile, int block_n) {
    if (tile == nt || bias == nullptr) return;   // uniform over the epilogue threads
    const int n_epi = (int)blockDim.x - 64, t = (int)threadIdx.x - 64;
    asm volatile("bar.sync 2, %0;" ::"r"(n_epi) : "memory");   // nobody still reads the previous tile's values
    for (int i = t; i < block_n; i += n_epi) s[i] = (tile * block_n + i < N) ? __ldg(bias + tile * block_n + i) : 0.0f;
    asm volatile("bar.sync 2, %0;" ::"r"(n_epi) : "memory");
    nt = tile;
  }
  __device__ __forceinline__ const float* at(int col0, int block_n) const { return s + (col0 - nt * block_n); }
};

// -------------------------------------------------------------------------------------------
// y = act(acc + bias) written through the TMA unit. A thread owns a ROW of the accumulator, so direct global
// stores put 32 different cache lines into every store instruction (ncu: 32 sectors/request, LSU-bound
// epilogue). Here each warp packs its 32x32 chunk into a swizzled shared-memory staging tile (conflict-free
// 16-byte stores) and one lane hands it to cp.async.bulk.tensor: full-line writes, no LSU traffic, and
// out-of-range rows of the last tile are clipped by the tensor map.
// -------------------------------------------------------------------------------------------
template <bool BF16_OUT>
struct EpiBiasActTma : EpiDefaults {
  struct Params {
    alignas(64) CUtensorMap tmap_out;  // [M][N] row-major, box = 32 cols x 32 rows, swizzle = row bytes of the box
    const float* bias;                 // [N] or null
    int N;
    int act;                           // 0 none, 1 relu, 2 gelu(erf)
    const float* pe;                   // [max_len][N] positional table or null: + pe[token_pos[row]] (token embedding)
    const int* token_pos;              // [M]
    int M;                             // rows (only read with pe)
  };
  // 16 epilogue warps on 256-column tiles (4 per TMEM lane quarter): the per-chunk chain tcgen05.ld -> math ->
  // staging -> fence -> TMA issue is latency-bound, more warps overlap more of it. One staging buffer per warp.
  static constexpr int kColumnSplit = 4;
  static constexpr int kChunkBytes = BF16_OUT ? 2048 : 4096;
  static constexpr int kBuffers = 1;
  static constexpr int kExtraSmemBytes = 16 * kBuffers * kChunkBytes + 1024;
  uint8_t* stage;
  int buf;
  BiasTileCache bias_cache;
  __device__ __forceinline__ void setup(const Params&, uint8_t* extra, int warp_slot, int) {
    stage = extra + warp_slot * (kBuffers * kChunkBytes);
    buf = 0;
    bias_cache.init(extra + 16 * kBuffers * kChunkBytes);
  }
  __device__ __forceinline__ void finish(const Params&, int lane) {
    if (lane == 0) tma_store_wait_read<0>();  // staging must stay valid until the TMA unit has read it
  }
  __device__ __forceinline__ void begin(const Params& p, int, int nt, int) { bias_cache.load(p.bias, p.N, nt, block_n_); }
  __device__ __forceinline__ void end(const Params&, int, int, int) {}
  __device__ __forceinline__ void chunk(const Params& p, int mt, int col0, int row, uint32_t (&v)[32], int) {
    if (col0 >= p.N) return;  // warp-uniform
    const int lane = row & 31;
    float x[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) x[i] = __uint_as_float(v[i]);
    if (p.bias) {
      const float* sb = bias_cache.at(col0, block_n_);
#pragma unroll
      for (int i = 0; i < 32; i += 4) {
        const float4 b = *reinterpret_cast<const float4*>(sb + i);
        x[i] += b.x; x[i + 1] += b.y; x[i + 2] += b.z; x[i + 3] += b.w;
      }
    }
    if (p.pe) {
      const long long grow = (long long)mt * 128 + row;
      if (grow < p.M) {
        const float* pr = p.pe + (long long)__ldg(p.token_pos + grow) * p.N + col0;
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const float4 b = __ldg(reinterpret_cast<const float4*>(pr + i));
          x[i] += b.x; x[i + 1] += b.y; x[i + 2] += b.z; x[i + 3] += b.w;
        }
      }
    }
    if (p.act == 1) {
#pragma unroll
      for (int i = 0; i < 32; ++i) x[i] = fmaxf(x[i], 0.0f);
    } else if (p.act == 2) {
#pragma unroll
      for (int i = 0; i < 32; i += 2) {
        const float2 y = gelu_erf2(make_float2(x[i], x[i + 1]));
        x[i] = y.x;
        x[i + 1] = y.y;
      }
    }
    uint8_t* dst = stage + buf * kChunkBytes;
    if (lane == 0) tma_store_wait_read<kBuffers - 1>();  // the store that last used this buffer has read it
    __syncwarp();
    if constexpr (BF16_OUT) {
      // 64-byte rows, SWIZZLE_64B: 16-byte chunk c of row r lives at chunk c ^ ((r >> 1) & 3)
      uint8_t* r0 = dst + lane * 64;
      const int sw = (lane >> 1) & 3;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint4 q;
        q.x = pack_bf16x2(x[8 * c + 0], x[8 * c + 1]);
        q.y = pack_bf16x2(x[8 * c + 2], x[8 * c + 3]);
        q.z = pack_bf16x2(x[8 * c + 4], x[8 * c + 5]);
        q.w = pack_bf16x2(x[8 * c + 6], x[8 * c + 7]);
        *reinterpret_cast<uint4*>(r0 + ((c ^ sw) << 4)) = q;
      }
    } else {
      // 128-byte rows, SWIZZLE_128B: chunk c of row r lives at chunk c ^ (r & 7)
      uint8_t* r0 = dst + lane * 128;
      const int sw = lane & 7;
#pragma unroll
      for (int c = 0; c < 8; ++c)
        *reinterpret_cast<float4*>(r0 + ((c ^ sw) << 4)) = make_float4(x[4 * c], x[4 * c + 1], x[4 * c + 2], x[4 * c + 3]);
    }
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) {
      tma_store_2d(&p.tmap_out, dst, col0, mt * 128 + (row & ~31));
      tma_store_commit();
    }
    buf = (buf + 1) % kBuffers;
  }
};

// -------------------------------------------------------------------------------------------
// conv4 epilogue: relu(acc + bias), then the 4x4 global average pool. A tile holds 8 frames x 16
// pixels, so each half-warp (16 lanes) is exactly one frame; a halving butterfly leaves lane j of
// the half-warp with the sums of columns 2j, 2j+1 of the chunk.
// -------------------------------------------------------------------------------------------
struct EpiConvPool16 : EpiDefaults {
  struct Params {
    const float* bias;        // [N]
    __nv_bfloat16* out_bf16;  // [frames][N]
    int frames, N;
  };
  static constexpr int kExtraSmemBytes = 1024;
  BiasTileCache bias_cache;
  __device__ __forceinline__ void setup(const Params&, uint8_t* extra, int, int) { bias_cache.init(extra); }
  __device__ __forceinline__ void begin(const Params& p, int, int nt, int) { bias_cache.load(p.bias, p.N, nt, block_n_); }
  __device__ __forceinline__ void end(const Params&, int, int, int) {}
  __device__ __forceinline__ void chunk(const Params& p, int mt, int col0, int row, uint32_t (&v)[32], int /*pass*/) {
    const int lane = threadIdx.x & 31;
    float x[32];
    const float* sb = bias_cache.at(col0, block_n_);
#pragma unroll
    for (int i = 0; i < 32; i += 4) {
      const float4 b = *reinterpret_cast<const float4*>(sb + i);
      x[i] = fmaxf(__uint_as_float(v[i]) + b.x, 0.0f);
      x[i + 1] = fmaxf(__uint_as_float(v[i + 1]) + b.y, 0.0f);
      x[i + 2] = fmaxf(__uint_as_float(v[i + 2]) + b.z, 0.0f);
      x[i + 3] = fmaxf(__uint_as_float(v[i + 3]) + b.w, 0.0f);
    }
#pragma unroll
    for (int half = 16, bit = 8; half >= 2; half >>= 1, bit >>= 1) {
      const bool upper = (lane & bit) != 0;
#pragma unroll
      for (int i = 0; i < half; ++i) {
        const float keep = upper ? x[i + half] : x[i];
        const float send = upper ? x[i] : x[i + half];
        x[i] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
      }
    }
    const long long frame = (long long)mt * 8 + (row >> 4);
    if (frame < p.frames) {
      const int c = col0 + 2 * (lane & 15);
      *reinterpret_cast<uint32_t*>(p.out_bf16 + frame * p.N + c) = pack_bf16x2(x[0] * 0.0625f, x[1] * 0.0625f);
    }
  }
};

// -------------------------------------------------------------------------------------------
// last layer of the head: e = acc + bias, out = e / max(||e||_2, 1e-12)  (F.normalize, model.py:294).
// BLOCK_N covers the whole embedding row, so the thread that owns the row owns the whole reduction:
// pass 0 accumulates the squared norm, pass 1 re-reads the accumulator from TMEM and writes the scaled row.
// -------------------------------------------------------------------------------------------
struct EpiBiasL2Norm : EpiDefaults {
  struct Params {
    const float* bias;  // [N]
    float* out_f32;     // [M][N]
    int M, N;           // N <= BLOCK_N, multiple of 32
  };
  static constexpr int kPasses = 2;
  static constexpr int kColumnSplit = 1;
  float sumsq;
  __device__ __forceinline__ void begin(const Params&, int, int, int) { sumsq = 0.f; }
  __device__ __forceinline__ void end(const Params&, int, int, int) {}
  __device__ __forceinline__ void chunk(const Params& p, int mt, int col0, int row, uint32_t (&v)[32], int pass) {
    const long long grow = (long long)mt * 128 + row;
    if (grow >= p.M || col0 >= p.N) return;
    float x[32];
#pragma unroll
    for (int i = 0; i < 32; i += 4) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + i));
      x[i] = __uint_as_float(v[i]) + b.x;
      x[i + 1] = __uint_as_float(v[i + 1]) + b.y;
      x[i + 2] = __uint_as_float(v[i + 2]) + b.z;
      x[i + 3] = __uint_as_float(v[i + 3]) + b.w;
    }
    if (pass == 0) {
#pragma unroll
      for (int i = 0; i < 32; ++i) sumsq += x[i] * x[i];
    } else {
      const float inv = 1.0f / fmaxf(sqrtf(sumsq), 1e-12f);
      float* o = p.out_f32 + grow * p.N + col0;
#pragma unroll
      for (int i = 0; i < 32; i += 4)
        *reinterpret_cast<float4*>(o + i) = make_float4(x[i] * inv, x[i + 1] * inv, x[i + 2] * inv, x[i + 3] * inv);
    }
  }
};

// -------------------------------------------------------------------------------------------
// similarity-join screen: emit (i, j, s) for every accumulator >= thr (bf16 inputs, fp32 accumulate).
// Survivors are rare, so one global atomic per hit is cheaper than any staging. `count` keeps
// counting past `capacity` so the caller can size a retry.
// -------------------------------------------------------------------------------------------
struct EpiJoinThreshold : EpiDefaults {
  struct Params {
    float thr;
    long long q_rows, db_rows;  // valid extents
    long long q_row0;           // global index of local query row 0 (row-block shard offset)
    int* out_i;
    int* out_j;
    float* out_s;
    unsigned long long* count;
    long long capacity;
    int tri;                    // self join: keep j >= i only (the mirrored pair is emitted by the re-score kernel)
  };
  __device__ __forceinline__ void begin(const Params&, int, int, int) {}
  __device__ __forceinline__ void end(const Params&, int, int, int) {}
  __device__ __forceinline__ void chunk(const Params& p, int mt, int col0, int row, uint32_t (&v)[32], int /*pass*/) {
    const long long qi = (long long)mt * 128 + row;
    if (qi >= p.q_rows) return;
    if (p.tri && (long long)col0 + 31 < qi) return;   // the whole chunk lies below the diagonal
    float m = __uint_as_float(v[0]);
#pragma unroll
    for (int i = 1; i < 32; ++i) m = fmaxf(m, __uint_as_float(v[i]));
    if (!(m >= p.thr)) return;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const float s = __uint_as_float(v[i]);
      const long long j = (long long)col0 + i;
      if (s >= p.thr && j < p.db_rows && (!p.tri || j >= qi)) {
        const unsigned long long slot = atomicAdd(p.count, 1ull);
        if ((long long)slot < p.capacity) {
          p.out_i[slot] = (int)(p.q_row0 + qi);
          p.out_j[slot] = (int)j;
          p.out_s[slot] = s;
        }
      }
    }
  }
};

}  // namespace vfp
