// Exact flat inner-product top-k (the arithmetic of faiss.IndexFlatIP.search, fingerprint.py:524-528):
//
//   1. screen   - the tcgen05 GEMM runs on bf16 copies with the "row-block resident" schedule; EpiTopK keeps,
//                 per query row, the 64 best APPROXIMATE scores seen over the row's column segment (sorted
//                 list in shared memory, one column of it per epilogue thread);
//   2. merge    - per query row, the segment lists are merged to the 64 best approximate candidates, which
//                 are re-scored EXACTLY in fp32 and ranked by (score desc, index asc); the top k are written;
//   3. proof    - every database row outside the candidate list has approximate score <= a64 (the worst kept
//                 one), hence exact score <= a64 + margin. If the exact k-th score beats that bound the result
//                 is provably the exact top-k; otherwise the row is flagged ...
//   4. fallback - ... and recomputed by a plain fp32 scan of the whole database (threshold = the exact k-th
//                 score found so far, which every true top-k member must reach), then ranked again.
#pragma once
#include <string>

#include "gemm_launch.cuh"
#include "token_kernels.cuh"

namespace vfp {

constexpr int kTopKCand = 64;        // approximate candidates kept per query row
constexpr int kTopKMaxK = 32;
constexpr int kTopKMaxSegments = 32;

// Candidate list of one query row = a 64-entry binary heap in shared memory with the WORST kept candidate at the root
// ((score asc, index desc) order, so the root is what a better newcomer must evict and its score is the admission
// threshold `kth`). A newcomer replaces the root and sifts down: <= 6 levels, against the ~20 shifted entries per insertion
// of the sorted list this replaces (ncu: the insertion loop was 47 % of all samples and the tensor pipe 2.6 % busy).
// Entry c of row r lives at word c*128 + r, so whatever positions the 32 lanes of a warp touch, they hit 32 different banks.
struct EpiTopK : EpiDefaults {
  struct Params {
    long long q_rows, db_rows;
    int n_segments;
    float* part_s;  // [m_tiles*128][n_segments][kTopKCand] approximate scores, descending
    int* part_i;    //   "  database indices (-1 = empty)
  };
  static constexpr int kColumnSplit = 1;
  static constexpr int kExtraSmemBytes = 2 * kTopKCand * 128 * 4;
  float kth;
  uint32_t hs, hi;   // shared-space byte addresses of this row's score / index columns
  __device__ __forceinline__ static float lds_f(uint32_t a) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; }
  __device__ __forceinline__ static int lds_i(uint32_t a) { int v; asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
  __device__ __forceinline__ static void sts_f(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
  __device__ __forceinline__ static void sts_i(uint32_t a, int v) { asm volatile("st.shared.s32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
  __device__ __forceinline__ static bool worse(float sa, int ia, float sb, int ib) { return sa < sb || (sa == sb && ia > ib); }
  // place (s, j) at the root of a heap of `n` entries and restore the heap property
  __device__ __forceinline__ void sift_down(float s, int j, int n) {
    int pos = 0;
    while (true) {
      int c = 2 * pos + 1;
      if (c >= n) break;
      float cs = lds_f(hs + c * 512);
      int ci = lds_i(hi + c * 512);
      if (c + 1 < n) {
        const float rs = lds_f(hs + (c + 1) * 512);
        const int ri = lds_i(hi + (c + 1) * 512);
        if (worse(rs, ri, cs, ci)) { cs = rs; ci = ri; ++c; }
      }
      if (!worse(cs, ci, s, j)) break;
      sts_f(hs + pos * 512, cs);
      sts_i(hi + pos * 512, ci);
      pos = c;
    }
    sts_f(hs + pos * 512, s);
    sts_i(hi + pos * 512, j);
  }
  __device__ __forceinline__ void begin(const Params&, int, int, int) {}
  __device__ __forceinline__ void end(const Params&, int, int, int) {}
  __device__ __forceinline__ void item_begin(const Params&, int, int, int row, uint8_t* extra) {
    hs = smem_u32(extra) + row * 4;
    hi = hs + kTopKCand * 128 * 4;
    for (int c = 0; c < kTopKCand; ++c) {   // 64 empty entries: a valid heap whose root any real score evicts
      sts_f(hs + c * 512, -INFINITY);
      sts_i(hi + c * 512, -1);
    }
    kth = -INFINITY;
  }
  __device__ __forceinline__ void item_end(const Params& p, int mt, int seg, int row, uint8_t*) {
    // pop the worst entry 64 times: the list comes out best-first, as the merge kernel expects ((score desc, index asc))
    const size_t base = (((size_t)mt * 128 + row) * p.n_segments + seg) * kTopKCand;
    for (int n = kTopKCand; n > 0; --n) {
      p.part_s[base + n - 1] = lds_f(hs);
      p.part_i[base + n - 1] = lds_i(hi);
      if (n > 1) sift_down(lds_f(hs + (n - 1) * 512), lds_i(hi + (n - 1) * 512), n - 1);
    }
  }
  __device__ __forceinline__ void chunk(const Params& p, int, int col0, int, uint32_t (&v)[32], int) {
    if (col0 >= p.db_rows) return;
    float m[8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
      m[i] = fmaxf(fmaxf(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1])), fmaxf(__uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3])));
    const float mx = fmaxf(fmaxf(fmaxf(m[0], m[1]), fmaxf(m[2], m[3])), fmaxf(fmaxf(m[4], m[5]), fmaxf(m[6], m[7])));
    if (!(mx > kth)) return;
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      if (!(m[g] > kth)) continue;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int i = 4 * g + e;
        const float s = __uint_as_float(v[i]);
        const int j = col0 + i;
        if (s > kth && j < p.db_rows) {  // strict: columns arrive in ascending order, so an equal score has a larger index = worse
          sift_down(s, j, kTopKCand);
          kth = lds_f(hs);
        }
      }
    }
  }
};

__device__ __forceinline__ bool topk_better(float sa, int ia, float sb, int ib) {
  return sa > sb || (sa == sb && ia < ib);
}

// One warp per fp32 dot product of two dim-wide rows (dim % 4 == 0, dim <= 128 * NV): lane l holds the NV float4 at
// l * NV .. l * NV + NV - 1 of the row, zeros past dim (each adds +0). NV = ceil(dim / 128); at dim = 256 (NV = 2) this
// is eight consecutive values per lane, the layout and summation order of the 256-wide kernels.
template <int NV>
__device__ __forceinline__ void warp_row_load(float (&v)[4 * NV], const float* __restrict__ row, int dim, int lane) {
  const float4* r = reinterpret_cast<const float4*>(row) + lane * NV;
#pragma unroll
  for (int u = 0; u < NV; ++u) {
    const float4 a = (dim == 128 * NV || lane * NV + u < dim / 4) ? r[u] : make_float4(0.f, 0.f, 0.f, 0.f);
    v[4 * u] = a.x; v[4 * u + 1] = a.y; v[4 * u + 2] = a.z; v[4 * u + 3] = a.w;
  }
}

// exact fp32 dot of the warp's query (warp_row_load layout in qv) with database row j
template <int NV>
__device__ __forceinline__ float warp_dot(const float (&qv)[4 * NV], const float* __restrict__ db, long long j, int dim, int lane) {
  float dv[4 * NV];
  warp_row_load<NV>(dv, db + (size_t)j * dim, dim, lane);
  float s = qv[0] * dv[0];
#pragma unroll
  for (int i = 1; i < 4 * NV; ++i) s += qv[i] * dv[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  return s;
}

// One warp per query row: merge segment lists -> 64 approximate candidates -> exact re-score -> rank -> top k.
template <int NV>
__global__ void __launch_bounds__(256)
topk_merge_rescore_kernel(const float* __restrict__ q, const float* __restrict__ db, long long n_q, long long n_db, int dim, int k,
                          int n_segments, const float* __restrict__ part_s, const int* __restrict__ part_i, float margin,
                          float* __restrict__ out_s, long long* __restrict__ out_idx, int* __restrict__ flagged_rows,
                          float* __restrict__ flagged_tau, unsigned long long* __restrict__ flags /*[0] = flagged rows*/) {
  const int lane = threadIdx.x & 31;
  const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n_q) return;
  const float* ps = part_s + (size_t)row * n_segments * kTopKCand;
  const int* pi = part_i + (size_t)row * n_segments * kTopKCand;

  // ---- merge: lane s walks segment s (each list is sorted); 64 rounds of warp arg-max over the heads ----
  int head = 0;
  float cs[2] = {-INFINITY, -INFINITY};  // candidate c lives in lane c % 32, slot c / 32
  int ci[2] = {-1, -1};
  for (int c = 0; c < kTopKCand; ++c) {
    float hs = -INFINITY;
    int hi = 0x7fffffff;
    if (lane < n_segments && head < kTopKCand) {
      hs = ps[lane * kTopKCand + head];
      hi = pi[lane * kTopKCand + head];
      if (hi < 0) { hs = -INFINITY; hi = 0x7fffffff; }
    }
    float bs = hs;
    int bi = hi, bl = lane;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float os = __shfl_xor_sync(0xffffffffu, bs, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      const int ol = __shfl_xor_sync(0xffffffffu, bl, o);
      if (topk_better(os, oi, bs, bi)) { bs = os; bi = oi; bl = ol; }
    }
    if (bi == 0x7fffffff) break;  // all lists exhausted (n_db < 64)
    if (lane == bl) ++head;
    if (lane == (c & 31)) { cs[c >> 5] = bs; ci[c >> 5] = bi; }
  }
  // worst approximate score kept (lane 31, slot 1 = candidate 63); -inf if the list is not full
  const float a_last = __shfl_sync(0xffffffffu, cs[1], 31);
  const int i_last = __shfl_sync(0xffffffffu, ci[1], 31);

  // ---- exact re-score ----
  float qv[4 * NV];
  warp_row_load<NV>(qv, q + (size_t)row * dim, dim, lane);
  float es[2] = {-INFINITY, -INFINITY};
  for (int c = 0; c < kTopKCand; ++c) {
    const int idx = __shfl_sync(0xffffffffu, ci[c >> 5], c & 31);
    if (idx < 0) continue;  // warp-uniform
    const float s = warp_dot<NV>(qv, db, idx, dim, lane);
    if (lane == (c & 31)) es[c >> 5] = s;
  }
  // ---- rank by (exact score desc, index asc) ----
  int rank[2] = {0, 0};
  for (int c = 0; c < kTopKCand; ++c) {
    const float s = __shfl_sync(0xffffffffu, es[c >> 5], c & 31);
    const int idx = __shfl_sync(0xffffffffu, ci[c >> 5], c & 31);
    if (idx < 0) continue;
#pragma unroll
    for (int h = 0; h < 2; ++h)
      if (ci[h] >= 0 && topk_better(s, idx, es[h], ci[h])) ++rank[h];
  }
  float kth_exact = -INFINITY;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    if (ci[h] >= 0 && rank[h] < k) {
      out_s[(size_t)row * k + rank[h]] = es[h];
      out_idx[(size_t)row * k + rank[h]] = ci[h];
      if (rank[h] == k - 1) kth_exact = es[h];
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) kth_exact = fmaxf(kth_exact, __shfl_xor_sync(0xffffffffu, kth_exact, o));
  // ---- proof of exactness ----
  const bool list_is_everything = i_last < 0;  // fewer than 64 database rows exist in total
  const bool proven = list_is_everything || (kth_exact > a_last + margin);
  if (!proven && lane == 0) {   // the flag lists hold one slot per query row: they cannot overflow
    const unsigned long long slot = atomicAdd(&flags[0], 1ull);
    flagged_rows[slot] = (int)row;
    flagged_tau[slot] = kth_exact;
  }
}

// Exact fallback, pass 1. A flagged query row is one whose 64 screened candidates could not be PROVEN to contain the exact
// top k (dense neighbourhoods, large groups of identical embeddings - both normal in a duplicate detector). Such a row is
// re-searched with a plain fp32 scan of the whole database; nothing here has a capacity a data set can overflow:
// block (slice s, flagged row f) scans database rows s*8 + warp, + 128, ... and every warp keeps its own exact best-32 list
// ((score desc, index asc), one entry per lane, sorted insertion with one ballot + one shuffle), the block merges its eight
// lists and writes its k best to part[f][s][0..k). tau (the exact k-th score among the screened candidates, a lower bound
// of the true k-th score) only prunes. Flagged rows are processed in batches of kTopKBatch so the part buffer stays small.
constexpr int kTopKSlices = 16;
constexpr int kTopKBatch = 8192;

template <int NV>
__global__ void __launch_bounds__(256)
topk_fallback_scan_kernel(const float* __restrict__ q, const float* __restrict__ db, long long n_db, int dim, int k, long long batch0,
                          const int* __restrict__ flagged_rows, const float* __restrict__ flagged_tau,
                          const unsigned long long* __restrict__ flags, float* __restrict__ part_s, int* __restrict__ part_i) {
  __shared__ float ms[8 * 32];
  __shared__ int mi[8 * 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long nf = (long long)flags[0];
  const int slice = blockIdx.x;
  for (long long f = batch0 + blockIdx.y; f < nf && f < batch0 + kTopKBatch; f += gridDim.y) {
    const int row = flagged_rows[f];
    const float tau = flagged_tau[f];
    float qv[4 * NV];
    warp_row_load<NV>(qv, q + (size_t)row * dim, dim, lane);
    float ls = -INFINITY;       // this lane's entry of the warp's sorted list (lane 0 = best)
    int li = 0x7fffffff;
    float ws = -INFINITY;       // entry k-1 (the admission threshold), known to every lane
    int wi = 0x7fffffff;
    for (long long j = (long long)slice * 8 + warp; j < n_db; j += kTopKSlices * 8) {
      const float sc = warp_dot<NV>(qv, db, j, dim, lane);
      if (sc >= tau && topk_better(sc, (int)j, ws, wi)) {   // warp-uniform
        const int pos = __popc(__ballot_sync(0xffffffffu, topk_better(ls, li, sc, (int)j)));
        const float us = __shfl_up_sync(0xffffffffu, ls, 1);
        const int ui = __shfl_up_sync(0xffffffffu, li, 1);
        if (lane == pos) { ls = sc; li = (int)j; }
        else if (lane > pos) { ls = us; li = ui; }
        ws = __shfl_sync(0xffffffffu, ls, k - 1);
        wi = __shfl_sync(0xffffffffu, li, k - 1);
      }
    }
    __syncthreads();   // the previous row's merge has been read
    ms[warp * 32 + lane] = ls;
    mi[warp * 32 + lane] = li;
    __syncthreads();
    {
      const float es = ms[threadIdx.x];
      const int ei = mi[threadIdx.x];
      if (ei != 0x7fffffff) {
        int rank = 0;
        for (int o = 0; o < 256; ++o) rank += topk_better(ms[o], mi[o], es, ei) ? 1 : 0;
        if (rank < k) {
          const size_t base = ((size_t)(f - batch0) * kTopKSlices + slice) * kTopKMaxK;
          part_s[base + rank] = es;
          part_i[base + rank] = ei;
        }
      }
    }
  }
}

// Exact fallback, pass 2: merge the slices' lists of each flagged row and overwrite its output row.
__global__ void __launch_bounds__(128)
topk_fallback_rank_kernel(int k, long long batch0, const int* __restrict__ flagged_rows, const unsigned long long* __restrict__ flags,
                          const float* __restrict__ part_s, const int* __restrict__ part_i, float* __restrict__ out_s,
                          long long* __restrict__ out_idx) {
  const long long nf = (long long)flags[0];
  constexpr int n = kTopKSlices * kTopKMaxK;
  for (long long f = batch0 + blockIdx.x; f < nf && f < batch0 + kTopKBatch; f += gridDim.x) {
    const int row = flagged_rows[f];
    const float* bs = part_s + (size_t)(f - batch0) * n;
    const int* bi = part_i + (size_t)(f - batch0) * n;
    for (int c = threadIdx.x; c < n; c += blockDim.x) {
      const int idx = bi[c];
      if (idx < 0 || (c & (kTopKMaxK - 1)) >= k) continue;   // empty slot / beyond the slice's k best
      const float sc = bs[c];
      int rank = 0;
      for (int o = 0; o < n; ++o) {
        const int oi = bi[o];
        if (oi >= 0 && (o & (kTopKMaxK - 1)) < k) rank += topk_better(bs[o], oi, sc, idx) ? 1 : 0;
      }
      if (rank < k) {
        out_s[(size_t)row * k + rank] = sc;
        out_idx[(size_t)row * k + rank] = idx;
      }
    }
  }
}

// part_i = -1 everywhere (a slice with fewer than k rows >= tau leaves empty slots)
__global__ void topk_fill_kernel(int* __restrict__ p, long long n, int v, const unsigned long long* __restrict__ flags, long long batch0) {
  if ((long long)flags[0] <= batch0) return;   // no flagged row in this batch
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) p[i] = v;
}

struct TopKWs {
  size_t qbf, dbbf, part_s, part_i, flagged_rows, flagged_tau, fb_s, fb_i, flags, total;
  int n_segments;
  long long rows_padded;
};
inline TopKWs topk_ws_layout(int64_t n_q, int64_t n_db, int dim) {
  TopKWs L{};
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off = (off + bytes + 1023) / 1024 * 1024;
    return o;
  };
  const int64_t m_tiles = (n_q + 127) / 128;
  const int64_t n_tiles = (n_db + 255) / 256;
  // Database segments per query tile: work item = (128 query rows, one contiguous segment). More segments fill the last round
  // of the persistent grid better, but every (row, segment) heap starts cold: its first ~64 ln(rows / 64) candidates are
  // all insertions. Measured on 10 M rows (profiles/r02_bench_n*.json, cfg 5): an item costs 7.7 ns per database row plus
  // ~1 ms per e-fold of segment length; e.g. 12 500 queries per GPU: 8 segments 125 ms, 3 segments (two full rounds) 74 ms.
  int seg = 1;
  double best = 1e300;
  for (int cand = 1; cand <= kTopKMaxSegments && cand <= n_tiles; ++cand) {
    const double len = (double)n_db / cand;
    const double item_ms = 7.68e-6 * len + 1.0 * log(std::max(len / 64.0, 2.0));
    const double cost = ceil((double)m_tiles * cand / 148.0) * item_ms;
    if (cost < 0.97 * best) { best = cost; seg = cand; }
  }
  L.n_segments = seg;
  L.rows_padded = m_tiles * 128;
  const int64_t batch = std::min<int64_t>(n_q, kTopKBatch);
  L.qbf = take((size_t)n_q * 2 * dim);    // bf16 screen copies, 2 * dim bytes per row
  L.dbbf = take((size_t)n_db * 2 * dim);
  L.part_s = take((size_t)L.rows_padded * seg * kTopKCand * 4);
  L.part_i = take((size_t)L.rows_padded * seg * kTopKCand * 4);
  L.flagged_rows = take((size_t)n_q * 4);
  L.flagged_tau = take((size_t)n_q * 4);
  L.fb_s = take((size_t)batch * kTopKSlices * kTopKMaxK * 4);
  L.fb_i = take((size_t)batch * kTopKSlices * kTopKMaxK * 4);
  L.flags = take(64);
  L.total = off;
  return L;
}
inline size_t topk_workspace_bytes(int64_t n_q, int64_t n_db, int k, int dim) {
  (void)k;
  if (n_q <= 0 || n_db <= 0) return 0;
  return topk_ws_layout(n_q, n_db, dim).total;
}

// Exact stages after the screen: merge + re-score, then the fallback scan of the flagged rows, kTopKBatch at a time. The
// number of flagged rows is only known on the device, so every possible batch is launched and the blocks of a batch past the
// count exit at once (no host synchronisation; a batch with nothing to do costs two empty launches).
template <int NV>
inline void topk_exact(const float* q, const float* db, int64_t n_q, int64_t n_db, int dim, int k, float margin, const TopKWs& L,
                       uint8_t* ws, float* out_s, int64_t* out_idx, cudaStream_t st) {
  float* part_s = reinterpret_cast<float*>(ws + L.part_s);
  int* part_i = reinterpret_cast<int*>(ws + L.part_i);
  int* flagged_rows = reinterpret_cast<int*>(ws + L.flagged_rows);
  float* flagged_tau = reinterpret_cast<float*>(ws + L.flagged_tau);
  float* fb_s = reinterpret_cast<float*>(ws + L.fb_s);
  int* fb_i = reinterpret_cast<int*>(ws + L.fb_i);
  unsigned long long* flags = reinterpret_cast<unsigned long long*>(ws + L.flags);
  topk_merge_rescore_kernel<NV><<<(unsigned)((n_q * 32 + 255) / 256), 256, 0, st>>>(
      q, db, n_q, n_db, dim, k, L.n_segments, part_s, part_i, margin, out_s, reinterpret_cast<long long*>(out_idx), flagged_rows,
      flagged_tau, flags);
  const long long batch_rows = std::min<long long>(n_q, kTopKBatch);
  for (long long b0 = 0; b0 < n_q; b0 += kTopKBatch) {
    topk_fill_kernel<<<device_sm_count() * 4, 256, 0, st>>>(fb_i, batch_rows * kTopKSlices * kTopKMaxK, -1, flags, b0);
    topk_fallback_scan_kernel<NV><<<dim3(kTopKSlices, (unsigned)std::min<long long>(batch_rows, 2 * device_sm_count())), 256, 0, st>>>(
        q, db, n_db, dim, k, b0, flagged_rows, flagged_tau, flags, fb_s, fb_i);
    topk_fallback_rank_kernel<<<(unsigned)std::min<long long>(batch_rows, 2 * device_sm_count()), 128, 0, st>>>(
        k, b0, flagged_rows, flags, fb_s, fb_i, out_s, reinterpret_cast<long long*>(out_idx));
  }
}

inline int topk_run(const float* q, const float* db, int64_t n_q, int64_t n_db, int dim, int k, float margin, float* out_s,
                    int64_t* out_idx, unsigned long long* flags_out, uint8_t* ws, cudaStream_t st, std::string* err) {
  const TopKWs L = topk_ws_layout(n_q, n_db, dim);
  const bool self = (q == db && n_q == n_db);
  __nv_bfloat16* qbf = reinterpret_cast<__nv_bfloat16*>(ws + L.qbf);
  __nv_bfloat16* dbbf = self ? qbf : reinterpret_cast<__nv_bfloat16*>(ws + L.dbbf);
  float* part_s = reinterpret_cast<float*>(ws + L.part_s);
  int* part_i = reinterpret_cast<int*>(ws + L.part_i);
  unsigned long long* flags = reinterpret_cast<unsigned long long*>(ws + L.flags);
  auto ck = [&](cudaError_t e, const char* what) {
    if (e != cudaSuccess) { *err = std::string(what) + ": " + cudaGetErrorString(e); return true; }
    return false;
  };
  if (ck(cudaMemsetAsync(flags, 0, 64, st), "memset")) return 1;
  const long long q8 = n_q * dim / 8, db8 = n_db * dim / 8;   // 8 elements per thread
  f32_to_bf16_kernel<<<(unsigned)((q8 + 255) / 256), 256, 0, st>>>(q, qbf, q8);
  if (!self) f32_to_bf16_kernel<<<(unsigned)((db8 + 255) / 256), 256, 0, st>>>(db, dbbf, db8);
  // unpadded bf16 rows (inner extent dim, pitch 2 * dim bytes): TMA zero-fills the columns past dim in the last K block. The
  // screen streams A and B through one ring of 3 stages of one K block each, so its shared memory does not depend on dim.
  CUtensorMap ta, tb;
  if (make_tmap_rows_bf16(&ta, qbf, (uint64_t)n_q, dim, dim, 128, 64) || make_tmap_rows_bf16(&tb, dbbf, (uint64_t)n_db, dim, dim, 256, 64)) {
    *err = "tensor map encode failed";
    return 1;
  }
  GemmShape s = plain_shape(n_q, 0, (dim + 63) / 64 * 64, 256, 64, 1);
  s.n_tiles = (int)((n_db + 255) / 256);
  s.row_resident = 1;
  s.n_segments = L.n_segments;
  EpiTopK::Params ep{};
  ep.q_rows = n_q; ep.db_rows = n_db; ep.n_segments = L.n_segments; ep.part_s = part_s; ep.part_i = part_i;
  if (ck((launch_gemm<256, 64, 3, EpiTopK>(ta, tb, s, ep, st)), "screen launch")) return 1;
  switch ((dim + 127) / 128) {
    case 1: topk_exact<1>(q, db, n_q, n_db, dim, k, margin, L, ws, out_s, out_idx, st); break;
    case 2: topk_exact<2>(q, db, n_q, n_db, dim, k, margin, L, ws, out_s, out_idx, st); break;
    case 3: topk_exact<3>(q, db, n_q, n_db, dim, k, margin, L, ws, out_s, out_idx, st); break;
    case 4: topk_exact<4>(q, db, n_q, n_db, dim, k, margin, L, ws, out_s, out_idx, st); break;
  }
  if (ck(cudaMemcpyAsync(flags_out, flags, 16, cudaMemcpyDeviceToDevice, st), "copy flags") || ck(cudaGetLastError(), "top-k kernels")) return 1;
  return 0;
}

}  // namespace vfp
