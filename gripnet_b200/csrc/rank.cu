// K16: filtered candidate ranking (OGB rank rule, per-relation MRR / Hits@k) and top-k link prediction of the
// DistMult decoder.  Every candidate tail c of a query (s, r) is scored as one row of S = Q . z^T with
// Q[g] = z[s_g] .* w[r_g]; the product itself is the existing dense GEMM (gn_sgemm / gn_tc_gemm).  This file holds
// what sits around it: the (src, rel)-grouped edge structure, the query rows, the filtered rank count, the
// per-relation reduction and the per-query top-k selection.
// Relation queries (s, ?, t) of a directed pair score every relation r' as one row of S = P . W^T with
// P[g] = z[s_g] .* z[t_g]; they share the count and top-k kernels, templated on how a row finds its filter row, and
// add a pair-grouped structure (rows = distinct directed pairs, sorted by (src, dst)) and a pair lookup.
#include "sortkit.cuh"

namespace gn {

constexpr int kRankMaxHits = 8;
constexpr int kTopkThreads = 256;
constexpr int kTopkMax = 256;                  // largest k: one selected key per thread of the sort
constexpr uint32_t kMaskedBits = 0xffffffffu;  // NaN payload no arithmetic produces: "filtered" in a top-k row

// ---------------------------------------------------------------------------------------------------------------
// grouped edge structure: rows s*R + r, entries (dst, edge id) sorted by dst inside a row (two stable counting
// sorts: by dst, then by row), and the compacted list of non-empty rows
// ---------------------------------------------------------------------------------------------------------------
__global__ void rank_dst_keys_kernel(const int64_t* __restrict__ dst, int64_t n, int32_t* __restrict__ key) {
  const int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e < n) key[e] = int32_t(dst[e]);
}

__global__ void rank_row_keys_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ etype,
                                     const int32_t* __restrict__ perm, int64_t n, int32_t n_rel,
                                     int32_t* __restrict__ key) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t e = perm[i];
  key[i] = int32_t(src[e]) * n_rel + int32_t(etype[e]);
}

__global__ void rank_fill_kernel(const int64_t* __restrict__ dst, const int32_t* __restrict__ eid, int64_t n,
                                 int32_t* __restrict__ ent_dst) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) ent_dst[i] = int32_t(dst[eid[i]]);
}

__global__ void rank_row_flags_kernel(const int32_t* __restrict__ rowptr, int32_t n_rows, int32_t* __restrict__ flag) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n_rows) flag[r] = rowptr[r + 1] > rowptr[r] ? 1 : 0;
}

__global__ void rank_groups_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ pos, int32_t n_rows,
                                   int32_t* __restrict__ group_row) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n_rows && rowptr[r + 1] > rowptr[r]) group_row[pos[r]] = r;
}

// ---------------------------------------------------------------------------------------------------------------
// pair-grouped structure: entries ordered by (src, dst, rel) with three stable counting sorts (by rel, by dst, by
// src), rows = the distinct directed pairs in that order, entries (rel, edge id) sorted by rel inside a row.  Rows
// are compacted pairs, not s*n + t: n^2 does not fit int32 for general n.
// ---------------------------------------------------------------------------------------------------------------
__global__ void rank_gather_keys_kernel(const int64_t* __restrict__ v, const int32_t* __restrict__ perm, int64_t n,
                                        int32_t* __restrict__ key) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) key[i] = int32_t(v[perm ? perm[i] : int32_t(i)]);
}

__global__ void rank_pair_heads_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                       const int32_t* __restrict__ eid, int64_t n, int32_t* __restrict__ flag) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t e = eid[i];
  flag[i] = i == 0 || src[e] != src[eid[i - 1]] || dst[e] != dst[eid[i - 1]] ? 1 : 0;
}

__global__ void rank_pair_fill_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                      const int64_t* __restrict__ etype, const int32_t* __restrict__ eid,
                                      const int32_t* __restrict__ flag, const int32_t* __restrict__ pos, int64_t n,
                                      int32_t* __restrict__ rowptr, int32_t* __restrict__ pair_src,
                                      int32_t* __restrict__ pair_dst, int32_t* __restrict__ ent_rel) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t e = eid[i];
  ent_rel[i] = int32_t(etype[e]);
  if (flag[i]) {
    const int32_t p = pos[i];
    rowptr[p] = int32_t(i);
    pair_src[p] = int32_t(src[e]);
    pair_dst[p] = int32_t(dst[e]);
  }
  if (i == n - 1) rowptr[pos[i] + flag[i]] = int32_t(n);
}

// row of the filter's pair (s, t) by binary search over its (src, dst)-sorted pairs, or -1
__global__ void rank_pair_lookup_kernel(const int32_t* __restrict__ f_src, const int32_t* __restrict__ f_dst,
                                        int32_t n_fpairs, const int32_t* __restrict__ pair_src,
                                        const int32_t* __restrict__ pair_dst, const int64_t* __restrict__ src,
                                        const int64_t* __restrict__ dst, int64_t count, int32_t* __restrict__ row) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const int32_t s = pair_src ? pair_src[i] : int32_t(src[i]);
  const int32_t t = pair_src ? pair_dst[i] : int32_t(dst[i]);
  int lo = 0, hi = n_fpairs;
  while (lo < hi) {
    const int mid = lo + ((hi - lo) >> 1);
    const int32_t ms = f_src[mid];
    if (ms < s || (ms == s && f_dst[mid] < t)) lo = mid + 1;
    else hi = mid;
  }
  row[i] = (lo < n_fpairs && f_src[lo] == s && f_dst[lo] == t) ? lo : -1;
}

// ---------------------------------------------------------------------------------------------------------------
// query rows q[i, :] = a_i .* b_i.  Tail queries: a = z[s], b = w[r], (s, r) from a group row id s*R + r or from two
// index lists.  Relation queries: a = z[s], b = z[t], (s, t) from a pair-grouped structure or from two index lists.
// ---------------------------------------------------------------------------------------------------------------
struct TailOperands {
  const float* z;
  int64_t ldz;
  const float* w;
  int D;
  int32_t n_rel;
  const int32_t* group_row;
  const int64_t* node;
  const int64_t* rel;
  __device__ __forceinline__ void at(int64_t i, const float*& a, const float*& b) const {
    int64_t s, r;
    if (group_row != nullptr) {
      const int32_t g = group_row[i];
      s = g / n_rel;
      r = g - s * n_rel;
    } else {
      s = node[i];
      r = rel[i];
    }
    a = z + s * ldz;
    b = w + r * D;
  }
};

struct PairOperands {
  const float* z;
  int64_t ldz;
  const int32_t* pair_src;    // group pairs, or nullptr: the index lists
  const int32_t* pair_dst;
  const int64_t* src;
  const int64_t* dst;
  __device__ __forceinline__ void at(int64_t i, const float*& a, const float*& b) const {
    const int64_t s = pair_src ? int64_t(pair_src[i]) : src[i];
    const int64_t t = pair_src ? int64_t(pair_dst[i]) : dst[i];
    a = z + s * ldz;
    b = z + t * ldz;
  }
};

template <class Operands>
__global__ void rank_query_rows_kernel(const Operands ops, int D, int64_t count, float* __restrict__ q, int64_t ldq) {
  const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= count * D) return;
  const int64_t i = t / D;
  const int f = int(t - i * D);
  const float *a, *b;
  ops.at(i, a, b);
  q[i * ldq + f] = a[f] * b[f];
}

// ---------------------------------------------------------------------------------------------------------------
// filtered rank: one warp per group (a row of S), the group's targets in turn.  opt / pess count the candidates
// c != t above / at-or-above S(t) over the whole row, then the distinct filtered candidates other than t that met
// the same comparisons are taken back out.  S(t) is read from the same row as every S(c).  Rows says where group g's
// targets and filter entries are: tail groups use the row s*R + r of both structures, relation groups (pairs) their
// own compacted row and the filter row found by gn_rank_pair_lookup (-1: the pair has no filtered triple).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kCountWarps = 8;

struct TailRows {
  const int32_t* group_row;
  bool filtered;
  __device__ __forceinline__ int32_t query(int g) const { return group_row[g]; }
  __device__ __forceinline__ int32_t filter(int g) const { return filtered ? group_row[g] : -1; }
};

struct PairRows {
  const int32_t* f_row;       // nullptr: no filter
  __device__ __forceinline__ int32_t query(int g) const { return g; }
  __device__ __forceinline__ int32_t filter(int g) const { return f_row ? f_row[g] : -1; }
};

template <class Rows>
__global__ void __launch_bounds__(kCountWarps * 32) rank_count_kernel(
    const float* __restrict__ S, int64_t lds, int32_t n, const Rows rows, int32_t n_groups,
    const int32_t* __restrict__ q_rowptr, const int32_t* __restrict__ q_dst, const int32_t* __restrict__ q_eid,
    const int32_t* __restrict__ f_rowptr, const int32_t* __restrict__ f_dst, float* __restrict__ rank) {
  const int lane = threadIdx.x & 31;
  const int g = blockIdx.x * kCountWarps + (threadIdx.x >> 5);
  if (g >= n_groups) return;
  const int32_t row = rows.query(g), frow = rows.filter(g);
  const float* srow = S + int64_t(g) * lds;
  const int f0 = frow >= 0 ? f_rowptr[frow] : 0, f1 = frow >= 0 ? f_rowptr[frow + 1] : 0;
  for (int j = q_rowptr[row]; j < q_rowptr[row + 1]; ++j) {
    const int t = q_dst[j];
    const float st = srow[t];
    int opt = 0, pess = 0;
    for (int c = lane; c < n; c += 32) {
      const float v = srow[c];
      opt += (c != t) & (v > st);
      pess += (c != t) & (v >= st);
    }
    for (int k = f0 + lane; k < f1; k += 32) {
      const int c = f_dst[k];
      if (c == t || (k > f0 && f_dst[k - 1] == c)) continue;   // the target itself; duplicates count once
      const float v = srow[c];
      opt -= v > st;
      pess -= v >= st;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      opt += __shfl_xor_sync(kFull, opt, o);
      pess += __shfl_xor_sync(kFull, pess, o);
    }
    if (lane == 0) rank[q_eid[j]] = 1.0f + 0.5f * float(opt + pess);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// per-relation MRR / Hits@k: one block per relation, a fixed entry -> thread assignment and a fixed tree (float64)
// ---------------------------------------------------------------------------------------------------------------
struct HitsK {
  int32_t k[kRankMaxHits];
};

constexpr int kMetricThreads = 256;

__global__ void __launch_bounds__(kMetricThreads) rank_metrics_kernel(const float* __restrict__ rank,
                                                                      const int32_t* __restrict__ rel_rowptr,
                                                                      const int32_t* __restrict__ rel_perm,
                                                                      int32_t n_rel, HitsK hk, int n_hits,
                                                                      double* __restrict__ out) {
  __shared__ double red[kMetricThreads];
  __shared__ int hred[kRankMaxHits][kMetricThreads];
  const int r = blockIdx.x;
  const int b = rel_rowptr[r], e = rel_rowptr[r + 1];
  double s = 0.0;
  int h[kRankMaxHits];
#pragma unroll
  for (int i = 0; i < kRankMaxHits; ++i) h[i] = 0;
  for (int i = b + threadIdx.x; i < e; i += kMetricThreads) {
    const float rk = rank[rel_perm[i]];
    s += 1.0 / double(rk);
#pragma unroll
    for (int m = 0; m < kRankMaxHits; ++m) h[m] += (m < n_hits && rk <= float(hk.k[m])) ? 1 : 0;
  }
  red[threadIdx.x] = s;
#pragma unroll
  for (int m = 0; m < kRankMaxHits; ++m) hred[m][threadIdx.x] = h[m];
  __syncthreads();
  for (int w = kMetricThreads / 2; w > 0; w >>= 1) {
    if (threadIdx.x < w) {
      red[threadIdx.x] += red[threadIdx.x + w];
#pragma unroll
      for (int m = 0; m < kRankMaxHits; ++m) hred[m][threadIdx.x] += hred[m][threadIdx.x + w];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const int cnt = e - b;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    out[r] = cnt ? red[0] / double(cnt) : nan;
    for (int m = 0; m < n_hits; ++m) out[int64_t(1 + m) * n_rel + r] = cnt ? double(hred[m][0]) / double(cnt) : nan;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// top-k: one block per query row.  A candidate's key is (order-preserving bits of its score) << 32 | ~id, so keys
// are distinct, a larger key is a higher score and, among equal scores, a smaller id; a filtered candidate (its S
// entry overwritten with kMaskedBits first) has key 0.  The k-th largest key is found by an MSB-first radix select
// (8 passes of 8 bits over the row, read from L1 / L2), the keys at or above it are gathered and bitonic-sorted.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t score_key(uint32_t b, uint32_t id) {
  const uint32_t u = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return (uint64_t(u) << 32) | uint64_t(~id);
}

__device__ __forceinline__ uint64_t topk_key(const float* srow, int c) {
  const uint32_t b = __float_as_uint(srow[c]);
  if (b == kMaskedBits) return 0ull;
  return score_key(b, uint32_t(c));
}

__device__ __forceinline__ float topk_score(uint64_t key) {
  const uint32_t u = uint32_t(key >> 32);
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// The k (<= kTopkMax) largest non-zero keys among keys(0 .. m-1), sorted descending into the returned shared array
// of kTopkMax slots (0 past the last one).  Block-wide, kTopkThreads threads; keys(c) is read several times.
template <class Keys>
__device__ __forceinline__ const uint64_t* topk_select(const Keys& keys, int m, int k) {
  __shared__ int hist[256];
  __shared__ uint64_t sel[kTopkMax];
  __shared__ int warp_cnt[kTopkThreads / 32];
  __shared__ uint64_t prefix_s;
  __shared__ int remaining_s, n_sel;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // admissible candidates
  int a = 0;
  for (int c = tid; c < m; c += kTopkThreads) a += keys(c) != 0ull;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(kFull, a, o);
  if (lane == 0) warp_cnt[warp] = a;
  __syncthreads();
  int admissible = 0;
#pragma unroll
  for (int w = 0; w < kTopkThreads / 32; ++w) admissible += warp_cnt[w];
  uint64_t thresh = 1ull;                      // fewer than k admissible: every admissible key
  if (admissible > k) {
    if (tid == 0) {
      prefix_s = 0ull;
      remaining_s = k;
    }
    uint64_t mask = 0ull;
    for (int shift = 56; shift >= 0; shift -= 8) {
      hist[tid] = 0;
      __syncthreads();
      const uint64_t prefix = prefix_s;
      for (int c = tid; c < m; c += kTopkThreads) {
        const uint64_t key = keys(c);
        if (key != 0ull && (key & mask) == prefix) atomicAdd(&hist[int(key >> shift) & 255], 1);
      }
      __syncthreads();
      if (warp == 0) {
        // lane l owns digits 255-8l .. 248-8l (descending); find the digit at which the running count from the
        // top reaches `remaining`
        int cnt[8], tot = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          cnt[i] = hist[255 - 8 * lane - i];
          tot += cnt[i];
        }
        int incl = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int t = __shfl_up_sync(kFull, incl, o);
          if (lane >= o) incl += t;
        }
        const int rem = remaining_s;
        const unsigned hit = __ballot_sync(kFull, incl >= rem);
        const int owner = __ffs(hit) - 1;
        if (lane == owner) {
          int run = incl - tot;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (run + cnt[i] >= rem) {
              prefix_s = prefix | (uint64_t(255 - 8 * lane - i) << shift);
              remaining_s = rem - run;
              break;
            }
            run += cnt[i];
          }
        }
      }
      mask |= 0xffull << shift;
      __syncthreads();
    }
    thresh = prefix_s;
  }
  if (tid == 0) n_sel = 0;
  sel[tid] = 0ull;
  __syncthreads();
  for (int c = tid; c < m; c += kTopkThreads) {
    const uint64_t key = keys(c);
    if (key != 0ull && key >= thresh) {
      const int at = atomicAdd(&n_sel, 1);
      if (at < kTopkMax) sel[at] = key;
    }
  }
  __syncthreads();
  // bitonic sort of the 256 slots, descending
  for (int size = 2; size <= kTopkMax; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      const int partner = tid ^ stride;
      if (partner > tid) {
        const uint64_t x = sel[tid], y = sel[partner];
        const bool desc = (tid & size) == 0;
        if (desc ? (x < y) : (x > y)) {
          sel[tid] = y;
          sel[partner] = x;
        }
      }
      __syncthreads();
    }
  }
  return sel;
}

// the returned score of a selected key (NaN for an empty slot), after the sigmoid when `sigmoid`
__device__ __forceinline__ float topk_out_score(uint64_t key, int sigmoid) {
  float v = __uint_as_float(0x7fc00000u);
  if (key != 0ull) {
    v = topk_score(key);
    if (sigmoid) v = 1.0f / (1.0f + expf(-v));
  }
  return v;
}

// the filter row of query row qi (-1: none): s*R + r of a tail query, the looked-up pair row of a relation query
struct TailFilterRow {
  const int64_t* node;
  const int64_t* rel;
  int32_t n_rel;
  bool filtered;
  __device__ __forceinline__ int64_t operator()(int64_t qi) const { return filtered ? node[qi] * n_rel + rel[qi] : -1; }
};

struct PairFilterRow {
  const int32_t* f_row;       // nullptr: no filter
  __device__ __forceinline__ int64_t operator()(int64_t qi) const { return f_row ? f_row[qi] : -1; }
};

struct RowKeys {
  const float* srow;
  __device__ __forceinline__ uint64_t operator()(int c) const { return topk_key(srow, c); }
};

template <class FilterRow>
__global__ void __launch_bounds__(kTopkThreads) rank_topk_kernel(float* __restrict__ S, int64_t lds, int32_t n,
                                                                 const FilterRow filter_row,
                                                                 const int32_t* __restrict__ f_rowptr,
                                                                 const int32_t* __restrict__ f_dst, int k, int sigmoid,
                                                                 float* __restrict__ out_score,
                                                                 int64_t* __restrict__ out_id) {
  const int tid = threadIdx.x;
  const int64_t qi = blockIdx.x;
  float* srow = S + qi * lds;
  const int64_t row = filter_row(qi);
  if (row >= 0) {
    for (int j = f_rowptr[row] + tid; j < f_rowptr[row + 1]; j += kTopkThreads) srow[f_dst[j]] = __uint_as_float(kMaskedBits);
  }
  __syncthreads();
  const uint64_t* sel = topk_select(RowKeys{srow}, n, k);
  if (tid < k) {
    const uint64_t key = sel[tid];
    out_score[qi * k + tid] = topk_out_score(key, sigmoid);
    out_id[qi * k + tid] = key != 0ull ? int64_t(~uint32_t(key)) : -1;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// top-k new pairs of a relation (?, r, ?): candidates are the unordered pairs {s, t}, s < t, scored with
// S = sum_k z[s,k] w[r,k] z[t,k] and keyed as in the top-k above with id s*n + t.  Stage 1, one block per (query,
// tile of kPairTile s rows): 64 x 64 score tiles of the triangle t > s by register-blocked FFMA (a 4 x 4 block per
// thread, operands staged through shared memory in chunks of kPairKc features), never written out.  Scores whose
// key beats the block's running threshold are tested against row s*R + r of the symmetrised filter (binary search)
// and pushed to a shared buffer; when the buffer cannot take another tile it is cut to its top k by topk_select
// and the threshold rises to the k-th key.  Each block writes its sorted top k keys; stage 2 (one block per query)
// selects the top k of its tiles' keys and decodes them.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kPairTile = 64;
constexpr int kPairKc = 8;
constexpr int kPairTileKeys = kPairTile * kPairTile;
constexpr int kPairBuf = kPairTileKeys + 1024;      // room for one tile above a cut buffer (k <= kTopkMax < 1024)

__device__ __forceinline__ bool pair_filtered(const int32_t* __restrict__ f_rowptr, const int32_t* __restrict__ f_dst,
                                              int64_t row, int32_t t) {
  int lo = f_rowptr[row];
  const int end = f_rowptr[row + 1];
  int hi = end;
  while (lo < hi) {
    const int mid = lo + ((hi - lo) >> 1);
    if (f_dst[mid] < t) lo = mid + 1;
    else hi = mid;
  }
  return lo < end && f_dst[lo] == t;
}

struct BufKeys {
  const uint64_t* buf;
  __device__ __forceinline__ uint64_t operator()(int c) const { return buf[c]; }
};

__global__ void __launch_bounds__(kTopkThreads) rank_rel_pairs_select_kernel(
    const float* __restrict__ z, int64_t ldz, int D, const float* __restrict__ w, int32_t n_rel, int32_t n,
    const int64_t* __restrict__ rel, int64_t count, int n_tiles, const int32_t* __restrict__ f_rowptr,
    const int32_t* __restrict__ f_dst, int k, uint64_t* __restrict__ keys_out) {
  __shared__ __align__(16) float As[kPairKc][kPairTile + 4];
  __shared__ __align__(16) float Bs[kPairKc][kPairTile + 4];
  __shared__ uint64_t buf[kPairBuf];
  __shared__ int n_buf;
  __shared__ uint64_t thr_s;
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  // heavy tiles (small s) first: block b is tile b / count of query b % count
  const int tile = int(blockIdx.x / count);
  const int64_t qi = int64_t(blockIdx.x) - int64_t(tile) * count;
  const int64_t r = rel[qi];
  const float* wr = w + r * D;
  const int s0 = tile * kPairTile;
  if (tid == 0) {
    n_buf = 0;
    thr_s = 0ull;
  }
  for (int t0 = s0; t0 < n; t0 += kPairTile) {
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
    for (int kc = 0; kc < D; kc += kPairKc) {
      __syncthreads();
#pragma unroll
      for (int e = tid; e < kPairTile * kPairKc; e += kTopkThreads) {
        const int row = e / kPairKc, kk = e - row * kPairKc, f = kc + kk;
        const int s = s0 + row, t = t0 + row;
        As[kk][row] = (s < n && f < D) ? z[int64_t(s) * ldz + f] * wr[f] : 0.0f;
        Bs[kk][row] = (t < n && f < D) ? z[int64_t(t) * ldz + f] : 0.0f;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < kPairKc; ++kk) {
        const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
        const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
        const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
      }
    }
    const uint64_t thr = thr_s;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int s = s0 + ty * 4 + i;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int t = t0 + tx * 4 + j;
        if (s >= n || t >= n || t <= s) continue;
        const uint64_t key = score_key(__float_as_uint(acc[i][j]), uint32_t(s * n + t));
        if (key <= thr) continue;
        if (f_rowptr != nullptr && pair_filtered(f_rowptr, f_dst, int64_t(s) * n_rel + r, t)) continue;
        buf[atomicAdd(&n_buf, 1)] = key;
      }
    }
    __syncthreads();
    const int m = n_buf;
    if (m > kPairBuf - kPairTileKeys) {                  // block-uniform: cut to the top k, raise the threshold
      const uint64_t* sel = topk_select(BufKeys{buf}, m, k);
      if (tid < k) buf[tid] = sel[tid];
      if (tid == 0) {
        n_buf = k;
        thr_s = sel[k - 1];
      }
    }
  }
  __syncthreads();
  const uint64_t* sel = topk_select(BufKeys{buf}, n_buf, k);
  if (tid < k) keys_out[(qi * n_tiles + tile) * k + tid] = sel[tid];
}

__global__ void __launch_bounds__(kTopkThreads) rank_rel_pairs_merge_kernel(const uint64_t* __restrict__ keys,
                                                                            int m, int32_t n, int k, int sigmoid,
                                                                            float* __restrict__ out_score,
                                                                            int64_t* __restrict__ out_src,
                                                                            int64_t* __restrict__ out_dst) {
  const int tid = threadIdx.x;
  const int64_t qi = blockIdx.x;
  const uint64_t* sel = topk_select(BufKeys{keys + qi * m}, m, k);
  if (tid < k) {
    const uint64_t key = sel[tid];
    const int64_t id = key != 0ull ? int64_t(~uint32_t(key)) : -1;
    out_score[qi * k + tid] = topk_out_score(key, sigmoid);
    out_src[qi * k + tid] = id >= 0 ? id / n : -1;
    out_dst[qi * k + tid] = id >= 0 ? id % n : -1;
  }
}

}  // namespace gn

using namespace gn;

extern "C" {

size_t gn_rank_csr_workspace_bytes(int64_t n_edges, int32_t n_nodes, int32_t n_rel) {
  const size_t E = size_t(n_edges > 0 ? n_edges : 1);
  const int64_t rows = int64_t(n_nodes > 0 ? n_nodes : 1) * (n_rel > 0 ? n_rel : 1);
  return 4 * align_up(E * 4) + sort_ws_bytes(n_edges) + 2 * align_up(size_t(rows) * 4) + scan_ws_bytes(rows) + 4096;
}

int gn_rank_csr(const int64_t* src, const int64_t* dst, const int64_t* etype, int64_t n_edges, int32_t n_nodes,
                int32_t n_rel, int32_t* rowptr, int32_t* ent_dst, int32_t* ent_eid, int32_t* group_row,
                int32_t* n_groups, void* ws, size_t ws_bytes, void* stream) {
  if (n_edges < 0 || n_nodes <= 0 || n_rel <= 0 || !rowptr) return GN_ERR_ARG;
  if (n_edges > 0 && (!src || !dst || !etype || !ent_dst || !ent_eid)) return GN_ERR_ARG;
  if ((group_row == nullptr) != (n_groups == nullptr)) return GN_ERR_ARG;
  if (n_edges >= (int64_t(1) << 31) || int64_t(n_nodes) * n_rel >= (int64_t(1) << 31)) return GN_ERR_RANGE;
  cudaStream_t st = as_stream(stream);
  const int32_t n_rows = n_nodes * n_rel;
  const size_t Ea = size_t(n_edges > 0 ? n_edges : 1);
  Arena a(ws, ws_bytes);
  int32_t* key1 = a.take<int32_t>(Ea);
  int32_t* sorted1 = a.take<int32_t>(Ea);
  int32_t* perm1 = a.take<int32_t>(Ea);
  int32_t* key2 = a.take<int32_t>(Ea);
  int32_t* flag = a.take<int32_t>(size_t(n_rows));
  int32_t* pos = a.take<int32_t>(size_t(n_rows));
  if (!a.ok()) return GN_ERR_WORKSPACE;
  void* rest = a.base + a.off;
  const size_t rest_bytes = a.cap - a.off;
  int32_t* sorted2 = sorted1;                        // free once key2 is formed
  if (n_edges > 0) {
    const unsigned ge = (unsigned)ceil_div(n_edges, 256);
    GN_LAUNCH(rank_dst_keys_kernel, ge, 256, 0, st, dst, n_edges, key1);
    GN_CHECK(sort_pairs(key1, nullptr, sorted1, perm1, n_edges, bits_for(n_nodes > 1 ? n_nodes : 2), rest,
                        rest_bytes, st));
    GN_LAUNCH(rank_row_keys_kernel, ge, 256, 0, st, src, etype, (const int32_t*)perm1, n_edges, n_rel, key2);
    GN_CHECK(sort_pairs(key2, perm1, sorted2, ent_eid, n_edges, bits_for(n_rows > 1 ? n_rows : 2), rest, rest_bytes,
                        st));
    GN_LAUNCH(rank_fill_kernel, ge, 256, 0, st, dst, (const int32_t*)ent_eid, n_edges, ent_dst);
  }
  GN_CHECK(rowptr_from_sorted(sorted2, n_edges, n_rows, rowptr, st));
  if (group_row != nullptr) {
    const unsigned gr = (unsigned)ceil_div(n_rows, 256);
    GN_LAUNCH(rank_row_flags_kernel, gr, 256, 0, st, (const int32_t*)rowptr, n_rows, flag);
    GN_CHECK(exclusive_scan_i32(flag, pos, n_rows, n_groups, rest, rest_bytes, st));
    GN_LAUNCH(rank_groups_kernel, gr, 256, 0, st, (const int32_t*)rowptr, (const int32_t*)pos, n_rows, group_row);
  }
  return GN_OK;
}

int gn_rank_query_rows(const float* z, int64_t ldz, int32_t D, const float* w, int32_t n_rel, const int32_t* group_row,
                       const int64_t* node, const int64_t* rel, int64_t count, float* q, int64_t ldq, void* stream) {
  if (count < 0 || D <= 0 || n_rel <= 0 || ldq < D) return GN_ERR_ARG;
  if (count == 0) return GN_OK;
  if (!z || !w || !q || (!group_row && (!node || !rel))) return GN_ERR_ARG;
  const TailOperands ops{z, ldz, w, D, n_rel, group_row, node, rel};
  GN_LAUNCH(rank_query_rows_kernel<TailOperands>, (unsigned)ceil_div(count * D, 256), 256, 0, as_stream(stream), ops,
            D, count, q, ldq);
  return GN_OK;
}

int gn_rank_count(const float* S, int64_t lds, int32_t n_nodes, const int32_t* group_row, int32_t n_groups,
                  const int32_t* q_rowptr, const int32_t* q_dst, const int32_t* q_eid, const int32_t* f_rowptr,
                  const int32_t* f_dst, float* rank, void* stream) {
  if (n_groups < 0 || n_nodes <= 0 || lds < n_nodes) return GN_ERR_ARG;
  if (n_groups == 0) return GN_OK;
  if (!S || !group_row || !q_rowptr || !q_dst || !q_eid || !rank || (f_rowptr && !f_dst)) return GN_ERR_ARG;
  const TailRows rows{group_row, f_rowptr != nullptr};
  GN_LAUNCH(rank_count_kernel<TailRows>, (unsigned)ceil_div(n_groups, kCountWarps), kCountWarps * 32, 0,
            as_stream(stream), S, lds, n_nodes, rows, n_groups, q_rowptr, q_dst, q_eid, f_rowptr, f_dst, rank);
  return GN_OK;
}

int gn_rank_max_hits(void) { return kRankMaxHits; }

int gn_rank_metrics(const float* rank, const int32_t* rel_rowptr, const int32_t* rel_perm, int32_t n_rel,
                    const int32_t* hits_k, int32_t n_hits, double* out, void* stream) {
  if (n_rel < 0 || n_hits < 0 || n_hits > kRankMaxHits || (n_hits > 0 && !hits_k)) return GN_ERR_ARG;
  if (n_rel == 0) return GN_OK;
  if (!rel_rowptr || !out) return GN_ERR_ARG;
  HitsK hk{};
  for (int i = 0; i < n_hits; ++i) hk.k[i] = hits_k[i];
  GN_LAUNCH(rank_metrics_kernel, (unsigned)n_rel, kMetricThreads, 0, as_stream(stream), rank, rel_rowptr, rel_perm,
            n_rel, hk, n_hits, out);
  return GN_OK;
}

int gn_rank_topk(float* S, int64_t lds, int32_t n_nodes, int32_t n_rel, const int64_t* node, const int64_t* rel,
                 int64_t count, const int32_t* f_rowptr, const int32_t* f_dst, int32_t k, int sigmoid,
                 float* out_score, int64_t* out_id, void* stream) {
  if (count < 0 || n_nodes <= 0 || n_rel <= 0 || lds < n_nodes || k < 1 || k > kTopkMax) return GN_ERR_ARG;
  if (count == 0) return GN_OK;
  if (count >= (int64_t(1) << 31)) return GN_ERR_RANGE;
  if (!S || !node || !rel || !out_score || !out_id || (f_rowptr && !f_dst)) return GN_ERR_ARG;
  const TailFilterRow frow{node, rel, n_rel, f_rowptr != nullptr};
  GN_LAUNCH(rank_topk_kernel<TailFilterRow>, (unsigned)count, kTopkThreads, 0, as_stream(stream), S, lds, n_nodes,
            frow, f_rowptr, f_dst, k, sigmoid, out_score, out_id);
  return GN_OK;
}

size_t gn_rank_pair_csr_workspace_bytes(int64_t n_edges) {
  const size_t E = size_t(n_edges > 0 ? n_edges : 1);
  return 4 * align_up(E * 4) + sort_ws_bytes(n_edges) + scan_ws_bytes(n_edges) + 4096;
}

int gn_rank_pair_csr(const int64_t* src, const int64_t* dst, const int64_t* etype, int64_t n_edges, int32_t n_nodes,
                     int32_t n_rel, int32_t* rowptr, int32_t* pair_src, int32_t* pair_dst, int32_t* ent_rel,
                     int32_t* ent_eid, int32_t* n_pairs, void* ws, size_t ws_bytes, void* stream) {
  if (n_edges < 0 || n_nodes <= 0 || n_rel <= 0 || !rowptr || !n_pairs) return GN_ERR_ARG;
  if (n_edges > 0 && (!src || !dst || !etype || !pair_src || !pair_dst || !ent_rel || !ent_eid)) return GN_ERR_ARG;
  if (n_edges >= (int64_t(1) << 31)) return GN_ERR_RANGE;
  cudaStream_t st = as_stream(stream);
  if (n_edges == 0) {
    if (cudaMemsetAsync(rowptr, 0, 4, st) != cudaSuccess || cudaMemsetAsync(n_pairs, 0, 4, st) != cudaSuccess)
      return GN_ERR_CUDA;
    return GN_OK;
  }
  Arena a(ws, ws_bytes);
  int32_t* key = a.take<int32_t>(size_t(n_edges));
  int32_t* sorted = a.take<int32_t>(size_t(n_edges));
  int32_t* perm1 = a.take<int32_t>(size_t(n_edges));
  int32_t* perm2 = a.take<int32_t>(size_t(n_edges));
  if (!a.ok()) return GN_ERR_WORKSPACE;
  void* rest = a.base + a.off;
  const size_t rest_bytes = a.cap - a.off;
  const unsigned ge = (unsigned)ceil_div(n_edges, 256);
  const int node_bits = bits_for(n_nodes > 1 ? n_nodes : 2);
  // stable passes by rel, then dst, then src: entries in (src, dst, rel) order
  GN_LAUNCH(rank_gather_keys_kernel, ge, 256, 0, st, etype, (const int32_t*)nullptr, n_edges, key);
  GN_CHECK(sort_pairs(key, nullptr, sorted, perm1, n_edges, bits_for(n_rel > 1 ? n_rel : 2), rest, rest_bytes, st));
  GN_LAUNCH(rank_gather_keys_kernel, ge, 256, 0, st, dst, (const int32_t*)perm1, n_edges, key);
  GN_CHECK(sort_pairs(key, perm1, sorted, perm2, n_edges, node_bits, rest, rest_bytes, st));
  GN_LAUNCH(rank_gather_keys_kernel, ge, 256, 0, st, src, (const int32_t*)perm2, n_edges, key);
  GN_CHECK(sort_pairs(key, perm2, sorted, ent_eid, n_edges, node_bits, rest, rest_bytes, st));
  // run heads -> compacted pair rows
  int32_t* flag = key;
  int32_t* pos = sorted;
  GN_LAUNCH(rank_pair_heads_kernel, ge, 256, 0, st, src, dst, (const int32_t*)ent_eid, n_edges, flag);
  GN_CHECK(exclusive_scan_i32(flag, pos, n_edges, n_pairs, rest, rest_bytes, st));
  GN_LAUNCH(rank_pair_fill_kernel, ge, 256, 0, st, src, dst, etype, (const int32_t*)ent_eid, (const int32_t*)flag,
            (const int32_t*)pos, n_edges, rowptr, pair_src, pair_dst, ent_rel);
  return GN_OK;
}

int gn_rank_pair_lookup(const int32_t* f_src, const int32_t* f_dst, int32_t n_fpairs, const int32_t* pair_src,
                        const int32_t* pair_dst, const int64_t* src, const int64_t* dst, int64_t count, int32_t* row,
                        void* stream) {
  if (count < 0 || n_fpairs < 0) return GN_ERR_ARG;
  if (count == 0) return GN_OK;
  if (!row || (n_fpairs > 0 && (!f_src || !f_dst)) || (pair_src ? !pair_dst : (!src || !dst))) return GN_ERR_ARG;
  GN_LAUNCH(rank_pair_lookup_kernel, (unsigned)ceil_div(count, 256), 256, 0, as_stream(stream), f_src, f_dst,
            n_fpairs, pair_src, pair_dst, src, dst, count, row);
  return GN_OK;
}

int gn_rank_pair_rows(const float* z, int64_t ldz, int32_t D, const int32_t* pair_src, const int32_t* pair_dst,
                      const int64_t* src, const int64_t* dst, int64_t count, float* p, int64_t ldp, void* stream) {
  if (count < 0 || D <= 0 || ldp < D) return GN_ERR_ARG;
  if (count == 0) return GN_OK;
  if (!z || !p || (pair_src ? !pair_dst : (!src || !dst))) return GN_ERR_ARG;
  const PairOperands ops{z, ldz, pair_src, pair_dst, src, dst};
  GN_LAUNCH(rank_query_rows_kernel<PairOperands>, (unsigned)ceil_div(count * D, 256), 256, 0, as_stream(stream), ops,
            D, count, p, ldp);
  return GN_OK;
}

int gn_rank_pair_count(const float* S, int64_t lds, int32_t n_rel, int32_t n_pairs, const int32_t* q_rowptr,
                       const int32_t* q_rel, const int32_t* q_eid, const int32_t* f_row, const int32_t* f_rowptr,
                       const int32_t* f_rel, float* rank, void* stream) {
  if (n_pairs < 0 || n_rel <= 0 || lds < n_rel) return GN_ERR_ARG;
  if (n_pairs == 0) return GN_OK;
  if (!S || !q_rowptr || !q_rel || !q_eid || !rank || (f_row && (!f_rowptr || !f_rel))) return GN_ERR_ARG;
  const PairRows rows{f_row};
  GN_LAUNCH(rank_count_kernel<PairRows>, (unsigned)ceil_div(n_pairs, kCountWarps), kCountWarps * 32, 0,
            as_stream(stream), S, lds, n_rel, rows, n_pairs, q_rowptr, q_rel, q_eid, f_rowptr, f_rel, rank);
  return GN_OK;
}

int gn_rank_pair_topk(float* S, int64_t lds, int32_t n_rel, int64_t count, const int32_t* f_row,
                      const int32_t* f_rowptr, const int32_t* f_rel, int32_t k, int sigmoid, float* out_score,
                      int64_t* out_id, void* stream) {
  if (count < 0 || n_rel <= 0 || lds < n_rel || k < 1 || k > kTopkMax) return GN_ERR_ARG;
  if (count == 0) return GN_OK;
  if (count >= (int64_t(1) << 31)) return GN_ERR_RANGE;
  if (!S || !out_score || !out_id || (f_row && (!f_rowptr || !f_rel))) return GN_ERR_ARG;
  const PairFilterRow frow{f_row};
  GN_LAUNCH(rank_topk_kernel<PairFilterRow>, (unsigned)count, kTopkThreads, 0, as_stream(stream), S, lds, n_rel, frow,
            f_rowptr, f_rel, k, sigmoid, out_score, out_id);
  return GN_OK;
}

static int rel_pairs_tiles(int32_t n_nodes) { return int(ceil_div(n_nodes, kPairTile)); }

size_t gn_rank_rel_pairs_workspace_bytes(int64_t count, int32_t n_nodes, int32_t k) {
  if (count <= 0 || n_nodes <= 0 || k <= 0) return 256;
  return align_up(size_t(count) * size_t(rel_pairs_tiles(n_nodes)) * size_t(k) * 8);
}

int gn_rank_rel_pairs_select(const float* z, int64_t ldz, int32_t D, const float* w, int32_t n_rel, int32_t n_nodes,
                             const int64_t* rel, int64_t count, const int32_t* f_rowptr, const int32_t* f_dst,
                             int32_t k, void* ws, size_t ws_bytes, void* stream) {
  if (count < 0 || D <= 0 || n_rel <= 0 || n_nodes <= 0 || ldz < D || k < 1 || k > kTopkMax) return GN_ERR_ARG;
  if (int64_t(n_nodes) * n_nodes >= (int64_t(1) << 31) || int64_t(n_nodes) * n_rel >= (int64_t(1) << 31))
    return GN_ERR_RANGE;
  if (count == 0) return GN_OK;
  const int n_tiles = rel_pairs_tiles(n_nodes);
  if (count * n_tiles >= (int64_t(1) << 31)) return GN_ERR_RANGE;
  if (!z || !w || !rel || (f_rowptr && !f_dst)) return GN_ERR_ARG;
  if (!ws || ws_bytes < gn_rank_rel_pairs_workspace_bytes(count, n_nodes, k)) return GN_ERR_WORKSPACE;
  GN_LAUNCH(rank_rel_pairs_select_kernel, (unsigned)(count * n_tiles), kTopkThreads, 0, as_stream(stream), z, ldz, D,
            w, n_rel, n_nodes, rel, count, n_tiles, f_rowptr, f_dst, k, static_cast<uint64_t*>(ws));
  return GN_OK;
}

int gn_rank_rel_pairs_merge(const void* ws, size_t ws_bytes, int32_t n_nodes, int64_t count, int32_t k, int sigmoid,
                            float* out_score, int64_t* out_src, int64_t* out_dst, void* stream) {
  if (count < 0 || n_nodes <= 0 || k < 1 || k > kTopkMax) return GN_ERR_ARG;
  if (count == 0) return GN_OK;
  if (count >= (int64_t(1) << 31)) return GN_ERR_RANGE;
  if (!out_score || !out_src || !out_dst) return GN_ERR_ARG;
  if (!ws || ws_bytes < gn_rank_rel_pairs_workspace_bytes(count, n_nodes, k)) return GN_ERR_WORKSPACE;
  GN_LAUNCH(rank_rel_pairs_merge_kernel, (unsigned)count, kTopkThreads, 0, as_stream(stream),
            static_cast<const uint64_t*>(ws), rel_pairs_tiles(n_nodes) * k, n_nodes, k, sigmoid, out_score, out_src,
            out_dst);
  return GN_OK;
}

}  // extern "C"
