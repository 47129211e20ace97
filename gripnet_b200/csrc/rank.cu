// K16: filtered candidate ranking (OGB rank rule, per-relation MRR / Hits@k) and top-k link prediction of the
// DistMult decoder.  Tail queries (s, r, ?) and relation queries (s, ?, t) are one computation over different data:
// the triples are grouped by a key pair (a, b) = (s, r) or (s, t); one query row q[g] = x[a_g] .* y[b_g] per group
// (y = w for tail queries, y = z for relation queries); one row of S = Q . C^T per group against the candidate table C
// (z: every tail, w: every relation), computed by the existing dense GEMM (gn_sgemm / gn_tc_gemm); then the filtered
// ranks of the group's entries, or the top k, over that row.  This file holds what sits around the product: the
// compacted grouped structure and its lookup, the query rows, the filtered rank count, the per-relation reduction
// and the per-query top-k selection.  Pair queries (?, r, ?) score node pairs in fused tiles (below) and read the
// dense symmetrised filter view of gn_rank_csr.
#include "sortkit.cuh"

namespace gn {

constexpr int kRankMaxHits = 8;
constexpr int kTopkThreads = 256;
constexpr int kTopkMax = 256;                  // largest k: one selected key per thread of the sort
constexpr uint32_t kMaskedBits = 0xffffffffu;  // NaN payload no arithmetic produces: "filtered" in a top-k row

__global__ void rank_gather_keys_kernel(const int64_t* __restrict__ v, const int32_t* __restrict__ perm, int64_t n,
                                        int32_t* __restrict__ key) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) key[i] = int32_t(v[perm ? perm[i] : int32_t(i)]);
}

// ---------------------------------------------------------------------------------------------------------------
// dense grouped structure (the symmetrised filter view of pair queries): rows s*R + r, entries (dst, edge id) sorted
// by dst inside a row (two stable counting sorts: by dst, then by row)
// ---------------------------------------------------------------------------------------------------------------
__global__ void rank_row_keys_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ etype,
                                     const int32_t* __restrict__ perm, int64_t n, int32_t n_rel,
                                     int32_t* __restrict__ key) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t e = perm[i];
  key[i] = int32_t(src[e]) * n_rel + int32_t(etype[e]);
}

// ---------------------------------------------------------------------------------------------------------------
// compacted grouped structure of three columns (a, b, c): entries ordered by (a, b, c) with three stable counting
// sorts (by c, by b, by a), rows = the distinct key pairs (a, b) in that order, entries (c, edge id) sorted by c
// inside a row.  Rows are compacted, not a*nb + b: n^2 does not fit int32 for general n.
// ---------------------------------------------------------------------------------------------------------------
__global__ void rank_group_heads_kernel(const int64_t* __restrict__ a, const int64_t* __restrict__ b,
                                        const int32_t* __restrict__ eid, int64_t n, int32_t* __restrict__ flag) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t e = eid[i];
  flag[i] = i == 0 || a[e] != a[eid[i - 1]] || b[e] != b[eid[i - 1]] ? 1 : 0;
}

__global__ void rank_group_fill_kernel(const int64_t* __restrict__ a, const int64_t* __restrict__ b,
                                       const int64_t* __restrict__ c, const int32_t* __restrict__ eid,
                                       const int32_t* __restrict__ flag, const int32_t* __restrict__ pos, int64_t n,
                                       int32_t* __restrict__ rowptr, int32_t* __restrict__ group_a,
                                       int32_t* __restrict__ group_b, int32_t* __restrict__ ent_c) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t e = eid[i];
  ent_c[i] = int32_t(c[e]);
  if (flag[i]) {
    const int32_t p = pos[i];
    rowptr[p] = int32_t(i);
    group_a[p] = int32_t(a[e]);
    group_b[p] = int32_t(b[e]);
  }
  if (i == n - 1) rowptr[pos[i] + flag[i]] = int32_t(n);
}

// row of the key pair (a, b) in a structure by binary search over its (a, b)-sorted groups, or -1
__global__ void rank_lookup_kernel(const int32_t* __restrict__ f_a, const int32_t* __restrict__ f_b, int32_t n_f,
                                   const int32_t* __restrict__ a32, const int32_t* __restrict__ b32,
                                   const int64_t* __restrict__ a64, const int64_t* __restrict__ b64, int64_t count,
                                   int32_t* __restrict__ row) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const int32_t s = a32 ? a32[i] : int32_t(a64[i]);
  const int32_t t = a32 ? b32[i] : int32_t(b64[i]);
  int lo = 0, hi = n_f;
  while (lo < hi) {
    const int mid = lo + ((hi - lo) >> 1);
    const int32_t ms = f_a[mid];
    if (ms < s || (ms == s && f_b[mid] < t)) lo = mid + 1;
    else hi = mid;
  }
  row[i] = (lo < n_f && f_a[lo] == s && f_b[lo] == t) ? lo : -1;
}

// ---------------------------------------------------------------------------------------------------------------
// query rows q[i, :] = x[a_i] .* y[b_i], (a_i, b_i) from a grouped structure's key columns (int32) or from two index
// lists (int64)
// ---------------------------------------------------------------------------------------------------------------
__global__ void rank_rows_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ y, int64_t ldy,
                                 int D, const int32_t* __restrict__ a32, const int32_t* __restrict__ b32,
                                 const int64_t* __restrict__ a64, const int64_t* __restrict__ b64, int64_t count,
                                 float* __restrict__ q, int64_t ldq) {
  const int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= count * D) return;
  const int64_t i = t / D;
  const int f = int(t - i * D);
  const int64_t a = a32 ? int64_t(a32[i]) : a64[i];
  const int64_t b = a32 ? int64_t(b32[i]) : b64[i];
  q[i * ldq + f] = x[a * ldx + f] * y[b * ldy + f];
}

// ---------------------------------------------------------------------------------------------------------------
// filtered rank: one warp per group g (row g of S), the group's entries (target candidates) in turn.  opt / pess
// count the candidates c != t above / at-or-above S(t) over the whole row, then the distinct filtered candidates
// other than t that met the same comparisons are taken back out.  S(t) is read from the same row as every S(c).
// f_row[g] is the group's row in the filter (gn_rank_lookup; -1: the filter holds no triple of its key pair).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kCountWarps = 8;

__global__ void __launch_bounds__(kCountWarps * 32) rank_count_kernel(
    const float* __restrict__ S, int64_t lds, int32_t n, int32_t n_groups, const int32_t* __restrict__ q_rowptr,
    const int32_t* __restrict__ q_c, const int32_t* __restrict__ q_eid, const int32_t* __restrict__ f_row,
    const int32_t* __restrict__ f_rowptr, const int32_t* __restrict__ f_c, float* __restrict__ rank) {
  const int lane = threadIdx.x & 31;
  const int g = blockIdx.x * kCountWarps + (threadIdx.x >> 5);
  if (g >= n_groups) return;
  const int32_t frow = f_row ? f_row[g] : -1;
  const float* srow = S + int64_t(g) * lds;
  const int f0 = frow >= 0 ? f_rowptr[frow] : 0, f1 = frow >= 0 ? f_rowptr[frow + 1] : 0;
  for (int j = q_rowptr[g]; j < q_rowptr[g + 1]; ++j) {
    const int t = q_c[j];
    const float st = srow[t];
    int opt = 0, pess = 0;
    for (int c = lane; c < n; c += 32) {
      const float v = srow[c];
      opt += (c != t) & (v > st);
      pess += (c != t) & (v >= st);
    }
    for (int k = f0 + lane; k < f1; k += 32) {
      const int c = f_c[k];
      if (c == t || (k > f0 && f_c[k - 1] == c)) continue;   // the target itself; duplicates count once
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
// order-preserving bits of a float: a larger unsigned value is a larger score
__device__ __forceinline__ uint32_t order_bits(uint32_t b) { return (b & 0x80000000u) ? ~b : (b | 0x80000000u); }

__device__ __forceinline__ uint64_t score_key(uint32_t b, uint32_t id) {
  return (uint64_t(order_bits(b)) << 32) | uint64_t(~id);
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

struct RowKeys {
  const float* srow;
  __device__ __forceinline__ uint64_t operator()(int c) const { return topk_key(srow, c); }
};

// f_row[qi]: the filter row of query row qi (gn_rank_lookup; -1: none), or f_row == nullptr: no filter
__global__ void __launch_bounds__(kTopkThreads) rank_topk_kernel(float* __restrict__ S, int64_t lds, int32_t n,
                                                                 const int32_t* __restrict__ f_row,
                                                                 const int32_t* __restrict__ f_rowptr,
                                                                 const int32_t* __restrict__ f_c, int k, int sigmoid,
                                                                 float* __restrict__ out_score,
                                                                 int64_t* __restrict__ out_id) {
  const int tid = threadIdx.x;
  const int64_t qi = blockIdx.x;
  float* srow = S + qi * lds;
  const int32_t row = f_row ? f_row[qi] : -1;
  if (row >= 0) {
    for (int j = f_rowptr[row] + tid; j < f_rowptr[row + 1]; j += kTopkThreads) srow[f_c[j]] = __uint_as_float(kMaskedBits);
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

// The score tiles of one 64-row tile of s, s0 = 64 * tile: for t0 = s0, s0 + 64, ... < n, thread (ty, tx) holds
// acc[i][j] = S(s0 + 4 ty + i, t0 + 4 tx + j) and the block calls epi(t0, acc).  Every score is the one per-pair
// sequence q_f = z[s,f] * w[r,f] (rounded), acc = fmaf(q_f, z[t,f], acc) for f = 0 .. D-1, then zero padding to a
// multiple of kPairKc (which can only turn -0 into +0); rank_rel_pairs_query_kernel restates it per pair.
template <class Epilogue>
__device__ __forceinline__ void pair_tiles(const float* __restrict__ z, int64_t ldz, int D,
                                           const float* __restrict__ wr, int32_t n, int s0, Epilogue&& epi) {
  __shared__ __align__(16) float As[kPairKc][kPairTile + 4];
  __shared__ __align__(16) float Bs[kPairKc][kPairTile + 4];
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
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
    epi(t0, acc);
  }
}

__global__ void __launch_bounds__(kTopkThreads) rank_rel_pairs_select_kernel(
    const float* __restrict__ z, int64_t ldz, int D, const float* __restrict__ w, int32_t n_rel, int32_t n,
    const int64_t* __restrict__ rel, int64_t count, int n_tiles, const int32_t* __restrict__ f_rowptr,
    const int32_t* __restrict__ f_dst, int k, uint64_t* __restrict__ keys_out) {
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
  pair_tiles(z, ldz, D, wr, n, s0, [&](int t0, const float (&acc)[4][4]) {
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
  });
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

// ---------------------------------------------------------------------------------------------------------------
// filtered pair ranks (?, r, ?): every query triple (s, r, t), s != t, is ranked against the unordered pairs
// {a, b}, a < b, of its relation.  The query triples are grouped by relation (gn_index_prep order i, edge
// rel_perm[i]); per call their scores are computed with the tiles' per-pair sequence and sorted ascending inside
// their relation.  The count kernel walks the same score tiles as rank_rel_pairs_select_kernel and, for a
// candidate at or above the relation's smallest query score, finds lb = #{query scores < S} and whether S ties
// query score lb; an unfiltered candidate adds 1 to gt[lb] (lb > 0) and to eq[lb] (tie).  A query at tie block
// [L, U) of the sorted scores then has opt = sum_{j >= U} gt[j] and pess = opt + eq[L] - [its own pair counted].
// Relation r's counters are the m_r + 1 slots from rel_rowptr[r] + r of gt and of eq.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kRankStage = 3072;     // a relation of at most kRankStage - 1 query triples is staged in shared memory
constexpr int kFinishThreads = 256;

__device__ __forceinline__ void canonical_pair(const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                               int32_t e, int64_t& a, int64_t& b) {
  const int64_t s = src[e], t = dst[e];
  a = s < t ? s : t;
  b = s < t ? t : s;
}

// whether the pair of query i is in the symmetrised filter (construction time)
__global__ void rank_rel_pairs_targets_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                              const int64_t* __restrict__ etype, const int32_t* __restrict__ perm,
                                              int32_t count, int32_t n_rel, const int32_t* __restrict__ f_rowptr,
                                              const int32_t* __restrict__ f_dst, int32_t* __restrict__ filtered) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const int32_t e = perm[i];
  int64_t a, b;
  canonical_pair(src, dst, e, a, b);
  filtered[i] = pair_filtered(f_rowptr, f_dst, a * n_rel + etype[e], int32_t(b)) ? 1 : 0;
}

// score of query i in the tiles' per-pair sequence, its order-preserving key and its relation
__global__ void rank_rel_pairs_query_kernel(const float* __restrict__ z, int64_t ldz, int D,
                                            const float* __restrict__ w, const int64_t* __restrict__ src,
                                            const int64_t* __restrict__ dst, const int64_t* __restrict__ etype,
                                            const int32_t* __restrict__ perm, int32_t count,
                                            float* __restrict__ score, int32_t* __restrict__ key,
                                            int32_t* __restrict__ qrel) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const int32_t e = perm[i];
  int64_t a, b;
  canonical_pair(src, dst, e, a, b);
  const int64_t r = etype[e];
  const float *za = z + a * ldz, *zb = z + b * ldz, *wr = w + r * D;
  float acc = 0.0f;
  for (int f = 0; f < D; ++f) acc = fmaf(__fmul_rn(za[f], wr[f]), zb[f], acc);
  score[i] = acc;
  key[i] = int32_t(order_bits(__float_as_uint(acc)));
  qrel[i] = int32_t(r);
}

template <class T>
__global__ void rank_gather_kernel(const T* __restrict__ v, const int32_t* __restrict__ idx, int32_t count,
                                   T* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) out[i] = v[idx[i]];
}

__global__ void __launch_bounds__(kTopkThreads) rank_rel_pairs_count_kernel(
    const float* __restrict__ z, int64_t ldz, int D, const float* __restrict__ w, int32_t n_rel, int32_t n,
    const int32_t* __restrict__ group_rel, int32_t n_groups, const int32_t* __restrict__ rel_rowptr,
    const float* __restrict__ sorted, const int32_t* __restrict__ f_rowptr, const int32_t* __restrict__ f_dst,
    int32_t* __restrict__ gt, int32_t* __restrict__ eq) {
  __shared__ float ss_s[kRankStage];
  __shared__ int gt_s[kRankStage], eq_s[kRankStage];
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  // tile order of rank_rel_pairs_select_kernel: block b is tile b / n_groups of query relation b % n_groups
  const int tile = int(blockIdx.x / n_groups);
  const int32_t r = group_rel[blockIdx.x - tile * n_groups];
  const int b = rel_rowptr[r], m = rel_rowptr[r + 1] - b;
  const int64_t c0 = int64_t(b) + r;
  const bool staged = m < kRankStage;
  const float* ss = staged ? ss_s : sorted + b;
  int* gtp = staged ? gt_s : gt + c0;
  int* eqp = staged ? eq_s : eq + c0;
  if (staged) {
    for (int j = tid; j <= m; j += kTopkThreads) {
      if (j < m) ss_s[j] = sorted[b + j];
      gt_s[j] = 0;
      eq_s[j] = 0;
    }
  }
  __syncthreads();
  const float smin = ss[0];
  const int s0 = tile * kPairTile;
  pair_tiles(z, ldz, D, w + int64_t(r) * D, n, s0, [&](int t0, const float (&acc)[4][4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int s = s0 + ty * 4 + i;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int t = t0 + tx * 4 + j;
        const float v = acc[i][j];
        if (s >= n || t >= n || t <= s || !(v >= smin)) continue;   // most candidates: below every query score
        int lo = 0, hi = m;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (ss[mid] < v) lo = mid + 1;
          else hi = mid;
        }
        const bool tie = lo < m && ss[lo] == v;
        if (f_rowptr != nullptr && pair_filtered(f_rowptr, f_dst, int64_t(s) * n_rel + r, t)) continue;
        if (lo > 0) atomicAdd(&gtp[lo], 1);
        if (tie) atomicAdd(&eqp[lo], 1);
      }
    }
  });
  if (staged) {
    __syncthreads();
    for (int j = tid; j <= m; j += kTopkThreads) {
      if (gt_s[j] != 0) atomicAdd(&gt[c0 + j], gt_s[j]);
      if (eq_s[j] != 0) atomicAdd(&eq[c0 + j], eq_s[j]);
    }
  }
}

// one block per relation r < n_rel: suffix sums of gt in place, then the rank of each query; block n_rel writes NaN
// for the self-pair triples (key n_rel of the relation index)
__global__ void __launch_bounds__(kFinishThreads) rank_rel_pairs_finish_kernel(
    const int32_t* __restrict__ rel_rowptr, const int32_t* __restrict__ rel_perm, int32_t n_rel,
    const float* __restrict__ score, const float* __restrict__ sorted, int32_t* __restrict__ gt,
    const int32_t* __restrict__ eq, const int32_t* __restrict__ t_filtered, float* __restrict__ rank) {
  __shared__ int warp_sum[kFinishThreads / 32];
  const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = rel_rowptr[r], e = rel_rowptr[r + 1], m = e - b;
  if (r == n_rel) {
    for (int i = b + tid; i < e; i += kFinishThreads) rank[rel_perm[i]] = __uint_as_float(0x7fc00000u);
    return;
  }
  if (m == 0) return;
  int* g = gt + b + r;
  const int* q = eq + b + r;
  // suffix sums over the m + 1 slots, chunks of kFinishThreads from the top (thread 0 takes the highest slot)
  int carry = 0;
  for (int top = m; top >= 0; top -= kFinishThreads) {
    const int j = top - tid;
    int incl = j >= 0 ? g[j] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(kFull, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    int off = carry, total = carry;
#pragma unroll
    for (int w2 = 0; w2 < kFinishThreads / 32; ++w2) {
      off += w2 < warp ? warp_sum[w2] : 0;
      total += warp_sum[w2];
    }
    if (j >= 0) g[j] = incl + off;
    carry = total;
    __syncthreads();
  }
  const float* ss = sorted + b;
  for (int i = b + tid; i < e; i += kFinishThreads) {
    const float x = score[i];
    int lo = 0, hi = m;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (ss[mid] < x) lo = mid + 1;
      else hi = mid;
    }
    const int L = lo;
    hi = m;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (ss[mid] <= x) lo = mid + 1;
      else hi = mid;
    }
    const int opt = g[lo];                                   // lo = U <= m
    const int pess = opt + q[L] - ((t_filtered != nullptr && t_filtered[i]) ? 0 : 1);
    rank[rel_perm[i]] = 1.0f + 0.5f * float(opt + pess);
  }
}

}  // namespace gn

using namespace gn;

extern "C" {

size_t gn_rank_csr_workspace_bytes(int64_t n_edges) {
  const size_t E = size_t(n_edges > 0 ? n_edges : 1);
  return 4 * align_up(E * 4) + sort_ws_bytes(n_edges) + 4096;
}

int gn_rank_csr(const int64_t* src, const int64_t* dst, const int64_t* etype, int64_t n_edges, int32_t n_nodes,
                int32_t n_rel, int32_t* rowptr, int32_t* ent_dst, int32_t* ent_eid, void* ws, size_t ws_bytes,
                void* stream) {
  if (n_edges < 0 || n_nodes <= 0 || n_rel <= 0 || !rowptr) return GN_ERR_ARG;
  if (n_edges > 0 && (!src || !dst || !etype || !ent_dst || !ent_eid)) return GN_ERR_ARG;
  if (n_edges >= (int64_t(1) << 31) || int64_t(n_nodes) * n_rel >= (int64_t(1) << 31)) return GN_ERR_RANGE;
  cudaStream_t st = as_stream(stream);
  const int32_t n_rows = n_nodes * n_rel;
  const size_t Ea = size_t(n_edges > 0 ? n_edges : 1);
  Arena a(ws, ws_bytes);
  int32_t* key1 = a.take<int32_t>(Ea);
  int32_t* sorted1 = a.take<int32_t>(Ea);
  int32_t* perm1 = a.take<int32_t>(Ea);
  int32_t* key2 = a.take<int32_t>(Ea);
  if (!a.ok()) return GN_ERR_WORKSPACE;
  void* rest = a.base + a.off;
  const size_t rest_bytes = a.cap - a.off;
  int32_t* sorted2 = sorted1;                        // free once key2 is formed
  if (n_edges > 0) {
    const unsigned ge = (unsigned)ceil_div(n_edges, 256);
    GN_LAUNCH(rank_gather_keys_kernel, ge, 256, 0, st, dst, (const int32_t*)nullptr, n_edges, key1);
    GN_CHECK(sort_pairs(key1, nullptr, sorted1, perm1, n_edges, bits_for(n_nodes > 1 ? n_nodes : 2), rest,
                        rest_bytes, st));
    GN_LAUNCH(rank_row_keys_kernel, ge, 256, 0, st, src, etype, (const int32_t*)perm1, n_edges, n_rel, key2);
    GN_CHECK(sort_pairs(key2, perm1, sorted2, ent_eid, n_edges, bits_for(n_rows > 1 ? n_rows : 2), rest, rest_bytes,
                        st));
    GN_LAUNCH(rank_gather_keys_kernel, ge, 256, 0, st, dst, (const int32_t*)ent_eid, n_edges, ent_dst);
  }
  GN_CHECK(rowptr_from_sorted(sorted2, n_edges, n_rows, rowptr, st));
  return GN_OK;
}

size_t gn_rank_group_workspace_bytes(int64_t n_edges) {
  const size_t E = size_t(n_edges > 0 ? n_edges : 1);
  return 4 * align_up(E * 4) + sort_ws_bytes(n_edges) + scan_ws_bytes(n_edges) + 4096;
}

int gn_rank_group(const int64_t* a, const int64_t* b, const int64_t* c, int64_t n_edges, int32_t na, int32_t nb,
                  int32_t nc, int32_t* rowptr, int32_t* group_a, int32_t* group_b, int32_t* ent_c, int32_t* ent_eid,
                  int32_t* n_groups, void* ws, size_t ws_bytes, void* stream) {
  if (n_edges < 0 || na <= 0 || nb <= 0 || nc <= 0 || !rowptr || !n_groups) return GN_ERR_ARG;
  if (n_edges > 0 && (!a || !b || !c || !group_a || !group_b || !ent_c || !ent_eid)) return GN_ERR_ARG;
  if (n_edges >= (int64_t(1) << 31)) return GN_ERR_RANGE;
  cudaStream_t st = as_stream(stream);
  if (n_edges == 0) {
    if (cudaMemsetAsync(rowptr, 0, 4, st) != cudaSuccess || cudaMemsetAsync(n_groups, 0, 4, st) != cudaSuccess)
      return GN_ERR_CUDA;
    return GN_OK;
  }
  Arena ar(ws, ws_bytes);
  int32_t* key = ar.take<int32_t>(size_t(n_edges));
  int32_t* sorted = ar.take<int32_t>(size_t(n_edges));
  int32_t* perm1 = ar.take<int32_t>(size_t(n_edges));
  int32_t* perm2 = ar.take<int32_t>(size_t(n_edges));
  if (!ar.ok()) return GN_ERR_WORKSPACE;
  void* rest = ar.base + ar.off;
  const size_t rest_bytes = ar.cap - ar.off;
  const unsigned ge = (unsigned)ceil_div(n_edges, 256);
  // stable passes by c, then b, then a: entries in (a, b, c) order
  GN_LAUNCH(rank_gather_keys_kernel, ge, 256, 0, st, c, (const int32_t*)nullptr, n_edges, key);
  GN_CHECK(sort_pairs(key, nullptr, sorted, perm1, n_edges, bits_for(nc > 1 ? nc : 2), rest, rest_bytes, st));
  GN_LAUNCH(rank_gather_keys_kernel, ge, 256, 0, st, b, (const int32_t*)perm1, n_edges, key);
  GN_CHECK(sort_pairs(key, perm1, sorted, perm2, n_edges, bits_for(nb > 1 ? nb : 2), rest, rest_bytes, st));
  GN_LAUNCH(rank_gather_keys_kernel, ge, 256, 0, st, a, (const int32_t*)perm2, n_edges, key);
  GN_CHECK(sort_pairs(key, perm2, sorted, ent_eid, n_edges, bits_for(na > 1 ? na : 2), rest, rest_bytes, st));
  // run heads -> compacted group rows
  int32_t* flag = key;
  int32_t* pos = sorted;
  GN_LAUNCH(rank_group_heads_kernel, ge, 256, 0, st, a, b, (const int32_t*)ent_eid, n_edges, flag);
  GN_CHECK(exclusive_scan_i32(flag, pos, n_edges, n_groups, rest, rest_bytes, st));
  GN_LAUNCH(rank_group_fill_kernel, ge, 256, 0, st, a, b, c, (const int32_t*)ent_eid, (const int32_t*)flag,
            (const int32_t*)pos, n_edges, rowptr, group_a, group_b, ent_c);
  return GN_OK;
}

int gn_rank_lookup(const int32_t* f_a, const int32_t* f_b, int32_t n_f, const int32_t* a32, const int32_t* b32,
                   const int64_t* a64, const int64_t* b64, int64_t count, int32_t* row, void* stream) {
  if (count < 0 || n_f < 0) return GN_ERR_ARG;
  if (count == 0) return GN_OK;
  if (!row || (n_f > 0 && (!f_a || !f_b)) || (a32 ? !b32 : (!a64 || !b64))) return GN_ERR_ARG;
  GN_LAUNCH(rank_lookup_kernel, (unsigned)ceil_div(count, 256), 256, 0, as_stream(stream), f_a, f_b, n_f, a32, b32,
            a64, b64, count, row);
  return GN_OK;
}

int gn_rank_rows(const float* x, int64_t ldx, const float* y, int64_t ldy, int32_t D, const int32_t* a32,
                 const int32_t* b32, const int64_t* a64, const int64_t* b64, int64_t count, float* q, int64_t ldq,
                 void* stream) {
  if (count < 0 || D <= 0 || ldq < D) return GN_ERR_ARG;
  if (count == 0) return GN_OK;
  if (!x || !y || !q || (a32 ? !b32 : (!a64 || !b64))) return GN_ERR_ARG;
  GN_LAUNCH(rank_rows_kernel, (unsigned)ceil_div(count * D, 256), 256, 0, as_stream(stream), x, ldx, y, ldy, D, a32,
            b32, a64, b64, count, q, ldq);
  return GN_OK;
}

int gn_rank_count(const float* S, int64_t lds, int32_t n_cand, int32_t n_groups, const int32_t* q_rowptr,
                  const int32_t* q_c, const int32_t* q_eid, const int32_t* f_row, const int32_t* f_rowptr,
                  const int32_t* f_c, float* rank, void* stream) {
  if (n_groups < 0 || n_cand <= 0 || lds < n_cand) return GN_ERR_ARG;
  if (n_groups == 0) return GN_OK;
  if (!S || !q_rowptr || !q_c || !q_eid || !rank || (f_row && (!f_rowptr || !f_c))) return GN_ERR_ARG;
  GN_LAUNCH(rank_count_kernel, (unsigned)ceil_div(n_groups, kCountWarps), kCountWarps * 32, 0, as_stream(stream), S,
            lds, n_cand, n_groups, q_rowptr, q_c, q_eid, f_row, f_rowptr, f_c, rank);
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

int gn_rank_topk(float* S, int64_t lds, int32_t n_cand, int64_t count, const int32_t* f_row, const int32_t* f_rowptr,
                 const int32_t* f_c, int32_t k, int sigmoid, float* out_score, int64_t* out_id, void* stream) {
  if (count < 0 || n_cand <= 0 || lds < n_cand || k < 1 || k > kTopkMax) return GN_ERR_ARG;
  if (count == 0) return GN_OK;
  if (count >= (int64_t(1) << 31)) return GN_ERR_RANGE;
  if (!S || !out_score || !out_id || (f_row && (!f_rowptr || !f_c))) return GN_ERR_ARG;
  GN_LAUNCH(rank_topk_kernel, (unsigned)count, kTopkThreads, 0, as_stream(stream), S, lds, n_cand, f_row, f_rowptr,
            f_c, k, sigmoid, out_score, out_id);
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

// the per-call workspace of the pair ranks: what gn_rank_rel_pairs_finish reads first, the sort scratch after it
struct RelPairsRankWs {
  float* score;       // [Q] query scores, grouped order
  float* sorted;      // [Q] ascending inside each relation
  int32_t* cnt;       // [2 (Q + R)] gt, then eq
  int32_t *key, *qrel, *skey, *idx1, *idx2;
  void* rest;
  size_t rest_bytes;
  bool ok;
  RelPairsRankWs(void* ws, size_t ws_bytes, int64_t nq, int32_t n_rel) {
    Arena a(ws, ws_bytes);
    const size_t q = size_t(nq > 0 ? nq : 1);
    score = a.take<float>(q);
    sorted = a.take<float>(q);
    cnt = a.take<int32_t>(2 * (size_t(nq) + size_t(n_rel)));
    key = a.take<int32_t>(q);
    qrel = a.take<int32_t>(q);
    skey = a.take<int32_t>(q);
    idx1 = a.take<int32_t>(q);
    idx2 = a.take<int32_t>(q);
    ok = a.ok();
    rest = ok ? a.base + a.off : nullptr;
    rest_bytes = ok ? a.cap - a.off : 0;
  }
};

static bool rel_pairs_rank_args(int32_t n_rel, int64_t n_queries) {
  return n_rel > 0 && n_queries >= 0 && n_queries < (int64_t(1) << 31) - n_rel;
}

size_t gn_rank_rel_pairs_rank_workspace_bytes(int64_t n_queries, int32_t n_rel) {
  const size_t q = align_up(size_t(n_queries > 0 ? n_queries : 1) * 4);
  const size_t r = size_t(n_rel > 0 ? n_rel : 1);
  return 7 * q + align_up(2 * (size_t(n_queries > 0 ? n_queries : 0) + r) * 4) + sort_ws_bytes(n_queries) + 4096;
}

int gn_rank_rel_pairs_targets(const int64_t* src, const int64_t* dst, const int64_t* etype, const int32_t* rel_perm,
                              int64_t n_queries, int32_t n_rel, const int32_t* f_rowptr, const int32_t* f_dst,
                              int32_t* filtered, void* stream) {
  if (!rel_pairs_rank_args(n_rel, n_queries)) return GN_ERR_ARG;
  if (n_queries == 0) return GN_OK;
  if (!src || !dst || !etype || !rel_perm || !f_rowptr || !f_dst || !filtered) return GN_ERR_ARG;
  GN_LAUNCH(rank_rel_pairs_targets_kernel, (unsigned)ceil_div(n_queries, 256), 256, 0, as_stream(stream), src, dst,
            etype, rel_perm, int32_t(n_queries), n_rel, f_rowptr, f_dst, filtered);
  return GN_OK;
}

int gn_rank_rel_pairs_count(const float* z, int64_t ldz, int32_t D, const float* w, int32_t n_rel, int32_t n_nodes,
                            const int64_t* src, const int64_t* dst, const int64_t* etype, const int32_t* rel_rowptr,
                            const int32_t* rel_perm, int64_t n_queries, const int32_t* group_rel, int32_t n_groups,
                            const int32_t* f_rowptr, const int32_t* f_dst, void* ws, size_t ws_bytes, void* stream) {
  if (D <= 0 || n_nodes <= 0 || ldz < D || n_groups < 0 || !rel_pairs_rank_args(n_rel, n_queries)) return GN_ERR_ARG;
  if (int64_t(n_nodes) * n_nodes >= (int64_t(1) << 31) || int64_t(n_nodes) * n_rel >= (int64_t(1) << 31))
    return GN_ERR_RANGE;
  if (n_queries == 0 || n_groups == 0) return GN_OK;
  const int n_tiles = rel_pairs_tiles(n_nodes);
  if (int64_t(n_groups) * n_tiles >= (int64_t(1) << 31)) return GN_ERR_RANGE;
  if (!z || !w || !src || !dst || !etype || !rel_rowptr || !rel_perm || !group_rel || (f_rowptr && !f_dst))
    return GN_ERR_ARG;
  const RelPairsRankWs p(ws, ws_bytes, n_queries, n_rel);
  if (!p.ok) return GN_ERR_WORKSPACE;
  cudaStream_t st = as_stream(stream);
  const int32_t nq = int32_t(n_queries);
  const unsigned gq = (unsigned)ceil_div(nq, 256);
  GN_LAUNCH(rank_rel_pairs_query_kernel, gq, 256, 0, st, z, ldz, D, w, src, dst, etype, rel_perm, nq, p.score, p.key,
            p.qrel);
  // stable: by score key, then by relation -> ascending scores inside each relation's range of the grouped order
  GN_CHECK(sort_pairs(p.key, nullptr, p.skey, p.idx1, nq, 32, p.rest, p.rest_bytes, st));
  GN_LAUNCH(rank_gather_kernel<int32_t>, gq, 256, 0, st, (const int32_t*)p.qrel, (const int32_t*)p.idx1, nq, p.key);
  GN_CHECK(sort_pairs(p.key, p.idx1, p.skey, p.idx2, nq, bits_for(n_rel > 1 ? n_rel : 2), p.rest, p.rest_bytes, st));
  GN_LAUNCH(rank_gather_kernel<float>, gq, 256, 0, st, (const float*)p.score, (const int32_t*)p.idx2, nq, p.sorted);
  if (cudaMemsetAsync(p.cnt, 0, 2 * (size_t(nq) + size_t(n_rel)) * 4, st) != cudaSuccess) return GN_ERR_CUDA;
  GN_LAUNCH(rank_rel_pairs_count_kernel, (unsigned)(int64_t(n_groups) * n_tiles), kTopkThreads, 0, st, z, ldz, D, w,
            n_rel, n_nodes, group_rel, n_groups, rel_rowptr, (const float*)p.sorted, f_rowptr, f_dst, p.cnt,
            p.cnt + nq + n_rel);
  return GN_OK;
}

int gn_rank_rel_pairs_finish(void* ws, size_t ws_bytes, int32_t n_rel, const int32_t* rel_rowptr,
                             const int32_t* rel_perm, int64_t n_queries, const int32_t* target_filtered, float* rank,
                             void* stream) {
  if (!rel_pairs_rank_args(n_rel, n_queries) || !rel_rowptr || !rel_perm || !rank) return GN_ERR_ARG;
  const RelPairsRankWs p(ws, ws_bytes, n_queries, n_rel);
  if (!p.ok) return GN_ERR_WORKSPACE;
  GN_LAUNCH(rank_rel_pairs_finish_kernel, (unsigned)n_rel + 1, kFinishThreads, 0, as_stream(stream), rel_rowptr,
            rel_perm, n_rel, (const float*)p.score, (const float*)p.sorted, p.cnt, (const int32_t*)(p.cnt + n_queries + n_rel),
            target_filtered, rank);
  return GN_OK;
}

}  // extern "C"
