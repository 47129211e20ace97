// K9/K10/K11: DistMult link decoder (fused gather-multiply-reduce), its
// deterministic backward, and the softmax pieces of the multi-class decoder.
// Reference arithmetic restated: gripnet/decoder.py:19-23, :38-45.
#include "rowsplit.cuh"
#include "sortkit.cuh"

namespace gn {

constexpr int kMaxNV = 8;  // vectors per feature lane

// ---------------------------------------------------------------------------
// forward: one edge per group of LPE lanes; nothing of size [E,D] is materialised
// ---------------------------------------------------------------------------
template <int LPE, int VEC>
__global__ void __launch_bounds__(256) distmult_fwd_kernel(const float* __restrict__ z, int64_t ldz, int D,
                                                           const float* __restrict__ w,
                                                           const int64_t* __restrict__ src,
                                                           const int64_t* __restrict__ dst,
                                                           const int64_t* __restrict__ etype, int64_t n_edges,
                                                           int sigmoid, float* __restrict__ out) {
  constexpr int EPI = 32 / LPE;
  const int lane = threadIdx.x & 31;
  const int slot = lane / LPE, fl = lane % LPE;
  const int64_t warp = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = (int64_t(gridDim.x) * blockDim.x) >> 5;
  for (int64_t e0 = warp * EPI; e0 < n_edges; e0 += n_warps * EPI) {
    const int64_t e = e0 + slot;
    float s = 0.f;
    if (e < n_edges) {
      const float* za = z + src[e] * ldz;
      const float* zb = z + dst[e] * ldz;
      const float* wr = w + etype[e] * int64_t(D);
      for (int f = fl * VEC; f < D; f += LPE * VEC) {
        const Vec<VEC> a = load_vec<VEC>(za + f), b = load_vec<VEC>(zb + f), c = load_vec<VEC>(wr + f);
#pragma unroll
        for (int i = 0; i < VEC; ++i) s = fmaf(a.v[i] * b.v[i], c.v[i], s);
      }
    }
#pragma unroll
    for (int o = LPE / 2; o > 0; o >>= 1) s += __shfl_xor_sync(kFull, s, o);
    if (e < n_edges && fl == 0) out[e] = sigmoid ? 1.0f / (1.0f + expf(-s)) : s;
  }
}

// ---------------------------------------------------------------------------
// forward, batch form (D % 4 == 0, D <= 128): a warp takes 32 consecutive edges per step of its loop.
//  * the three index arrays are read ONCE per edge with coalesced loads (lane l = edge l of the batch) and handed to
//    the feature lanes with shuffles — the per-edge form above reads them once per feature lane and spends most of
//    its issue slots on index / address arithmetic (ncu r02_v17: 28 warp instructions per edge, 7 needed);
//  * 8 feature lanes per edge: one 128-byte piece of an embedding row per quarter-warp, the unit the L1 serves per
//    wavefront (4 lanes x 16 B touch two rows per wavefront and move 64 B);
//  * edge lists are relation-major in every pose pipeline (GripNet-pose.py:59-70 builds them from `range_list`), so
//    the 32 edges of a batch normally share one relation: its weight row then lives in registers for the batch and
//    one third of the row gathers disappears.  Mixed batches fetch the row per edge.
// Summation order per edge: feature lane fl adds its vectors v = 0..NV-1 in order, then the fixed 8-lane tree.
// ---------------------------------------------------------------------------
// row `i` of a table whose rows are `ld_bytes` apart, as ONE 32x32 -> 64-bit multiply-add (IMAD.WIDE.U32)
__device__ __forceinline__ const float4* row_ptr(const float4* base, int i, unsigned ld_bytes) {
  return reinterpret_cast<const float4*>(reinterpret_cast<const char*>(base) +
                                         static_cast<unsigned long long>(static_cast<unsigned>(i)) * ld_bytes);
}

template <int NV>
__global__ void __launch_bounds__(256, NV <= 3 ? 4 : 3) distmult_fwd_batch_kernel(const float* __restrict__ z, int64_t ldz, int D,
                                                                    const float* __restrict__ w,
                                                                    const int64_t* __restrict__ src,
                                                                    const int64_t* __restrict__ dst,
                                                                    const int64_t* __restrict__ etype,
                                                                    int64_t n_edges, int sigmoid,
                                                                    float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int slot = lane >> 3, fl = lane & 7;
  const int D4 = D >> 2;
  const unsigned ldb = unsigned(ldz) * 4u, wdb = unsigned(D) * 4u;
  const float4* __restrict__ z4 = reinterpret_cast<const float4*>(z) + fl;
  const float4* __restrict__ w4 = reinterpret_cast<const float4*>(w) + fl;
  bool ok[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) ok[v] = (v * 8 + fl) < D4;
  const int64_t warp = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = (int64_t(gridDim.x) * blockDim.x) >> 5;
  const int64_t n_batches = (n_edges + 31) >> 5;
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  // the indices of this warp's NEXT batch are fetched while the rows of the current one are in flight
  int s_nxt = 0, d_nxt = 0, r_nxt = 0;
  if (warp < n_batches && (warp << 5) + lane < n_edges) {
    s_nxt = int(__ldg(src + (warp << 5) + lane));
    d_nxt = int(__ldg(dst + (warp << 5) + lane));
    r_nxt = int(__ldg(etype + (warp << 5) + lane));
  }
  for (int64_t b = warp; b < n_batches; b += n_warps) {
    const int64_t e = (b << 5) + lane;
    const bool live = e < n_edges;
    const int s = s_nxt, d = d_nxt;
    const int r_first = __shfl_sync(kFull, r_nxt, 0);          // lane 0 of a batch is always a live edge
    const int r = live ? r_nxt : r_first;
    s_nxt = d_nxt = r_nxt = 0;
    const int64_t e2 = ((b + n_warps) << 5) + lane;
    if (e2 < n_edges) {
      s_nxt = int(__ldg(src + e2));
      d_nxt = int(__ldg(dst + e2));
      r_nxt = int(__ldg(etype + e2));
    }
    const bool uniform = __all_sync(kFull, r == r_first);
    float4 wv[NV];
    if (uniform) {
#pragma unroll
      for (int v = 0; v < NV; ++v) wv[v] = ok[v] ? __ldg(row_ptr(w4, r_first, wdb) + v * 8) : zero;
    }
    float mine = 0.f;
#pragma unroll 2
    for (int t = 0; t < 8; ++t) {
      const int from = t * 4 + slot;
      const int ss = __shfl_sync(kFull, s, from), dd = __shfl_sync(kFull, d, from);
      const float4* za = row_ptr(z4, ss, ldb);
      const float4* zb = row_ptr(z4, dd, ldb);
      float4 a[NV], c[NV];
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        a[v] = ok[v] ? __ldg(za + v * 8) : zero;
        c[v] = ok[v] ? __ldg(zb + v * 8) : zero;
      }
      if (!uniform) {
        const int rr = __shfl_sync(kFull, r, from);
#pragma unroll
        for (int v = 0; v < NV; ++v) wv[v] = ok[v] ? __ldg(row_ptr(w4, rr, wdb) + v * 8) : zero;
      }
      float acc = 0.f;
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        acc = fmaf(a[v].x * c[v].x, wv[v].x, acc);
        acc = fmaf(a[v].y * c[v].y, wv[v].y, acc);
        acc = fmaf(a[v].z * c[v].z, wv[v].z, acc);
        acc = fmaf(a[v].w * c[v].w, wv[v].w, acc);
      }
      acc += __shfl_xor_sync(kFull, acc, 4);
      acc += __shfl_xor_sync(kFull, acc, 2);
      acc += __shfl_xor_sync(kFull, acc, 1);
      // edge L of the batch was scored at step L / 4 by the lane group L % 4
      const float got = __shfl_sync(kFull, acc, (lane & 3) << 3);
      if ((lane >> 2) == t) mine = got;
    }
    if (live) out[e] = sigmoid ? 1.0f / (1.0f + expf(-mine)) : mine;
  }
}

__global__ void distmult_coef_kernel(const float* __restrict__ grad_out, const float* __restrict__ out, int64_t n,
                                     int sigmoid, float* __restrict__ coef) {
  const int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= n) return;
  float g = grad_out[e];
  if (sigmoid) {
    const float s = out[e];
    g *= s * (1.0f - s);
  }
  coef[e] = g;
}

// ---------------------------------------------------------------------------
// backward in ONE gather pass (K10).  The endpoint entries of an edge list are grouped by (node, relation)
// — the "pair CSR", rows = node * n_rel + rel — and one walk forms
//     T[n, r, :] = sum over the entries (other, e) of pair row (n, r) of coef[e] * z[other, :].
// Both gradients follow from T without touching the edges again:
//     dz[n]  = sum_r T[n, r] .* w[r]
//     dw[r]  = 1/2 sum_n z[n] .* T[n, r]          (every edge sits in two pair rows: (src, r) and (dst, r))
// so the second gather pass of the two-walk scheme (z[src] and z[dst] per edge for dw) disappears, and the
// walk itself carries no relation logic (no w gather, no run accumulator): fewer registers, more warps.
// Positive and negative lists write their own T; distmult_grads_kernel adds them on the fly.
// ---------------------------------------------------------------------------
template <int LPE, int VEC, int NV>
__global__ void __launch_bounds__(256) pair_walk_kernel(const gn_csr csr, const int32_t* __restrict__ ent_other,
                                                        const int32_t* __restrict__ ent_eid,
                                                        const float* __restrict__ coef, const float* __restrict__ z,
                                                        int64_t ldz, int D, float* __restrict__ T,
                                                        float* __restrict__ partial) {
  ChunkInfo ci;
  if (!chunk_info(csr, ci)) return;
  constexpr int EPI = 32 / LPE;
  const int lane = threadIdx.x & 31;
  const int slot = lane / LPE, fl = lane % LPE;
  Vec<VEC> acc[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v)
#pragma unroll
    for (int i = 0; i < VEC; ++i) acc[v].v[i] = 0.f;
  for (int s0 = ci.beg + slot; s0 < ci.end; s0 += 2 * EPI) {
    const int s1 = s0 + EPI;
    const bool has1 = s1 < ci.end;
    const float* pa0 = z + int64_t(__ldg(ent_other + s0)) * ldz;
    const float* pa1 = has1 ? z + int64_t(__ldg(ent_other + s1)) * ldz : z;
    const float g0 = __ldg(coef + __ldg(ent_eid + s0));
    const float g1 = has1 ? __ldg(coef + __ldg(ent_eid + s1)) : 0.f;
    Vec<VEC> a0[NV], a1[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int f = (v * LPE + fl) * VEC;
      if (f < D) {
        a0[v] = load_vec<VEC>(pa0 + f);
        a1[v] = load_vec<VEC>(pa1 + f);
      }
    }
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int f = (v * LPE + fl) * VEC;
      if (f < D) {
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
          acc[v].v[i] = fmaf(g0, a0[v].v[i], acc[v].v[i]);
          acc[v].v[i] = fmaf(g1, a1[v].v[i], acc[v].v[i]);     // g1 == 0 when the slot has no 2nd entry
        }
      }
    }
  }
#pragma unroll
  for (int v = 0; v < NV; ++v) reduce_slots<LPE, VEC>(acc[v]);
  const int row = ci.row;
  auto emit = [&](int, int f, const Vec<VEC>& sum) { store_vec<VEC>(T + int64_t(row) * D + f, sum); };
  finish_row<LPE, VEC, NV>(csr, ci, acc, D, partial, emit);
}

// Batch form of the walk (D % 4 == 0, D <= 128): like spmm_kernel, a warp reads 32 entries (other endpoint, coef of
// the entry's edge) with one coalesced load + one gather per lane, then hands them to 4 entry slots x 8 feature lanes
// with shuffles: no dependent index -> row round trip per step, a third of the instructions of the form above
// (ncu r02_v17: 11 warp instructions per entry), 128-byte row pieces per quarter-warp.  Same row-split finish.
template <int NV>
__global__ void __launch_bounds__(256, 4) pair_walk_batch_kernel(const gn_csr csr, const int32_t* __restrict__ ent_other,
                                                                 const int32_t* __restrict__ ent_eid,
                                                                 const float* __restrict__ coef,
                                                                 const float* __restrict__ z, int64_t ldz, int D,
                                                                 float* __restrict__ T, float* __restrict__ partial) {
  ChunkInfo ci;
  if (!chunk_info(csr, ci)) return;
  const int lane = threadIdx.x & 31;
  const int slot = lane >> 3, fl = lane & 7;
  const int D4 = D >> 2;
  const unsigned ldb = unsigned(ldz) * 4u;
  const float4* __restrict__ z4 = reinterpret_cast<const float4*>(z) + fl;
  bool ok[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) ok[v] = (v * 8 + fl) < D4;
  Vec<4> acc[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v)
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[v].v[i] = 0.f;
  for (int base = ci.beg; base < ci.end; base += 32) {
    const int mine = base + lane;
    int o = 0;            // entries past the end of the chunk: row 0 with coefficient 0
    float g = 0.f;
    if (mine < ci.end) {
      o = __ldg(ent_other + mine);
      g = __ldg(coef + __ldg(ent_eid + mine));
    }
    const int steps = min(8, (ci.end - base + 3) >> 2);
#pragma unroll 2
    for (int t = 0; t < steps; ++t) {
      const int from = t * 4 + slot;
      const int oo = __shfl_sync(kFull, o, from);
      const float gg = __shfl_sync(kFull, g, from);
      const float4* za = row_ptr(z4, oo, ldb);
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        if (ok[v]) {
          const float4 a = __ldg(za + v * 8);
          acc[v].v[0] = fmaf(gg, a.x, acc[v].v[0]);
          acc[v].v[1] = fmaf(gg, a.y, acc[v].v[1]);
          acc[v].v[2] = fmaf(gg, a.z, acc[v].v[2]);
          acc[v].v[3] = fmaf(gg, a.w, acc[v].v[3]);
        }
      }
    }
  }
#pragma unroll
  for (int v = 0; v < NV; ++v) reduce_slots<8, 4>(acc[v]);
  const int row = ci.row;
  auto emit = [&](int, int f, const Vec<4>& sum) { store_vec<4>(T + int64_t(row) * D + f, sum); };
  finish_row<8, 4, NV>(csr, ci, acc, D, partial, emit);
}

// dz / dw from T (and an optional second T of another edge list).
//   dz[n] = sum_r T[n,r] .* w[r]          one CTA per node: its threads are G groups of D columns, group g adds the
//                                          relations g, g + G, ... in order, then the G partial rows in group order;
//   dw[r] = 1/2 sum_n z[n] .* T[n,r]      the long reduction (n_nodes terms per relation, strided rows of T): every
//                                          relation is cut into n_slabs slabs of nodes, one CTA each, whose partial
//                                          rows go to `ws`; the LAST slab of a relation to arrive (integer counter)
//                                          adds the slabs in slab order.
// Fixed summation orders everywhere: bit-reproducible.  dw CTAs take the first blocks so the long ones start first.
constexpr int kGradThreads = 1024;
constexpr int kGradSlabNodes = 96;     // nodes per dw slab: 8 rounds of 12 groups at D = 80

__device__ __forceinline__ float grads_reduce_groups(float acc, int g, int G, int f, int D, float* red) {
  if (g < G && f < D) red[g * D + f] = acc;
  __syncthreads();
  float s = 0.f;
  if (g == 0 && f < D) {
    s = red[f];
    for (int k = 1; k < G; ++k) s += red[k * D + f];
  }
  __syncthreads();
  return s;
}

__global__ void __launch_bounds__(kGradThreads) distmult_grads_kernel(const float* __restrict__ T,
                                                                     const float* __restrict__ T2, int n_nodes,
                                                                     int n_rel, int D, const float* __restrict__ z,
                                                                     int64_t ldz, const float* __restrict__ w,
                                                                     float* __restrict__ dz, int64_t lddz,
                                                                     float* __restrict__ dw, int n_slabs,
                                                                     float* __restrict__ slab_part,
                                                                     unsigned int* __restrict__ slab_count) {
  extern __shared__ float red[];                       // [G][D]
  __shared__ int s_last;
  const int G = kGradThreads / D;
  const int g = int(threadIdx.x) / D, f = int(threadIdx.x) % D;
  const int n_dw_blocks = dw ? n_rel * n_slabs : 0;
  constexpr int kU = 8;
  if (int(blockIdx.x) >= n_dw_blocks) {
    // ---------------------------------------------------------------- dz row
    const int row = int(blockIdx.x) - n_dw_blocks;
    if (dz == nullptr || row >= n_nodes) return;
    float acc = 0.f;
    if (g < G) {
      for (int i0 = g; i0 < n_rel; i0 += kU * G) {
        float tv[kU], ov[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          const int i = i0 + u * G;
          tv[u] = ov[u] = 0.f;
          if (i < n_rel) {
            const int64_t t = (int64_t(row) * n_rel + i) * D + f;
            tv[u] = __ldg(T + t);
            if (T2) tv[u] += __ldg(T2 + t);
            ov[u] = __ldg(w + int64_t(i) * D + f);
          }
        }
#pragma unroll
        for (int u = 0; u < kU; ++u) acc = fmaf(tv[u], ov[u], acc);
      }
    }
    const float s = grads_reduce_groups(acc, g, G, f, D, red);
    if (g == 0) dz[int64_t(row) * lddz + f] = s;
    return;
  }
  // ------------------------------------------------------------------ dw slab
  const int rel = int(blockIdx.x) / n_slabs, slab = int(blockIdx.x) % n_slabs;
  const int n0 = slab * kGradSlabNodes;
  const int n1 = n0 + kGradSlabNodes < n_nodes ? n0 + kGradSlabNodes : n_nodes;
  float acc = 0.f;
  if (g < G) {
    for (int i0 = n0 + g; i0 < n1; i0 += kU * G) {
      float tv[kU], ov[kU];
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        const int i = i0 + u * G;
        tv[u] = ov[u] = 0.f;
        if (i < n1) {
          const int64_t t = (int64_t(i) * n_rel + rel) * D + f;
          tv[u] = __ldg(T + t);
          if (T2) tv[u] += __ldg(T2 + t);
          ov[u] = __ldg(z + int64_t(i) * ldz + f);
        }
      }
#pragma unroll
      for (int u = 0; u < kU; ++u) acc = fmaf(tv[u], ov[u], acc);
    }
  }
  const float s = grads_reduce_groups(acc, g, G, f, D, red);
  if (n_slabs == 1) {
    if (g == 0) dw[int64_t(rel) * D + f] = 0.5f * s;
    return;
  }
  if (g == 0) slab_part[(int64_t(rel) * n_slabs + slab) * D + f] = s;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(slab_count + rel, 1u) == unsigned(n_slabs - 1)) ? 1 : 0;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if (g == 0) {
    const float* p = slab_part + int64_t(rel) * n_slabs * D + f;
    float t = 0.f;
    int k = 0;
    for (; k + 7 < n_slabs; k += 8) {                 // eight slabs in flight, added in slab order
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = __ldcg(p + int64_t(k + u) * D);
#pragma unroll
      for (int u = 0; u < 8; ++u) t += v[u];
    }
    for (; k < n_slabs; ++k) t += __ldcg(p + int64_t(k) * D);
    dw[int64_t(rel) * D + f] = 0.5f * t;
  }
  if (threadIdx.x == 0) slab_count[rel] = 0;
}

// ---- 128-bit variant (D % 4 == 0, D <= 128): CTAs of C4 * 16 threads (C4 = D / 4 float4 columns x 16 sub-rows).
//   dz CTA: `nodes` nodes x `gr` relation groups (nodes * gr == 16); a sub-row adds the relations gr, gr + GR, ...
//           of its node with kVU float4 pairs in flight, the GR partial rows are added in group order;
//   dw CTA: one (relation, slab of kVSlab nodes): 16 sub-rows stride over the slab's nodes, partial rows added in
//           sub-row order, slabs combined by the last-arriving CTA in slab order (as in the scalar kernel).
// A few hundred CTAs that each stream contiguous 4*D-byte rows of T, instead of one 1024-thread CTA per node.
constexpr int kVSub = 16;
constexpr int kVSlab = 128;
constexpr int kVU = 4;

__device__ __forceinline__ void f4_fma(float4& a, const float4& x, const float4& y) {
  a.x = fmaf(x.x, y.x, a.x); a.y = fmaf(x.y, y.y, a.y); a.z = fmaf(x.z, y.z, a.z); a.w = fmaf(x.w, y.w, a.w);
}
__device__ __forceinline__ float4 f4_add(const float4& x, const float4& y) {
  return make_float4(x.x + y.x, x.y + y.y, x.z + y.z, x.w + y.w);
}

__global__ void __launch_bounds__(512) distmult_grads_vec_kernel(const float* __restrict__ T,
                                                                 const float* __restrict__ T2, int n_nodes, int n_rel,
                                                                 int D, const float* __restrict__ z, int64_t ldz,
                                                                 const float* __restrict__ w, float* __restrict__ dz,
                                                                 int64_t lddz, float* __restrict__ dw, int n_slabs,
                                                                 float* __restrict__ slab_part,
                                                                 unsigned int* __restrict__ slab_count, int gr_count) {
  extern __shared__ float4 red4[];                     // [kVSub][C4]
  __shared__ int s_last;
  const int C4 = D >> 2;
  const int c4 = int(threadIdx.x) % C4, sub = int(threadIdx.x) / C4;
  const int n_dw_blocks = dw ? n_rel * n_slabs : 0;
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 acc = zero;
  if (int(blockIdx.x) >= n_dw_blocks) {
    // ---------------------------------------------------------------- dz rows
    const int GR = gr_count, nodes = kVSub / GR;
    const int node = (int(blockIdx.x) - n_dw_blocks) * nodes + sub / GR, g = sub % GR;
    if (dz == nullptr) return;
    if (node < n_nodes) {
      const float4* t1 = reinterpret_cast<const float4*>(T + int64_t(node) * n_rel * D) + c4;
      const float4* t2 = T2 ? reinterpret_cast<const float4*>(T2 + int64_t(node) * n_rel * D) + c4 : nullptr;
      const float4* wp = reinterpret_cast<const float4*>(w) + c4;
      for (int r0 = g; r0 < n_rel; r0 += kVU * GR) {
        float4 tv[kVU], wv[kVU];
#pragma unroll
        for (int u = 0; u < kVU; ++u) {
          const int r = r0 + u * GR;
          tv[u] = wv[u] = zero;
          if (r < n_rel) {
            tv[u] = __ldg(t1 + int64_t(r) * C4);
            if (t2) tv[u] = f4_add(tv[u], __ldg(t2 + int64_t(r) * C4));
            wv[u] = __ldg(wp + int64_t(r) * C4);
          }
        }
#pragma unroll
        for (int u = 0; u < kVU; ++u) f4_fma(acc, tv[u], wv[u]);
      }
    }
    if (GR > 1) {
      red4[sub * C4 + c4] = acc;
      __syncthreads();
      if (g == 0 && node < n_nodes) {
        for (int k = 1; k < GR; ++k) acc = f4_add(acc, red4[(sub + k) * C4 + c4]);
      }
    }
    if (g == 0 && node < n_nodes) *reinterpret_cast<float4*>(dz + int64_t(node) * lddz + 4 * c4) = acc;
    return;
  }
  // ------------------------------------------------------------------ dw slab
  const int rel = int(blockIdx.x) / n_slabs, slab = int(blockIdx.x) % n_slabs;
  const int n0 = slab * kVSlab;
  const int n1 = n0 + kVSlab < n_nodes ? n0 + kVSlab : n_nodes;
  for (int i0 = n0 + sub; i0 < n1; i0 += kVU * kVSub) {
    float4 tv[kVU], zv[kVU];
#pragma unroll
    for (int u = 0; u < kVU; ++u) {
      const int i = i0 + u * kVSub;
      tv[u] = zv[u] = zero;
      if (i < n1) {
        const int64_t t = (int64_t(i) * n_rel + rel) * C4 + c4;
        tv[u] = __ldg(reinterpret_cast<const float4*>(T) + t);
        if (T2) tv[u] = f4_add(tv[u], __ldg(reinterpret_cast<const float4*>(T2) + t));
        zv[u] = __ldg(reinterpret_cast<const float4*>(z + int64_t(i) * ldz) + c4);
      }
    }
#pragma unroll
    for (int u = 0; u < kVU; ++u) f4_fma(acc, tv[u], zv[u]);
  }
  red4[sub * C4 + c4] = acc;
  __syncthreads();
  if (sub == 0) {
    for (int k = 1; k < kVSub; ++k) acc = f4_add(acc, red4[k * C4 + c4]);
    if (n_slabs == 1) {
      *reinterpret_cast<float4*>(dw + int64_t(rel) * D + 4 * c4) =
          make_float4(0.5f * acc.x, 0.5f * acc.y, 0.5f * acc.z, 0.5f * acc.w);
    } else {
      *reinterpret_cast<float4*>(slab_part + (int64_t(rel) * n_slabs + slab) * D + 4 * c4) = acc;
    }
  }
  if (n_slabs == 1) return;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(slab_count + rel, 1u) == unsigned(n_slabs - 1)) ? 1 : 0;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if (sub == 0) {
    const float4* p = reinterpret_cast<const float4*>(slab_part + int64_t(rel) * n_slabs * D) + c4;
    float4 t = zero;
    int k = 0;
    for (; k + 7 < n_slabs; k += 8) {                 // eight slabs in flight, added in slab order
      float4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = __ldcg(p + int64_t(k + u) * C4);
#pragma unroll
      for (int u = 0; u < 8; ++u) t = f4_add(t, v[u]);
    }
    for (; k < n_slabs; ++k) t = f4_add(t, __ldcg(p + int64_t(k) * C4));
    *reinterpret_cast<float4*>(dw + int64_t(rel) * D + 4 * c4) = make_float4(0.5f * t.x, 0.5f * t.y, 0.5f * t.z, 0.5f * t.w);
  }
  if (threadIdx.x == 0) slab_count[rel] = 0;
}

// arrival counters of the dw reduction: cleared by a KERNEL node — a memset node between two kernels of a captured
// graph costs several microseconds of dependency latency on the decoder backward's chain
// (profiles/r02_v15_pose_n1_rank0_summary.txt: 7.5 us between the memset and distmult_grads_vec_kernel)
__global__ void zero_u32_kernel(unsigned int* __restrict__ p, int n) {
  const int i = int(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) p[i] = 0u;
}

__global__ void pair_keys_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                 const int64_t* __restrict__ etype, int64_t n_edges, int32_t n_rel,
                                 int32_t* __restrict__ key) {
  const int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (e >= n_edges) return;
  const int r = int32_t(etype[e]);
  key[e] = int32_t(src[e]) * n_rel + r;
  key[n_edges + e] = int32_t(dst[e]) * n_rel + r;
}

__global__ void pair_fill_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst, int64_t n_edges,
                                 const int32_t* __restrict__ perm, int32_t* __restrict__ ent_other,
                                 int32_t* __restrict__ ent_eid) {
  const int64_t s = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (s >= 2 * n_edges) return;
  const int64_t q = perm[s];
  const int64_t e = q < n_edges ? q : q - n_edges;
  ent_other[s] = int32_t(q < n_edges ? dst[e] : src[e]);
  ent_eid[s] = int32_t(e);
}

// ---------------------------------------------------------------------------
// softmax (warp per row)
// ---------------------------------------------------------------------------
__global__ void softmax_fwd_kernel(const float* __restrict__ x, int64_t n, int C, float* __restrict__ y) {
  const int64_t row = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  const float* xr = x + row * C;
  float m = -INFINITY;
  for (int c = lane; c < C; c += 32) m = fmaxf(m, xr[c]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kFull, m, o));
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += expf(xr[c] - m);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(kFull, s, o);
  const float inv = 1.0f / s;
  for (int c = lane; c < C; c += 32) y[row * C + c] = expf(xr[c] - m) * inv;
}

__global__ void softmax_bwd_kernel(const float* __restrict__ y, const float* __restrict__ gy, int64_t n, int C,
                                   float* __restrict__ gx) {
  const int64_t row = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  float dot = 0.f;
  for (int c = lane; c < C; c += 32) dot = fmaf(y[row * C + c], gy[row * C + c], dot);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(kFull, dot, o);
  for (int c = lane; c < C; c += 32) gx[row * C + c] = y[row * C + c] * (gy[row * C + c] - dot);
}

struct WidthPlan {
  int vec, lpe, nv;
  bool ok;
};

// lanes-per-entry and vectors-per-lane for a D-wide row (at most kMaxNV vectors per lane)
inline WidthPlan plan_width(int D, bool can_vec4) {
  WidthPlan p{can_vec4 ? 4 : 1, 0, 0, true};
  const int units = (D + p.vec - 1) / p.vec;
  if (units <= 4 * kMaxNV) p.lpe = 4;
  else if (units <= 32 * kMaxNV) p.lpe = 32;
  else p.ok = false;
  if (p.ok) {
    const int need = (units + p.lpe - 1) / p.lpe;
    p.nv = need <= 1 ? 1 : need <= 2 ? 2 : need <= 4 ? 4 : need <= 5 ? 5 : kMaxNV;
  }
  return p;
}

}  // namespace gn

using namespace gn;

extern "C" {

int gn_distmult_fwd(const float* z, int64_t ldz, int32_t D, const float* w, const int64_t* src, const int64_t* dst,
                    const int64_t* etype, int64_t n_edges, int sigmoid, float* out, void* stream) {
  if (n_edges < 0 || D <= 0) return GN_ERR_ARG;
  if (n_edges == 0) return GN_OK;
  if (!z || !w || !src || !dst || !etype || !out) return GN_ERR_ARG;
  cudaStream_t st = as_stream(stream);
  // float4 rows.  Up to D = 128 they take the batch form, which steps rows with a 32-bit byte stride, so there a z row
  // stride of 2^30 floats or more takes the scalar per-edge form.
  const bool v4 = (D % 4 == 0) && (ldz % 4 == 0) && aligned16(z) && aligned16(w) &&
                  (D > 128 || ldz < (int64_t(1) << 30));
  if (v4 && D <= 128) {
    const int nv = (D / 4 + 7) / 8;
    int64_t nwarps = ceil_div(n_edges, 32);
    const int64_t cap = int64_t(148) * 4 * 8;                // one wave of resident warps; each walks its batches
    if (nwarps > cap) nwarps = cap;
    const unsigned g = (unsigned)ceil_div(nwarps, 8);
#define GN_FWDB_CASE(N)                                                                                              \
  if (nv == N) {                                                                                                     \
    GN_LAUNCH((distmult_fwd_batch_kernel<N>), g, 256, 0, st, z, ldz, D, w, src, dst, etype, n_edges, sigmoid, out);  \
    return GN_OK;                                                                                                    \
  }
    GN_FWDB_CASE(1)
    GN_FWDB_CASE(2)
    GN_FWDB_CASE(3)
    GN_FWDB_CASE(4)
#undef GN_FWDB_CASE
  }
  const int units = v4 ? D / 4 : D;
  const int lpe = units <= 32 ? 4 : (units <= 64 ? 8 : 32);
  const int epi = 32 / lpe;
  int64_t warps = ceil_div(n_edges, epi);
  const int64_t max_warps = int64_t(148) * 64 * 4;
  if (warps > max_warps) warps = max_warps;
  const unsigned grid = (unsigned)ceil_div(warps, 8);
#define GN_FWD_CASE(L, V)                                                                                           \
  if (lpe == L && (v4 ? 4 : 1) == V) {                                                                              \
    GN_LAUNCH((distmult_fwd_kernel<L, V>), grid, 256, 0, st, z, ldz, D, w, src, dst, etype, n_edges, sigmoid, out); \
    return GN_OK;                                                                                                   \
  }
  GN_FWD_CASE(8, 4)
  GN_FWD_CASE(32, 4)
  GN_FWD_CASE(4, 1)
  GN_FWD_CASE(8, 1)
  GN_FWD_CASE(32, 1)
#undef GN_FWD_CASE
  return GN_ERR_ARG;
}

int gn_distmult_coef(const float* grad_out, const float* out, int64_t n_edges, int sigmoid, float* coef,
                     void* stream) {
  if (n_edges < 0) return GN_ERR_ARG;
  if (n_edges == 0) return GN_OK;
  if (!grad_out || !coef || (sigmoid && !out)) return GN_ERR_ARG;
  GN_LAUNCH(distmult_coef_kernel, (unsigned)ceil_div(n_edges, 256), 256, 0, as_stream(stream), grad_out, out, n_edges,
            sigmoid, coef);
  return GN_OK;
}

int gn_softmax_fwd(const float* logits, int64_t n, int32_t C, float* out, void* stream) {
  if (n < 0 || C <= 0) return GN_ERR_ARG;
  if (n == 0) return GN_OK;
  if (!logits || !out) return GN_ERR_ARG;
  GN_LAUNCH(softmax_fwd_kernel, (unsigned)ceil_div(n * 32, 256), 256, 0, as_stream(stream), logits, n, C, out);
  return GN_OK;
}

int gn_softmax_bwd(const float* out, const float* grad_out, int64_t n, int32_t C, float* grad_logits, void* stream) {
  if (n < 0 || C <= 0) return GN_ERR_ARG;
  if (n == 0) return GN_OK;
  if (!out || !grad_out || !grad_logits) return GN_ERR_ARG;
  GN_LAUNCH(softmax_bwd_kernel, (unsigned)ceil_div(n * 32, 256), 256, 0, as_stream(stream), out, grad_out, n, C,
            grad_logits);
  return GN_OK;
}

size_t gn_pair_prep_workspace_bytes(int64_t n_edges) {
  const size_t E2 = size_t(n_edges > 0 ? 2 * n_edges : 1);
  return 3 * align_up(E2 * 4) + sort_ws_bytes(2 * n_edges) + 4096;
}

int gn_pair_prep(const int64_t* src, const int64_t* dst, const int64_t* etype, int64_t n_edges, int32_t n_nodes,
                 int32_t n_rel, int32_t* pair_rowptr, int32_t* ent_other, int32_t* ent_eid, void* ws, size_t ws_bytes,
                 void* stream) {
  if (n_edges < 0 || n_nodes <= 0 || n_rel <= 0 || !pair_rowptr) return GN_ERR_ARG;
  if (n_edges > 0 && (!src || !dst || !etype || !ent_other || !ent_eid)) return GN_ERR_ARG;
  if (2 * n_edges >= (int64_t(1) << 31) || int64_t(n_nodes) * n_rel >= (int64_t(1) << 31)) return GN_ERR_RANGE;
  cudaStream_t st = as_stream(stream);
  const int32_t n_rows = n_nodes * n_rel;
  const int64_t E2 = 2 * n_edges;
  const size_t Ea = size_t(E2 > 0 ? E2 : 1);
  Arena a(ws, ws_bytes);
  int32_t* key = a.take<int32_t>(Ea);
  int32_t* sorted = a.take<int32_t>(Ea);
  int32_t* perm = a.take<int32_t>(Ea);
  if (!a.ok()) return GN_ERR_WORKSPACE;
  if (n_edges > 0) {
    GN_LAUNCH(pair_keys_kernel, (unsigned)ceil_div(n_edges, 256), 256, 0, st, src, dst, etype, n_edges, n_rel, key);
  }
  GN_CHECK(sort_pairs(key, nullptr, sorted, perm, E2, bits_for(n_rows > 1 ? n_rows : 2), a.base + a.off,
                      a.cap - a.off, st));
  GN_CHECK(rowptr_from_sorted(sorted, E2, n_rows, pair_rowptr, st));
  if (n_edges > 0) {
    GN_LAUNCH(pair_fill_kernel, (unsigned)ceil_div(E2, 256), 256, 0, st, src, dst, n_edges, (const int32_t*)perm,
              ent_other, ent_eid);
  }
  return GN_OK;
}

int gn_distmult_bwd_pairs(const gn_csr* pair_csr, const int32_t* ent_other, const int32_t* ent_eid, const float* coef,
                          const float* z, int64_t ldz, int32_t D, float* T, float* partial, void* stream) {
  if (!pair_csr || !z || !T || D <= 0) return GN_ERR_ARG;
  if (pair_csr->nnz > 0 && (!ent_other || !ent_eid || !coef)) return GN_ERR_ARG;
  const gn_csr& csr = *pair_csr;
  if (csr.n_rows == 0 || csr.n_chunks == 0) return GN_OK;
  if (csr.n_chunks > csr.n_rows && !partial) return GN_ERR_ARG;
  // float4 rows: the batch form up to D = 128, where (as in gn_distmult_fwd) the z row stride must stay below 2^30
  const bool v4 = (D % 4 == 0) && (ldz % 4 == 0) && aligned16(z) && aligned16(T) && (!partial || aligned16(partial)) &&
                  (D > 128 || ldz < (int64_t(1) << 30));
  const WidthPlan p = plan_width(D, v4);
  if (!p.ok) return GN_ERR_ARG;
  cudaStream_t st = as_stream(stream);
  const unsigned grid = (unsigned)ceil_div(csr.n_chunks, 8);
  if (v4 && D <= 128) {
    const int nv = (D / 4 + 7) / 8;
#define GN_PWB_CASE(N)                                                                                        \
  if (nv == N) {                                                                                              \
    GN_LAUNCH((pair_walk_batch_kernel<N>), grid, 256, 0, st, csr, ent_other, ent_eid, coef, z, ldz, D, T,     \
              partial);                                                                                       \
    return GN_OK;                                                                                             \
  }
    GN_PWB_CASE(1)
    GN_PWB_CASE(2)
    GN_PWB_CASE(3)
    GN_PWB_CASE(4)
#undef GN_PWB_CASE
  }
#define GN_PW_CASE(L, V, N)                                                                                  \
  if (p.lpe == L && p.vec == V && p.nv == N) {                                                               \
    GN_LAUNCH((pair_walk_kernel<L, V, N>), grid, 256, 0, st, csr, ent_other, ent_eid, coef, z, ldz, D, T,    \
              partial);                                                                                      \
    return GN_OK;                                                                                            \
  }
// the per-entry form serves float4 rows only past D = 128, and 32 lanes per entry only past 32 units per row
// (so at least two vectors per lane)
#define GN_PW_CASES(L, V) GN_PW_CASE(L, V, 2) GN_PW_CASE(L, V, 4) GN_PW_CASE(L, V, 5) GN_PW_CASE(L, V, 8)
  GN_PW_CASES(32, 4)
  GN_PW_CASE(4, 1, 1)
  GN_PW_CASES(4, 1)
  GN_PW_CASES(32, 1)
#undef GN_PW_CASES
#undef GN_PW_CASE
  return GN_ERR_ARG;
}

static bool grads_vec_ok(int D, const float* T, const float* T2, const float* z, int64_t ldz, const float* w,
                         const float* dz, int64_t lddz, const float* dw) {
  return D % 4 == 0 && D <= 128 && ldz % 4 == 0 && lddz % 4 == 0 && aligned16(T) && (!T2 || aligned16(T2)) &&
         aligned16(z) && aligned16(w) && (!dz || aligned16(dz)) && (!dw || aligned16(dw));
}

size_t gn_distmult_grads_workspace_bytes(int32_t n_nodes, int32_t n_rel, int32_t D) {
  const size_t slabs = size_t(ceil_div(n_nodes > 0 ? n_nodes : 1, kGradSlabNodes));   // the smaller slab size
  return align_up(size_t(n_rel > 0 ? n_rel : 1) * 4) + size_t(n_rel > 0 ? n_rel : 1) * slabs * size_t(D > 0 ? D : 1) * 4 + 256;
}

int gn_distmult_grads(const float* T, const float* T2, int32_t n_nodes, int32_t n_rel, int32_t D, const float* z,
                      int64_t ldz, const float* w, float* dz, int64_t lddz, float* dw, void* ws, size_t ws_bytes,
                      void* stream) {
  if (n_nodes <= 0 || n_rel <= 0 || D <= 0 || D > kGradThreads || !T || !z || !w || (!dz && !dw)) return GN_ERR_ARG;
  cudaStream_t st = as_stream(stream);
  const bool vec = grads_vec_ok(D, T, T2, z, ldz, w, dz, lddz, dw);
  const int n_slabs = int(ceil_div(n_nodes, vec ? kVSlab : kGradSlabNodes));
  unsigned int* count = nullptr;
  float* part = nullptr;
  if (dw && n_slabs > 1) {
    if (!ws || ws_bytes < gn_distmult_grads_workspace_bytes(n_nodes, n_rel, D)) return GN_ERR_WORKSPACE;
    count = static_cast<unsigned int*>(ws);
    part = reinterpret_cast<float*>(static_cast<char*>(ws) + align_up(size_t(n_rel) * 4));
    GN_LAUNCH(zero_u32_kernel, (unsigned)ceil_div(n_rel, 256), 256, 0, st, count, n_rel);
  }
  if (vec) {
    const int C4 = D / 4;
    const int GR = n_rel > 32 ? 8 : 1;                       // many relations: eight sub-rows share a node
    const int nodes_per_cta = kVSub / GR;
    const int64_t blocks = int64_t(dw ? n_rel * n_slabs : 0) + (dz ? ceil_div(n_nodes, nodes_per_cta) : 0);
    GN_LAUNCH(distmult_grads_vec_kernel, (unsigned)blocks, C4 * kVSub, size_t(kVSub) * C4 * sizeof(float4), st, T, T2,
              n_nodes, n_rel, D, z, ldz, w, dz, lddz, dw, n_slabs, part, count, GR);
    return GN_OK;
  }
  const int G = kGradThreads / D;
  const size_t smem = size_t(G) * size_t(D) * sizeof(float);
  const int64_t blocks = int64_t(dw ? n_rel * n_slabs : 0) + (dz ? n_nodes : 0);
  GN_LAUNCH(distmult_grads_kernel, (unsigned)blocks, kGradThreads, smem, st, T, T2, n_nodes, n_rel, D, z, ldz, w, dz,
            lddz, dw, n_slabs, part, count);
  return GN_OK;
}

}  // extern "C"
