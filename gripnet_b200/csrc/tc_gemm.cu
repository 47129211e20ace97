// K2/K6 tensor path: C[M,N] = A[M,K] * op(B) on the 5th-generation tensor cores
// (tcgen05.mma kind::tf32, accumulators in TMEM) with fp32-grade accuracy by an
// error-compensated 3xTF32 split.
//
// Why: north_star item 3 sends the dense X.W / X.W_r feature transforms to tcgen05, but
// the parity bar is 1e-5 relative in fp32 and a TF32 operand keeps 10 mantissa bits.
// Every operand element is split  x = hi + lo  (hi = rna-tf32(x), lo = rna-tf32(x - hi))
// while it is staged, and each k-step issues three MMAs: hi*hi into the main fp32 accumulator,
// lo*hi + hi*lo into a second one (the lo*lo term, <= 2^-22 relative, is dropped).  The tensor
// core TRUNCATES when it adds into the accumulator, so the small cross terms get their own
// TMEM columns (their truncation error is 2^-11 of the main one's) and the main accumulator
// takes one add per k-step instead of three; the two are summed in fp32 in the epilogue.
//
// Shape regime: M = number of nodes (huge), K <= 512, N <= 512 (feature widths).  These
// products are HBM-bound (read A once, write C once), so the kernel is built around the
// A stream, not around the tensor pipe:
//   * one CTA per 128-row tile of A (x one N tile of <= 256 columns); 10 warps:
//       warps 0-7  stage A: coalesced 128-bit global loads -> split -> st.shared in the
//                  canonical no-swizzle K-major core-matrix layout (software-pipelined
//                  one k-block ahead), later the epilogue (tcgen05.ld -> fused addend /
//                  ReLU mask -> 128-bit stores);
//       warp 8     allocates TMEM and issues the MMAs (one lane), commits to mbarriers;
//       warp 9     brings the pre-split image of B for each k-block with ONE bulk
//                  async copy (cp.async.bulk, TMA engine) completing on the stage's mbarrier;
//   * B is shared by every CTA.  A layer's weight matrix (N <= 64 columns, a few KB) is split by the
//     B-producer warp itself, k-block by k-block, straight into the stage: no extra launch on the
//     step's dependency chain.  A wide B (the [in, R*out] relation transform of pose-2) is split once
//     per call by a prep kernel into the caller's workspace, already in the shared-memory layout
//     (k-block major), and each k-block arrives with ONE bulk async copy;
//   * 2-3 smem stages, full/empty mbarriers; tcgen05.commit releases a stage when the
//     MMAs that read it have retired.
#include "tc_common.cuh"

namespace gn {
namespace tc {

struct Params {
  int M, N, K;
  const float* A; int64_t lda;
  float* C; int64_t ldc;
  const float* addend; int64_t ldd;
  const float* mask; int64_t ldm;
  const char* b_image;   // [n_tile][k_block][hi|lo][chunk][row][4 floats] (+ plane padding); NULL: split B in the kernel
  const float* B; int64_t ldb; int transB;   // op(B) itself, read by the B producer when b_image == NULL
  int nt;                // columns per N tile (multiple of 16, <= 256)
  int n_kb;              // k-blocks
  int stages;
  int tmem_cols;
  int n_acc;             // TMEM accumulator PAIRS (hi*hi | cross terms); each covers kb_per_acc k-blocks
  int kb_per_acc;
  int b_resident;        // the whole split image of this N tile of B stays in shared memory for every M tile
};

// ---------------------------------------------------------------------------------------
// B image: hi/lo split of op(B), laid out exactly as one smem stage wants it
// ---------------------------------------------------------------------------------------
// op(B)[k, n] for the four layouts of B the callers have:
//   0  B stored [K, N]:  B[k*ldb + n]                 1  B stored [N, K] (op = transpose):  B[n*ldb + k]
//   2  relation-batched along N (forward of myRGCN, Y[:, r, :] = X W[r], W stored [R][K][inner]):
//        n = r*inner + c  ->  B[r*stride + k*ldb + c]
//   3  relation-batched along K (dX = sum_r dY[:, r, :] W[r]^T):
//        k = r*inner + c  ->  B[r*stride + n*ldb + c]
struct BView {
  const float* B;
  int64_t ldb, stride;
  int mode, inner;
  __device__ __forceinline__ float at(int k, int n) const {
    switch (mode) {
      case 0: return __ldg(B + int64_t(k) * ldb + n);
      case 1: return __ldg(B + int64_t(n) * ldb + k);
      case 2: return __ldg(B + int64_t(n / inner) * stride + int64_t(k) * ldb + (n % inner));
      default: return __ldg(B + int64_t(k / inner) * stride + int64_t(n) * ldb + (k % inner));
    }
  }
};

__global__ void __launch_bounds__(256) b_image_kernel(const BView bv, int K, int N, int nt, int n_kb,
                                                      char* __restrict__ image) {
  // one thread per (n_tile, k_block, chunk, row)
  const int64_t idx = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int n_tiles = (N + nt - 1) / nt;
  const int64_t total = int64_t(n_tiles) * n_kb * CHUNKS * nt;
  if (idx >= total) return;
  const int row = int(idx % nt);
  const int c = int((idx / nt) % CHUNKS);
  const int kb = int((idx / (int64_t(nt) * CHUNKS)) % n_kb);
  const int t = int(idx / (int64_t(nt) * CHUNKS * n_kb));
  const int n = t * nt + row;
  float v[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int k = kb * BK + c * 4 + e;
    float x = 0.f;
    if (n < N && k < K) x = bv.at(k, n);
    v[e] = x;
  }
  float4 hi, lo;
  split4(make_float4(v[0], v[1], v[2], v[3]), hi, lo);
  char* base = image + (int64_t(t) * n_kb + kb) * (2 * part_bytes(nt));
  *reinterpret_cast<float4*>(base + c * plane_bytes(nt) + row * 16) = hi;
  *reinterpret_cast<float4*>(base + part_bytes(nt) + c * plane_bytes(nt) + row * 16) = lo;
}

// ---------------------------------------------------------------------------------------
// main kernel
// ---------------------------------------------------------------------------------------
// PF = k-blocks of A a loader thread keeps in flight beyond the one it is converting.  One CTA per SM (large
// operands: three A stages + resident B) streams A from HBM with only its own loads in flight, and ncu showed it
// latency-bound at ~25 % of the HBM peak with PF = 1 (profiles/r02_v17_ncu_full_{aminer,freebase-d}.csv:
// 16 KB per SM and round trip); PF = 3 keeps 64 KB per SM in flight, also across the epilogue of a tile.  Two CTAs
// per SM keep PF = 1 (register budget of 102 per thread).
template <int PF>
__global__ void __launch_bounds__(kThreads, PF == 1 ? 2 : 1) tc_gemm_kernel(const Params p) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ uint64_t full_bar[3], empty_bar[3], acc_bar, acc_free, b_ready;
  __shared__ uint32_t tmem_base_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile_n = blockIdx.y;
  const int nt = p.nt;
  const int S = p.stages;
  // B RESIDENT (the usual case: K*N*8 bytes of hi/lo image fit next to the A stages): B is split / copied ONCE per
  // CTA into its own region behind the stages and every M tile of the persistent loop multiplies against it; the
  // stages then hold A only.  Otherwise B streams through the stages k-block by k-block, for every tile.
  const int stage_sz = p.b_resident ? 2 * part_bytes(BM) : stage_bytes(nt);
  unsigned char* b_res = smem + S * stage_sz;
  const int b_kb_bytes = 2 * part_bytes(nt);
  // PERSISTENT over M tiles: this CTA handles tiles blockIdx.x, blockIdx.x + gridDim.x, ...  The barriers, the TMEM
  // allocation and the stage ring live across tiles (k-block counter `it` keeps running), the loaders fetch the
  // first k-block of the NEXT tile before they turn into the epilogue of the current one, so the fixed per-tile
  // latencies (allocation, barrier set-up, first global round trip) are paid once per CTA instead of once per tile.
  const int m_tiles = (p.M + BM - 1) / BM;
  const int my_tiles = (m_tiles - int(blockIdx.x) + int(gridDim.x) - 1) / int(gridDim.x);

  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(&full_bar[s], kLoaderThreads + (p.b_resident ? 0 : 1));
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&acc_bar, 1);
    mbar_init(&acc_free, kLoaderThreads);
    mbar_init(&b_ready, 1);
    fence_barrier_init();
  }
  if (warp == kLoaderWarps) {  // TMEM allocation by the MMA warp (whole warp, .sync.aligned)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)),
                 "r"(uint32_t(p.tmem_cols)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_acc = tmem_base_slot;

  if (warp < kLoaderWarps) {
    // =============================== A loaders ===============================
    const int c = threadIdx.x & 7;           // k-chunk of this thread
    const int r_base = threadIdx.x >> 3;     // rows r_base + 32*i
    float4 q[PF + 1][4];                     // q[0]: the k-block being converted, q[d]: d k-blocks ahead
    auto issue = [&](int m0, int kb, float4(&dst)[4]) {
      const int k = kb * BK + c * 4;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int m = m0 + r_base + 32 * i;
        if (m < p.M && k < p.K) dst[i] = __ldg(reinterpret_cast<const float4*>(p.A + int64_t(m) * p.lda + k));
        else dst[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    };
    // k-block `itx` of this CTA's flattened (tile, k-block) sequence; runs ahead across tile boundaries, so the
    // next tiles' loads are in flight during the epilogue of the current one
    const int total_it = my_tiles * p.n_kb;
    auto issue_it = [&](int itx, float4(&dst)[4]) {
      if (itx < total_it) {
        const int tt = itx / p.n_kb;
        issue((int(blockIdx.x) + tt * int(gridDim.x)) * BM, itx - tt * p.n_kb, dst);
      }
    };
    const int quarter = warp & 3;                      // TMEM lanes 32*quarter .. +31
    const int halves = (warp >> 2);                    // 0: low column half, 1: high column half
    const int n_tile0 = tile_n * nt;
    const int groups = nt / 16;                        // 16-column groups in this tile
    const int g_begin = halves * ((groups + 1) / 2);
    const int g_end = halves ? groups : (groups + 1) / 2;
#pragma unroll
    for (int d = 0; d < PF; ++d) issue_it(d, q[d]);
    for (int t = 0; t < my_tiles; ++t) {
      const int m0 = (int(blockIdx.x) + t * int(gridDim.x)) * BM;
      for (int kb = 0; kb < p.n_kb; ++kb) {
        const int it = t * p.n_kb + kb;
        const int s = it % S, use = it / S;
        issue_it(it + PF, q[PF]);
        if (use > 0) mbar_wait(&empty_bar[s], (use - 1) & 1);
        unsigned char* a_hi = smem + s * stage_sz;
        unsigned char* a_lo = a_hi + part_bytes(BM);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float4 hi, lo;
          split4(q[0][i], hi, lo);
          const int off = c * plane_bytes(BM) + (r_base + 32 * i) * 16;
          *reinterpret_cast<float4*>(a_hi + off) = hi;
          *reinterpret_cast<float4*>(a_lo + off) = lo;
        }
        fence_proxy_async();                 // generic-proxy stores -> visible to the tensor core
        mbar_arrive(&full_bar[s]);
#pragma unroll
        for (int d = 0; d < PF; ++d)
#pragma unroll
          for (int i = 0; i < 4; ++i) q[d][i] = q[d + 1][i];
      }
      // =============================== epilogue of tile t ================================
      mbar_wait(&acc_bar, t & 1);
      tc_fence_after();
      const int row = quarter * 32 + lane;
      const int m = m0 + row;
      for (int g = g_begin; g < g_end; ++g) {
        // cross-term accumulators first (small), then the hi*hi ones: round-to-nearest fp32 adds
        uint32_t r[16];
        tmem_ld16(tmem_acc + (uint32_t(quarter * 32) << 16) + uint32_t(p.n_acc * nt + g * 16), r);
        for (int a = 1; a < 2 * p.n_acc; ++a) {
          const int col = (a < p.n_acc ? p.n_acc + a : a - p.n_acc) * nt + g * 16;
          uint32_t r2[16];
          tmem_ld16(tmem_acc + (uint32_t(quarter * 32) << 16) + uint32_t(col), r2);
#pragma unroll
          for (int i = 0; i < 16; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) + __uint_as_float(r2[i]));
        }
        if (m >= p.M) continue;
        const int n_first = n_tile0 + g * 16;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int n = n_first + q * 4;
          if (n >= p.N) break;
          float4 v = make_float4(__uint_as_float(r[q * 4 + 0]), __uint_as_float(r[q * 4 + 1]),
                                 __uint_as_float(r[q * 4 + 2]), __uint_as_float(r[q * 4 + 3]));
          if (n + 3 < p.N) {
            if (p.addend) {
              const float4 a = *reinterpret_cast<const float4*>(p.addend + int64_t(m) * p.ldd + n);
              v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
            }
            if (p.mask) {
              const float4 k = *reinterpret_cast<const float4*>(p.mask + int64_t(m) * p.ldm + n);
              if (!(k.x > 0.f)) v.x = 0.f;
              if (!(k.y > 0.f)) v.y = 0.f;
              if (!(k.z > 0.f)) v.z = 0.f;
              if (!(k.w > 0.f)) v.w = 0.f;
            }
            *reinterpret_cast<float4*>(p.C + int64_t(m) * p.ldc + n) = v;
          } else {
            const float vv[4] = {v.x, v.y, v.z, v.w};
            for (int e = 0; e < 4 && n + e < p.N; ++e) {
              float x = vv[e];
              if (p.addend) x += p.addend[int64_t(m) * p.ldd + n + e];
              if (p.mask && !(p.mask[int64_t(m) * p.ldm + n + e] > 0.f)) x = 0.f;
              p.C[int64_t(m) * p.ldc + n + e] = x;
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&acc_free);                // the accumulators may be overwritten by the next tile's MMAs
    }
  } else if (warp == kLoaderWarps) {
    // =============================== MMA issuer ==============================
    if (lane == 0) {
      const uint32_t idesc = make_idesc(BM, nt);
      const uint32_t lbo_a = plane_bytes(BM), lbo_b = plane_bytes(nt);
      // The tensor core truncates when it adds into the fp32 accumulator, so the error of one
      // accumulator grows linearly with K: long reductions are cut into runs of kb_per_acc
      // k-blocks, each with its own TMEM accumulator pair.
      if (p.b_resident && my_tiles > 0) mbar_wait(&b_ready, 0);
      for (int t = 0; t < my_tiles; ++t) {
        if (t > 0) {                         // the epilogue of the previous tile has read the accumulators
          mbar_wait(&acc_free, (t - 1) & 1);
          tc_fence_after();
        }
        uint32_t accumulate = 0;
        for (int kb = 0; kb < p.n_kb; ++kb) {
          const int it = t * p.n_kb + kb;
          const int s = it % S, use = it / S;
          const uint32_t tmem_d = tmem_acc + uint32_t((kb / p.kb_per_acc) * nt);              // hi*hi
          const uint32_t tmem_x = tmem_acc + uint32_t((p.n_acc + kb / p.kb_per_acc) * nt);    // lo*hi + hi*lo
          if (kb % p.kb_per_acc == 0) accumulate = 0;
          mbar_wait(&full_bar[s], use & 1);
          tc_fence_after();
          const uint32_t a_hi = smem_u32(smem + s * stage_sz);
          const uint32_t a_lo = a_hi + part_bytes(BM);
          const uint32_t b_hi = p.b_resident ? smem_u32(b_res + kb * b_kb_bytes) : a_lo + part_bytes(BM);
          const uint32_t b_lo = b_hi + part_bytes(nt);
          const int k_left = p.K - kb * BK;
          const int ksteps = k_left >= BK ? BK / 8 : (k_left + 7) / 8;
          for (int j = 0; j < ksteps; ++j) {
            const uint32_t ao = 2 * j * lbo_a, bo = 2 * j * lbo_b;
            const uint64_t dah = make_desc(a_hi + ao, lbo_a, 128), dal = make_desc(a_lo + ao, lbo_a, 128);
            const uint64_t dbh = make_desc(b_hi + bo, lbo_b, 128), dbl = make_desc(b_lo + bo, lbo_b, 128);
            umma_tf32(tmem_x, dal, dbh, idesc, accumulate);
            umma_tf32(tmem_x, dah, dbl, idesc, 1);
            umma_tf32(tmem_d, dah, dbh, idesc, accumulate);
            accumulate = 1;
          }
          umma_commit(&empty_bar[s]);        // stage reusable once these MMAs have read it
        }
        umma_commit(&acc_bar);               // accumulators of tile t complete
      }
    }
    __syncwarp();
  } else {
    // =============================== B producer ===============================
    if (p.b_resident && my_tiles > 0) {
      if (p.b_image != nullptr) {
        // the pre-split image of this N tile: all its k-blocks are contiguous -> bulk async copies of <= 64 KB
        if (lane == 0) {
          const uint32_t total = uint32_t(p.n_kb) * uint32_t(b_kb_bytes);
          const char* src = p.b_image + int64_t(tile_n) * total;
          mbar_arrive_expect_tx(&b_ready, total);
          for (uint32_t off = 0; off < total; off += 65536) {
            const uint32_t bytes = total - off < 65536 ? total - off : 65536;
            bulk_g2s(b_res + off, src + off, bytes, &b_ready);
          }
        }
      } else {
        const int n_tile0 = tile_n * nt;
        for (int kb = 0; kb < p.n_kb; ++kb) {
          unsigned char* b_hi = b_res + kb * b_kb_bytes;
          unsigned char* b_lo = b_hi + part_bytes(nt);
          for (int i = lane; i < CHUNKS * nt; i += 32) {
            const int row = i % nt, c = i / nt;
            const int n = n_tile0 + row, k = kb * BK + c * 4;
            float v[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              float x = 0.f;
              if (n < p.N && k + e < p.K)
                x = p.transB ? __ldg(p.B + int64_t(n) * p.ldb + k + e) : __ldg(p.B + int64_t(k + e) * p.ldb + n);
              v[e] = x;
            }
            float4 hi, lo;
            split4(make_float4(v[0], v[1], v[2], v[3]), hi, lo);
            *reinterpret_cast<float4*>(b_hi + c * plane_bytes(nt) + row * 16) = hi;
            *reinterpret_cast<float4*>(b_lo + c * plane_bytes(nt) + row * 16) = lo;
          }
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&b_ready);
      }
    } else if (p.b_image != nullptr) {
      // large B: ONE bulk async copy per k-block of the image a prep kernel split beforehand
      if (lane == 0) {
        const uint32_t bytes = 2 * part_bytes(nt);
        const char* src = p.b_image + int64_t(tile_n) * p.n_kb * bytes;
        for (int t = 0; t < my_tiles; ++t) {
          for (int kb = 0; kb < p.n_kb; ++kb) {
            const int it = t * p.n_kb + kb;
            const int s = it % S, use = it / S;
            if (use > 0) mbar_wait(&empty_bar[s], (use - 1) & 1);
            mbar_arrive_expect_tx(&full_bar[s], bytes);
            bulk_g2s(smem + s * stage_sz + 2 * part_bytes(BM), src + int64_t(kb) * bytes, bytes, &full_bar[s]);
          }
        }
      }
    } else {
      // small B (a layer's weight matrix, a few KB, L2-resident): this warp splits the k-block's slice of
      // op(B) straight into the stage — no prep kernel, no extra launch on the step's dependency chain
      const int n_tile0 = tile_n * nt;
      for (int t = 0; t < my_tiles; ++t) {
        for (int kb = 0; kb < p.n_kb; ++kb) {
          const int it = t * p.n_kb + kb;
          const int s = it % S, use = it / S;
          if (use > 0) mbar_wait(&empty_bar[s], (use - 1) & 1);
          unsigned char* b_hi = smem + s * stage_sz + 2 * part_bytes(BM);
          unsigned char* b_lo = b_hi + part_bytes(nt);
          for (int i = lane; i < CHUNKS * nt; i += 32) {
            const int row = i % nt, c = i / nt;
            const int n = n_tile0 + row, k = kb * BK + c * 4;
            float v[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              float x = 0.f;
              if (n < p.N && k + e < p.K)
                x = p.transB ? __ldg(p.B + int64_t(n) * p.ldb + k + e) : __ldg(p.B + int64_t(k + e) * p.ldb + n);
              v[e] = x;
            }
            float4 hi, lo;
            split4(make_float4(v[0], v[1], v[2], v[3]), hi, lo);
            *reinterpret_cast<float4*>(b_hi + c * plane_bytes(nt) + row * 16) = hi;
            *reinterpret_cast<float4*>(b_lo + c * plane_bytes(nt) + row * 16) = lo;
          }
          fence_proxy_async();               // generic-proxy stores -> visible to the tensor core
          __syncwarp();
          if (lane == 0) mbar_arrive(&full_bar[s]);
        }
      }
    }
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kLoaderWarps) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_acc), "r"(uint32_t(p.tmem_cols)));
  }
}

struct Plan {
  bool ok;
  int nt, n_tiles, n_kb, stages, tmem_cols, n_acc, kb_per_acc, b_resident;
  size_t image_bytes, smem_bytes;
};

static Plan make_plan(int M, int N, int K, int nt_cap = kMaxNt) {
  Plan pl{};
  pl.ok = false;
  if (M <= 0 || N <= 0 || K <= 0) return pl;
  const int n16 = (N + 15) / 16 * 16;
  pl.nt = n16 <= nt_cap ? n16 : nt_cap;
  pl.n_tiles = (N + pl.nt - 1) / pl.nt;
  pl.n_kb = (K + BK - 1) / BK;
  pl.stages = pl.nt <= 64 ? 2 : (pl.nt <= 128 ? 3 : 2);
  if (pl.stages > pl.n_kb) pl.stages = pl.n_kb;
  pl.kb_per_acc = 4;                                   // 128 k per accumulator
  pl.n_acc = (pl.n_kb + pl.kb_per_acc - 1) / pl.kb_per_acc;
  if (2 * pl.n_acc * pl.nt > 512) {                    // TMEM has 512 columns; two accumulators per run
    pl.n_acc = 256 / pl.nt;
    pl.kb_per_acc = (pl.n_kb + pl.n_acc - 1) / pl.n_acc;
    pl.n_acc = (pl.n_kb + pl.kb_per_acc - 1) / pl.kb_per_acc;
  }
  const int cols = 2 * pl.n_acc * pl.nt;
  pl.tmem_cols = cols <= 32 ? 32 : cols <= 64 ? 64 : cols <= 128 ? 128 : cols <= 256 ? 256 : 512;
  pl.image_bytes = size_t(pl.n_tiles) * pl.n_kb * 2 * part_bytes(pl.nt);
  // resident B: the A ring is independent of n_kb (it keeps turning across the tiles of the persistent loop):
  // two stages when that lets two CTAs share an SM, else three if they fit
  const size_t b_bytes = size_t(pl.n_kb) * 2 * part_bytes(pl.nt);
  const size_t a_stage = 2 * size_t(part_bytes(BM));
  int res_stages = 0;
  if (2 * a_stage + b_bytes <= 110 * 1024) res_stages = 2;
  else if (3 * a_stage + b_bytes <= 200 * 1024) res_stages = 3;
  else if (2 * a_stage + b_bytes <= 200 * 1024) res_stages = 2;
  // residency pays when a CTA walks several M tiles; with one tile per CTA (M up to ~38 k rows) the k-block-wise
  // streaming of B lets the first MMA start one k-block earlier (measured: 1.2 us per launch at pose-0 size)
  const bool several_tiles = int64_t((M + BM - 1) / BM) * pl.n_tiles > 2 * 148;
  pl.b_resident = (res_stages > 0 && several_tiles) ? 1 : 0;
  if (pl.b_resident) pl.stages = res_stages;
  pl.smem_bytes = pl.b_resident ? size_t(pl.stages) * a_stage + b_bytes : size_t(pl.stages) * stage_bytes(pl.nt);
  pl.ok = pl.smem_bytes <= 200 * 1024;
  return pl;
}

}  // namespace tc
}  // namespace gn

using namespace gn;

static int tc_set_smem_attr() {
  static std::atomic<int> attr_set{0};
  if (!attr_set.load(std::memory_order_acquire)) {
    cudaError_t e =
        cudaFuncSetAttribute(tc::tc_gemm_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(tc::tc_gemm_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(tc::tc_gemm_kernel<3>, cudaFuncAttributePreferredSharedMemoryCarveout,
                               cudaSharedmemCarveoutMaxShared);
    // the products are HBM-bound streams of A: two CTAs per SM (smem <= 99 KB and <= 256 TMEM columns each for the
    // layer transforms) double the loads in flight, so ask for the largest shared-memory carveout
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(tc::tc_gemm_kernel<1>, cudaFuncAttributePreferredSharedMemoryCarveout,
                               cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      g_last_cuda_error.store(int(e), std::memory_order_relaxed);
      return GN_ERR_CUDA;
    }
    attr_set.store(1, std::memory_order_release);
  }
  return GN_OK;
}

// CTAs along M: persistent over the M tiles — as many CTAs as can be resident (two per SM when shared memory and
// TMEM allow it), each walking its tiles with a stride of the grid
static int tc_ctas_per_sm(const tc::Plan& pl) {
  return (2 * pl.smem_bytes <= 220 * 1024 && 2 * pl.tmem_cols <= 512) ? 2 : 1;
}

static unsigned tc_grid_x(int M, const tc::Plan& pl) {
  const int64_t m_tiles = ceil_div(M, tc::BM);
  const int per_sm = tc_ctas_per_sm(pl);
  int64_t resident = int64_t(148) * per_sm / pl.n_tiles;
  if (resident < 1) resident = 1;
  return unsigned(m_tiles < resident ? m_tiles : resident);
}

// deep prefetch when one CTA owns an SM and walks several M tiles (a long stream of A); PF = 1 otherwise
static int tc_launch(const tc::Plan& pl, int M, dim3 grid, const tc::Params& p, cudaStream_t st) {
  const bool deep = tc_ctas_per_sm(pl) == 1 && ceil_div(M, tc::BM) > int64_t(grid.x);
  if (deep) {
    GN_LAUNCH(tc::tc_gemm_kernel<3>, grid, tc::kThreads, pl.smem_bytes, st, p);
  } else {
    GN_LAUNCH(tc::tc_gemm_kernel<1>, grid, tc::kThreads, pl.smem_bytes, st, p);
  }
  return GN_OK;
}

// B small enough for the B-producer warp to split it inside the main kernel (one N tile, <= 16 float4 per lane
// and k-block): no prep launch.  Larger B (the [in, R*out] relation transform of pose-2) keeps the image.
static bool b_direct(const tc::Plan& pl) { return pl.n_tiles == 1 && pl.nt <= 64; }

extern "C" size_t gn_tc_gemm_workspace_bytes(int32_t M, int32_t N, int32_t K) {
  const tc::Plan pl = tc::make_plan(M, N, K);
  return pl.ok ? align_up(pl.image_bytes) : 0;
}

extern "C" int gn_tc_gemm(int transB, int32_t M, int32_t N, int32_t K, const float* A, int64_t lda, const float* B,
                          int64_t ldb, float* C, int64_t ldc, const float* addend, int64_t ld_addend,
                          const float* relu_mask, int64_t ld_mask, void* ws, size_t ws_bytes, void* stream) {
  if (M < 0 || N < 0 || K <= 0 || !A || !B || !C) return GN_ERR_ARG;
  if (M == 0 || N == 0) return GN_OK;
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  if (!al16(A) || lda % 4 != 0 || K % 4 != 0) return GN_ERR_ARG;            // 128-bit A loads
  if (!al16(C) || ldc % 4 != 0) return GN_ERR_ARG;                          // 128-bit C stores
  if (addend && (!al16(addend) || ld_addend % 4 != 0)) return GN_ERR_ARG;
  if (relu_mask && (!al16(relu_mask) || ld_mask % 4 != 0)) return GN_ERR_ARG;
  const tc::Plan pl = tc::make_plan(M, N, K);
  if (!pl.ok) return GN_ERR_ARG;
  const bool direct = b_direct(pl);
  if (!direct && (!ws || ws_bytes < pl.image_bytes || !al16(ws))) return GN_ERR_WORKSPACE;
  cudaStream_t st = as_stream(stream);
  if (!direct) {
    const int64_t total = int64_t(pl.n_tiles) * pl.n_kb * tc::CHUNKS * pl.nt;
    const tc::BView bv{B, ldb, 0, transB ? 1 : 0, 1};
    GN_LAUNCH(tc::b_image_kernel, (unsigned)ceil_div(total, 256), 256, 0, st, bv, K, N, pl.nt, pl.n_kb,
              static_cast<char*>(ws));
  }
  tc::Params p;
  p.M = M; p.N = N; p.K = K;
  p.A = A; p.lda = lda; p.C = C; p.ldc = ldc;
  p.addend = addend; p.ldd = ld_addend; p.mask = relu_mask; p.ldm = ld_mask;
  p.b_image = direct ? nullptr : static_cast<const char*>(ws);
  p.B = B; p.ldb = ldb; p.transB = transB ? 1 : 0;
  p.nt = pl.nt; p.n_kb = pl.n_kb; p.stages = pl.stages; p.tmem_cols = pl.tmem_cols;
  p.n_acc = pl.n_acc; p.kb_per_acc = pl.kb_per_acc; p.b_resident = pl.b_resident;
  GN_CHECK(tc_set_smem_attr());
  dim3 grid(tc_grid_x(M, pl), (unsigned)pl.n_tiles);
  GN_CHECK(tc_launch(pl, M, grid, p, st));
  return GN_OK;
}

// ---------------------------------------------------------------------------------------
// relation-batched feature transform of myRGCN on the tensor cores (north_star item 3):
//   Y[:, r, :] = X W[r]   for every relation r at once  ==  Y[M, R*f] = X[M, K] . W_flat[K, R*f]
// (gripnet/layers.py:171-189 evaluates it per edge as matmul(x_j[s:e], w[et]); transform-then-gather
// evaluates it once per NODE and relation).  W is stored [R][K][f]; the B image is built from that layout
// directly (BView mode 2), so no transposed copy of W exists.  The N tile is picked so that the grid can
// fill the GPU when M is only a few hundred rows (the task supervertex of the pose family has 645 nodes).
// ---------------------------------------------------------------------------------------
static int rel_nt_cap(int M, int N) {
  const int64_t m_tiles = ceil_div(M, tc::BM);
  int cap = tc::kMaxNt;
  while (cap > 32 && m_tiles * ceil_div(N, cap) < 148) cap >>= 1;
  return cap;
}

extern "C" size_t gn_tc_gemm_rel_workspace_bytes(int32_t M, int32_t n_rel, int32_t f, int32_t K) {
  const int64_t N = int64_t(n_rel) * f;
  if (N <= 0 || N >= (int64_t(1) << 31)) return 0;
  const tc::Plan pl = tc::make_plan(M, int(N), K, rel_nt_cap(M, int(N)));
  return pl.ok ? align_up(pl.image_bytes) : 0;
}

// The image of W_flat depends on the weights only: gn_tc_rel_image builds it (e.g. at the top of a training step, off
// the dependency chain), gn_tc_gemm_rel_image runs the product with a prepared image, gn_tc_gemm_rel does both.
extern "C" int gn_tc_rel_image(int32_t M, int32_t n_rel, int32_t f, int32_t K, const float* W, void* ws,
                               size_t ws_bytes, void* stream) {
  if (M < 0 || n_rel <= 0 || f <= 0 || K <= 0 || !W) return GN_ERR_ARG;
  if (M == 0) return GN_OK;
  const int64_t N64 = int64_t(n_rel) * f;
  if (N64 >= (int64_t(1) << 31)) return GN_ERR_RANGE;
  const int N = int(N64);
  if (K % 4 != 0) return GN_ERR_ARG;
  const tc::Plan pl = tc::make_plan(M, N, K, rel_nt_cap(M, N));
  if (!pl.ok) return GN_ERR_ARG;
  if (!ws || ws_bytes < pl.image_bytes || (reinterpret_cast<uintptr_t>(ws) & 15u) != 0) return GN_ERR_WORKSPACE;
  const int64_t total = int64_t(pl.n_tiles) * pl.n_kb * tc::CHUNKS * pl.nt;
  const tc::BView bv{W, int64_t(f), int64_t(K) * f, 2, f};
  GN_LAUNCH(tc::b_image_kernel, (unsigned)ceil_div(total, 256), 256, 0, as_stream(stream), bv, K, N, pl.nt, pl.n_kb,
            static_cast<char*>(ws));
  return GN_OK;
}

extern "C" int gn_tc_gemm_rel_image(int32_t M, int32_t n_rel, int32_t f, int32_t K, const float* X, int64_t ldx,
                                    const void* image, size_t image_bytes, float* Y, int64_t ldy, void* stream) {
  if (M < 0 || n_rel <= 0 || f <= 0 || K <= 0 || !X || !Y) return GN_ERR_ARG;
  if (M == 0) return GN_OK;
  const int64_t N64 = int64_t(n_rel) * f;
  if (N64 >= (int64_t(1) << 31)) return GN_ERR_RANGE;
  const int N = int(N64);
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  if (!al16(X) || ldx % 4 != 0 || K % 4 != 0 || !al16(Y) || ldy % 4 != 0) return GN_ERR_ARG;
  const tc::Plan pl = tc::make_plan(M, N, K, rel_nt_cap(M, N));
  if (!pl.ok) return GN_ERR_ARG;
  if (!image || image_bytes < pl.image_bytes || !al16(image)) return GN_ERR_WORKSPACE;
  tc::Params p;
  p.M = M; p.N = N; p.K = K;
  p.A = X; p.lda = ldx; p.C = Y; p.ldc = ldy;
  p.addend = nullptr; p.ldd = 0; p.mask = nullptr; p.ldm = 0;
  p.b_image = static_cast<const char*>(image);
  p.B = nullptr; p.ldb = f; p.transB = 0;
  p.nt = pl.nt; p.n_kb = pl.n_kb; p.stages = pl.stages; p.tmem_cols = pl.tmem_cols;
  p.n_acc = pl.n_acc; p.kb_per_acc = pl.kb_per_acc; p.b_resident = pl.b_resident;
  GN_CHECK(tc_set_smem_attr());
  dim3 grid(tc_grid_x(M, pl), (unsigned)pl.n_tiles);
  GN_CHECK(tc_launch(pl, M, grid, p, as_stream(stream)));
  return GN_OK;
}

extern "C" int gn_tc_gemm_rel(int32_t M, int32_t n_rel, int32_t f, int32_t K, const float* X, int64_t ldx,
                              const float* W, float* Y, int64_t ldy, void* ws, size_t ws_bytes, void* stream) {
  if (!X || !W || !Y) return GN_ERR_ARG;
  GN_CHECK(gn_tc_rel_image(M, n_rel, f, K, W, ws, ws_bytes, stream));
  return gn_tc_gemm_rel_image(M, n_rel, f, K, X, ldx, ws, ws_bytes, Y, ldy, stream);
}
