/*
 * gripnet_b200 — C ABI of the B200-native GripNet message-passing hot path.
 *
 * The reference (NYXFLOWER/GripNet) is pure Python and has no FFI of its own: its
 * boundary for this path is the gripnet.layers / gripnet.decoder module API
 * (SURVEY.md §8b).  This header is the NEW boundary inserted beneath that API.
 * Each entry point names the reference lines whose arithmetic it replaces
 * (paths relative to the reference checkout).  INTEGRATION.md shows the ctypes
 * binding a maintainer of the reference would add.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless it says "host"; the caller owns all
 *    memory (incl. workspaces); the library never allocates or frees device
 *    memory, keeps no per-call global state and never synchronises the device.
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, so
 *    every call is CUDA-graph capturable.
 *  - features are fp32 row-major with an explicit leading dimension (`ld*`, in
 *    floats) so column slices of a concatenated buffer can be read and written
 *    in place.
 *  - return value: 0 on success, a negative gn_status otherwise
 *    (gn_error_string() for text).  No CPU fallback exists: without a CUDA
 *    device every compute entry point fails with GN_ERR_CUDA.
 *  - re-entrant: safe to call from the Python main thread (forward) and from
 *    autograd's device worker thread (backward) concurrently.
 */
#ifndef GRIPNET_B200_H
#define GRIPNET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  GN_OK = 0,
  GN_ERR_ARG = -1,       /* bad size / null pointer / misaligned buffer          */
  GN_ERR_RANGE = -2,     /* size does not fit the int32 index space (>= 2^31)    */
  GN_ERR_WORKSPACE = -3, /* workspace too small                                  */
  GN_ERR_CUDA = -4       /* a CUDA runtime call or kernel launch failed          */
} gn_status;

int gn_version(void);
const char* gn_error_string(int status);
/* cudaError_t (and its runtime text) of the most recent launch of this library that failed with
 * GN_ERR_CUDA; 0 / "no error" when none has */
int gn_last_cuda_error(void);
const char* gn_last_cuda_error_string(void);
/* number of kernels this library has launched in this process (monotonic) */
uint64_t gn_launch_count(void);

/* ------------------------------------------------------------------------- */
/* CSR with a row-split work list ("chunks") for load-balanced, atomic-free   */
/* row reductions.  All arrays are device pointers.                           */
/* ------------------------------------------------------------------------- */
typedef struct {
  int32_t n_rows;          /* output rows                                           */
  int32_t n_cols;          /* rows of the gathered operand                           */
  int32_t nnz;             /* stored entries (host copy; may be an upper bound)      */
  int32_t chunk_len;       /* max entries per chunk                                  */
  int32_t n_chunks;        /* chunks to launch (exact or an upper bound)             */
  int32_t flags;           /* GN_CSR_ROW_IS_CHUNK: every row is exactly one chunk (chunk i == row i, n_chunks ==
                              n_rows, known exactly on the host): kernels then take the row bounds from rowptr
                              alone and skip the chunk tables (one dependent round trip less per warp)      */
  const int32_t* rowptr;   /* [n_rows+1]                                             */
  const int32_t* col;      /* [nnz] gathered-row index                               */
  const float* val;        /* [nnz] per-entry coefficient, or NULL for all-ones      */
  const int32_t* chunk_ptr;/* [n_rows+1] first chunk of each row; [n_rows] = total   */
  const int32_t* chunk_row;/* [n_chunks] row of each chunk                           */
  const int32_t* chunk_beg;/* [n_chunks] first entry of each chunk                   */
  int32_t* row_counter;    /* [n_rows] zero-initialised; left zero by every call     */
} gn_csr;
enum { GN_CSR_ROW_IS_CHUNK = 1 };

/* ---- K1: graph preprocessing ------------------------------------------- */

/* Stable counting (LSD radix) sort of int32 keys in [0, 2^key_bits): rowptr by
 * histogram + exclusive scan, perm[k] = original position of the entry in slot k.
 * Replaces nothing 1:1 in the reference; it is the building block that turns
 * edge_index into the dst-sorted CSR and its transpose (north_star item 1). */
size_t gn_csr_from_keys_workspace_bytes(int64_t n, int32_t n_rows);
int gn_csr_from_keys(const int32_t* keys, int64_t n, int32_t n_rows,
                     int32_t* rowptr /*[n_rows+1]*/, int32_t* perm /*[n]*/,
                     void* ws, size_t ws_bytes, void* stream);

/* out[i] = rowptr[r0+i] - rowptr[r0], i in [0, n_rows]: rows [r0, r0+n_rows) of a CSR as a
 * stand-alone CSR — the per-rank slice of a destination-partitioned graph (new design: the
 * reference has no multi-GPU path, SURVEY.md §8e). */
int gn_rowptr_slice(const int32_t* rowptr, int32_t r0, int32_t n_rows, int32_t* out, void* stream);

/* Row-split work list for a CSR: a row of length L gets max(1, ceil(L/chunk_len))
 * chunks.  n_chunks_out (device int32) receives the total. */
size_t gn_build_chunks_workspace_bytes(int32_t n_rows);
int gn_build_chunks(const int32_t* rowptr, int32_t n_rows, int32_t chunk_len,
                    int32_t* chunk_ptr /*[n_rows+1]*/, int32_t* chunk_row, int32_t* chunk_beg,
                    int64_t chunk_capacity, int32_t* row_counter /*[n_rows] zeroed here, or NULL*/,
                    void* ws, size_t ws_bytes, void* stream);

/* GCN normalisation + CSR pair.  Replaces gripnet/layers.py:52-69 (myGCN.norm):
 * PyG add_remaining_self_loops, scatter_add degree by TARGET, deg^-1/2 (inf->0),
 * norm_e = (dis[row]*w)*dis[col].
 *   bipartite == 0: square graph over n_dst (== n_src) nodes, self-loop rewrite.
 *   bipartite == 1: interGraph's stacked graph (layers.py:363-368) in closed form:
 *                   rows = targets, cols = sources, deg_t = 1 + sum w, no loop entries.
 * Outputs (capacity E + n_dst each unless noted):
 *   aug_src/aug_dst/aug_norm : the reference-order augmented edge list (int64/fp32);
 *                              may be NULL when only the CSR is wanted
 *   rowptr/col/val/perm      : dst-sorted CSR  (perm -> position in the augmented list)
 *   rowptr_t/col_t/val_t/perm_t : src-sorted (transpose) CSR
 *   deg [n_dst] fp32 weighted in-degree incl. loop, indeg [n_dst] int32 entry count
 *   counts (device int32[4]) : {E_aug, n_self_loops_removed, 0, 0}                  */
size_t gn_gcn_prep_workspace_bytes(int64_t n_edges, int32_t n_src, int32_t n_dst);
int gn_gcn_prep(const int64_t* src, const int64_t* dst, const float* weight /*or NULL*/,
                int64_t n_edges, int32_t n_src, int32_t n_dst, int bipartite, float fill_value,
                int64_t* aug_src, int64_t* aug_dst, float* aug_norm,
                int32_t* rowptr, int32_t* col, float* val, int32_t* perm,
                int32_t* rowptr_t, int32_t* col_t, float* val_t, int32_t* perm_t,
                float* deg, int32_t* indeg, int32_t* counts,
                void* ws, size_t ws_bytes, void* stream);

/* ---- K1 for destination-partitioned graphs (SURVEY.md §8e; new design: the reference is single-device) ----
 * Every rank builds only ITS rows of the dst-sorted CSR (forward) and of the src-sorted transpose CSR
 * (backward); results are bit-identical to the matching rows of gn_gcn_prep's global CSR.
 *
 * gn_edge_filter: order-preserving selection of the edges whose destination (by_src == 0) or source
 * (by_src != 0) lies in [lo, hi).  count (device int32) receives the number selected; with out_src ==
 * NULL only the count is produced (size the outputs, then call again).  out_index (optional) receives
 * index_base + original position.  n_edges < 2^31 per call: longer lists are filtered chunk by chunk. */
size_t gn_edge_filter_workspace_bytes(int64_t n_edges);
int gn_edge_filter(const int64_t* src, const int64_t* dst, const float* weight /*or NULL*/, int64_t n_edges,
                   int by_src, int64_t lo, int64_t hi, int64_t* out_src, int64_t* out_dst,
                   float* out_weight /*or NULL*/, int64_t* out_index /*or NULL*/, int64_t index_base,
                   int32_t* count, void* ws, size_t ws_bytes, void* stream);
/* gn_gcn_part_structure: rows [row0, row0 + n_rows) of the CSR keyed by `key_end` (destinations for the
 * forward CSR, sources for the transpose) from a shard in which every key_end lies in that block;
 * `other_end` ids are global.  with_loops: the self-loop rewrite of gripnet/layers.py:52-60 restricted to
 * the block (loop entry = last slot of each row, column row0 + i, weight = that of the last listed
 * self-loop or fill_value).  Outputs: rowptr [n_rows + 1], col / val [n_edges + n_rows] (val holds the
 * per-entry WEIGHT), counts[0] = stored entries; dis / deg [n_rows] (dis != NULL): weighted in-degree in
 * list order and its -1/2 power (inf -> 0) — meaningful for the destination-keyed build
 * (with_loops == 0: the bipartite closed form, deg = 1 + sum w).
 * gn_gcn_part_values: val <- (dis_src[source] * w) * dis_dst[target] (layers.py:66-69) with GLOBAL deg^-1/2
 * vectors (all-gathered by the caller); dis_src == NULL means 1 (bipartite); transpose: rows are sources. */
size_t gn_gcn_part_workspace_bytes(int64_t n_edges, int32_t n_rows);
int gn_gcn_part_structure(const int64_t* key_end, const int64_t* other_end, const float* weight /*or NULL*/,
                          int64_t n_edges, int32_t row0, int32_t n_rows, int with_loops, float fill_value,
                          int32_t* rowptr, int32_t* col, float* val, float* deg /*or NULL*/, float* dis /*or NULL*/,
                          int32_t* counts, void* ws, size_t ws_bytes, void* stream);
int gn_gcn_part_values(const int32_t* rowptr, const int32_t* col, int32_t n_rows, int32_t row0,
                       const float* dis_src /*or NULL*/, const float* dis_dst, int transpose, float* val,
                       void* stream);

/* Multi-relational prep.  Replaces the structure implied by gripnet/layers.py:165-189
 * (relation of edge e = index of the range_list slice containing e; edge_type unused)
 * and PyG aggr="mean" (joint in-degree over all relations).
 *   fwd CSR : rows = targets, col = src*n_rel + rel, no val (row scale 1/max(1,c_i))
 *   bwd CSR : rows = src*n_rel + rel, col = target, val = 1/max(1,c_target)          */
size_t gn_rgcn_prep_workspace_bytes(int64_t n_edges, int32_t n_nodes, int32_t n_rel);
int gn_rgcn_prep(const int64_t* src, const int64_t* dst, int64_t n_edges,
                 const int64_t* range_list /*[n_rel,2]*/, int32_t n_nodes, int32_t n_rel,
                 int32_t* rowptr, int32_t* col, int32_t* perm, float* inv_cnt /*[n_nodes]*/,
                 int32_t* rowptr_t /*[n_nodes*n_rel+1]*/, int32_t* col_t, float* val_t, int32_t* perm_t,
                 void* ws, size_t ws_bytes, void* stream);

/* CSR of an index list (rows = nodes, entries = positions in the list) for the
 * deterministic backward of z[node_list] (gripnet/decoder.py:42). */
size_t gn_index_prep_workspace_bytes(int64_t n, int32_t n_nodes);
int gn_index_prep(const int64_t* index, int64_t n, int32_t n_nodes,
                  int32_t* rowptr, int32_t* perm, void* ws, size_t ws_bytes, void* stream);

/* ---- K3/K4/K5/K7/K8: SpMM  ---------------------------------------------- */
/* out[i, 0:F] = act( row_scale[i] * sum_{k in row i} val[k] * x[col[k], 0:F]
 *                    + bias + addend[i] )
 * Replaces MessagePassing.propagate + message + update at gripnet/layers.py:92-100
 * (GCN, aggr="add"), :167 + :191-197 (RGCN, aggr="mean" via row_scale, root term via
 * addend) and the ReLU at :279/:305/:370.  Backward passes call it with the
 * transpose CSR.  Warp per chunk, 128-bit gathers, no atomics on data: rows split
 * over several chunks are combined in a fixed order by the last-arriving warp.
 * partial: [n_chunks, F] fp32 scratch (may be NULL when no row has > 1 chunk). */
int gn_spmm(const gn_csr* csr, const float* x, int64_t ldx, int32_t F,
            const float* row_scale, const float* bias, const float* addend, int64_t ld_addend,
            int relu, float* out, int64_t ldo, float* partial, void* stream);

/* ---- K2/K6: dense transforms (fp32 FFMA, CUDA cores)  --------------------- */
/* C[b] = epilogue( alpha * op(A[b]) * op(B[b]) ), b in [0,batch):
 *   op(A) is M x K (transA: stored K x M), op(B) is K x N (transB: stored N x K);
 *   batch_reduce != 0: a single C = sum_b op(A[b]) op(B[b]);
 *   a_rows != NULL: row r of the STORED A is fetched from A + a_rows[r]*lda (row gather);
 *   epilogue: (+ C if accumulate) (+ addend) then zero where relu_mask <= 0.
 *   split_k != 0: when the output tiles alone cannot fill the GPU, the flattened
 *   (batch-to-reduce, K) reduction is cut into slices whose partial products are
 *   summed in slice order from `ws` (deterministic, no atomics); `ws` must hold
 *   gn_sgemm_workspace_bytes(M, N, K, batch, batch_reduce) bytes (0 = no split).
 * Replaces torch.matmul at gripnet/layers.py:73, :172, :181, :193, :383 and
 * gripnet/decoder.py:42, and their autograd transposes. */
size_t gn_sgemm_workspace_bytes(int32_t M, int32_t N, int32_t K, int32_t batch, int batch_reduce);
int gn_sgemm(int transA, int transB, int32_t M, int32_t N, int32_t K,
             const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
             int32_t batch, int64_t strideA, int64_t strideB, int64_t strideC, int batch_reduce,
             float alpha, int accumulate, const float* addend, int64_t ld_addend,
             const float* relu_mask, int64_t ld_mask, const int64_t* a_rows,
             int32_t split_k, float* ws, size_t ws_bytes, void* stream);

/* ---- K2/K6 tensor path: tcgen05 (kind::tf32) with 3xTF32 error compensation -- */
/* C = epilogue( A[M,K] * op(B) ),  op(B) = B [K,N] (transB == 0) or B^T with B stored [N,K].
 * Each operand element is split hi + lo in TF32 while it is staged and three MMAs per k-step
 * accumulate lo*hi + hi*lo + hi*hi in one fp32 TMEM accumulator: fp32-grade accuracy
 * (the 1e-5 parity bar) on the tensor cores.  Requirements: 16-byte aligned A / C / addend /
 * mask with leading dimensions and K multiples of 4.  `ws` (gn_tc_gemm_workspace_bytes) holds
 * the pre-split shared-memory image of B.  Epilogue: (+ addend) then zero where relu_mask <= 0.
 * Replaces torch.matmul at gripnet/layers.py:73 / :181 and its dX transpose for large M. */
size_t gn_tc_gemm_workspace_bytes(int32_t M, int32_t N, int32_t K);
int gn_tc_gemm(int transB, int32_t M, int32_t N, int32_t K, const float* A, int64_t lda,
               const float* B, int64_t ldb, float* C, int64_t ldc,
               const float* addend, int64_t ld_addend, const float* relu_mask, int64_t ld_mask,
               void* ws, size_t ws_bytes, void* stream);

/* Relation-batched feature transform of myRGCN on the tensor cores (north_star item 3):
 *   Y[:, r, :] = X W[r] for all r  ==  Y[M, n_rel*f] = X[M, K] . W_flat[K, n_rel*f],   W stored [n_rel][K][f]
 * (gripnet/layers.py:171-189 evaluates matmul(x_j[s:e], w[et]) per EDGE; here it is once per node and
 * relation, then the segmented SpMM gathers rows of Y).  Same 3xTF32 kernel and accuracy as gn_tc_gemm; the
 * shared-memory image of W_flat is built straight from the [n_rel][K][f] layout into `ws`
 * (gn_tc_gemm_rel_workspace_bytes).  Requirements: X / Y 16-byte aligned, ldx, ldy, K multiples of 4. */
size_t gn_tc_gemm_rel_workspace_bytes(int32_t M, int32_t n_rel, int32_t f, int32_t K);
int gn_tc_gemm_rel(int32_t M, int32_t n_rel, int32_t f, int32_t K, const float* X, int64_t ldx,
                   const float* W, float* Y, int64_t ldy, void* ws, size_t ws_bytes, void* stream);
/* The two halves of gn_tc_gemm_rel: the image depends on W only, so a training step builds it up front, off its
 * dependency chain (gn_tc_rel_image, `ws` of gn_tc_gemm_rel_workspace_bytes for the SAME M), and the product then
 * runs with the prepared image (gn_tc_gemm_rel_image). */
int gn_tc_rel_image(int32_t M, int32_t n_rel, int32_t f, int32_t K, const float* W, void* ws, size_t ws_bytes,
                    void* stream);
int gn_tc_gemm_rel_image(int32_t M, int32_t n_rel, int32_t f, int32_t K, const float* X, int64_t ldx,
                         const void* image, size_t image_bytes, float* Y, int64_t ldy, void* stream);

/* Weight-gradient products on the tensor cores: C[Mo, No] = A^T B with A [n, Mo], B [n, No] (features contiguous,
 * the reduction runs over the n node rows): dW = H_{l-1}^T dY of a GCN layer (autograd of gripnet/layers.py:73)
 * and, with c_inner = f and c_stride = k*f, dW[r] = X^T dY[:, r, :] for every relation at once, written in the
 * [R][k][f] layout of the relational weights (layers.py:171-189).  3xTF32 with fp32 running sums in registers
 * (the TMEM accumulator is drained every 128 rows); rows are split over CTAs and the split partials are added in
 * split order.  c_inner == 0: C row-major with leading dimension ldc.  Requirements: A / B 16-byte aligned, lda,
 * ldb, Mo, No multiples of 4; `ws` holds gn_tc_tn_workspace_bytes(n, Mo, No) bytes. */
size_t gn_tc_tn_workspace_bytes(int64_t n, int32_t Mo, int32_t No);
int gn_tc_tn(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t n, int32_t Mo, int32_t No,
             float* C, int64_t ldc, int32_t c_inner, int64_t c_stride, void* ws, size_t ws_bytes, void* stream);

/* ---- K9/K10: DistMult decoder  ------------------------------------------- */
/* score_e = sum_k z[src_e,k] z[dst_e,k] w[rel_e,k]; sigmoid optional.
 * Replaces gripnet/decoder.py:19-23 (three [E,D] gathers + two muls + sum). */
int gn_distmult_fwd(const float* z, int64_t ldz, int32_t D, const float* w,
                    const int64_t* src, const int64_t* dst, const int64_t* etype, int64_t n_edges,
                    int sigmoid, float* out, void* stream);
/* per-edge upstream coefficient g_e = grad_e * (sigmoid ? s(1-s) : 1) */
int gn_distmult_coef(const float* grad_out, const float* out, int64_t n_edges, int sigmoid,
                     float* coef, void* stream);
/* K10 in ONE gather pass.  gn_pair_prep groups the 2E endpoint entries of an edge list by (node, relation):
 * pair_rowptr [n_nodes * n_rel + 1] (row = node * n_rel + rel), entries (other endpoint, edge id) in their
 * original relative order (stable sort).  gn_distmult_bwd_pairs walks it once:
 *   T[n, r, :] = sum over the entries of pair row (n, r) of coef[e] * z[other]      (T: [n_nodes*n_rel, D])
 * and gn_distmult_grads finishes both gradients from T (plus an optional second T2 of another edge list,
 * e.g. the negatives of the same step) without touching the edges again:
 *   dz[n] = sum_r T[n,r] .* w[r],      dw[r] = 1/2 sum_n z[n] .* T[n,r]
 * (every edge sits in the pair rows of both of its endpoints, hence the 1/2; D <= 1024; `ws` holds
 * gn_distmult_grads_workspace_bytes: per-relation slab partials of dw + arrival counters).  Replaces the autograd of
 * gripnet/decoder.py:19-23 (three index_put scatters); atomic-free, fixed summation order. */
size_t gn_pair_prep_workspace_bytes(int64_t n_edges);
int gn_pair_prep(const int64_t* src, const int64_t* dst, const int64_t* etype, int64_t n_edges, int32_t n_nodes,
                 int32_t n_rel, int32_t* pair_rowptr, int32_t* ent_other, int32_t* ent_eid /*[2E]*/,
                 void* ws, size_t ws_bytes, void* stream);
int gn_distmult_bwd_pairs(const gn_csr* pair_csr, const int32_t* ent_other, const int32_t* ent_eid,
                          const float* coef, const float* z, int64_t ldz, int32_t D, float* T, float* partial,
                          void* stream);
size_t gn_distmult_grads_workspace_bytes(int32_t n_nodes, int32_t n_rel, int32_t D);
int gn_distmult_grads(const float* T, const float* T2 /*or NULL*/, int32_t n_nodes, int32_t n_rel, int32_t D,
                      const float* z, int64_t ldz, const float* w, float* dz /*or NULL*/, int64_t lddz,
                      float* dw /*or NULL*/, void* ws, size_t ws_bytes, void* stream);

/* ---- K11: multi-class decoder pieces  ------------------------------------ */
/* row softmax over C columns (gripnet/decoder.py:43) and its backward */
int gn_softmax_fwd(const float* logits, int64_t n, int32_t C, float* out, void* stream);
int gn_softmax_bwd(const float* out, const float* grad_out, int64_t n, int32_t C, float* grad_logits,
                   void* stream);

/* ---- elementwise / reductions used by the layer stacks  ------------------- */
enum { GN_EW_COPY = 0, GN_EW_ABS = 1, GN_EW_RELU = 2, GN_EW_ADD = 3 /* dst += src */ };
/* dst[i, 0:F] = op(src[i, 0:F])  (torch.cat / torch.abs at layers.py:309, :376) */
int gn_map2d(int op, const float* src, int64_t lds, float* dst, int64_t ldd, int64_t n, int32_t F,
             void* stream);
/* dst = g where y > 0 else 0   (ReLU backward, layers.py:279/305/370) */
int gn_relu_bwd(const float* g, int64_t ldg, const float* y, int64_t ldy, float* dst, int64_t ldd,
                int64_t n, int32_t F, void* stream);
/* dst (+)= g * sign(t)         (backward of torch.abs, layers.py:376/379) */
int gn_abs_bwd(const float* g, int64_t ldg, const float* t, int64_t ldt, float* dst, int64_t ldd,
               int64_t n, int32_t F, float scale, void* stream);
/* dst = alpha * a + beta * b  (b may be NULL; dst may alias a or b)
 * — the (x + u) / 2 mixes of interGraph, layers.py:379/382-384 */
int gn_axpby(const float* a, int64_t lda, float alpha, const float* b, int64_t ldb, float beta,
             float* dst, int64_t ldd, int64_t n, int32_t F, void* stream);
/* zero-fill (stream-ordered memset; gradient rows no kernel writes) */
int gn_zero(void* p, size_t bytes, void* stream);
/* dst = ((a + b) + c) / 3 — the three-way mix of the freebase-d model, GripNet-freebase-d.py:160-161
 * (same association order, true division) */
int gn_mean3(const float* a, int64_t lda, const float* b, int64_t ldb, const float* c, int64_t ldc,
             float* dst, int64_t ldd, int64_t n, int32_t F, void* stream);
/* out[0:F] = sum_i x[i, 0:F], deterministic two-level reduction; ws >= gn_colsum_workspace_bytes */
size_t gn_colsum_workspace_bytes(int64_t n, int32_t F);
int gn_colsum(const float* x, int64_t ldx, int64_t n, int32_t F, float* out, void* ws, size_t ws_bytes,
              void* stream);
/* fused link-prediction loss (GripNet-pose.py:140-142):
 *   loss = -mean(log(pos+eps)) - mean(log(1-neg+eps)); deterministic two-level sum.
 * backward reads the upstream gradient from DEVICE memory (no host sync). */
size_t gn_loss_workspace_bytes(int64_t n);
int gn_lp_loss_fwd(const float* pos, int64_t n_pos, const float* neg, int64_t n_neg, float eps,
                   float* loss /*[1]*/, void* ws, size_t ws_bytes, void* stream);
int gn_lp_loss_bwd(const float* pos, int64_t n_pos, const float* neg, int64_t n_neg, float eps,
                   const float* grad_loss /*[1]*/, float* grad_pos, float* grad_neg, void* stream);
/* fused node-classification loss (GripNet-aminer.py:133):
 *   loss = -mean(log(score[i, label_i] + eps)) */
int gn_nc_loss_fwd(const float* score, int64_t n, int32_t C, const int64_t* label, float eps,
                   float* loss /*[1]*/, void* ws, size_t ws_bytes, void* stream);
int gn_nc_loss_bwd(const float* score, int64_t n, int32_t C, const int64_t* label, float eps,
                   const float* grad_loss /*[1]*/, float* grad_score, void* stream);

/* ---- K13: negative sampling on the device (SURVEY.md §8f) ---------------------------------- */
/* Replaces gripnet/utils.py:98-112 (negative_sampling) and :115-119 (typed_negative_sampling): one
 * uniformly random non-positive node pair per positive edge.  `range_list` ([n_rel,2] int64, ascending
 * contiguous half-open slices, DEVICE) selects the typed rule (reject only pairs that are positive in
 * the edge's own slice); NULL / n_rel == 0 rejects against all positives.
 *   gn_negsample_build : hash the positives into `table` (gn_negsample_table_bytes(n_edges) bytes), once.
 *   gn_negsample_draw  : one draw per edge into neg_src / neg_dst (int64 [n_edges]).  Draw `a` of edge e in
 *                        epoch t = Philox4x32-10(counter (e_lo, e_hi, a, t), key seed); pair code =
 *                        mulhi64(x0 | x1 << 32, N^2).  `state` = u64[2], zero-initialised: state[0] is the
 *                        epoch, read by the kernel and advanced by it (CUDA-graph replays keep drawing new
 *                        negatives), state[1] is scratch.  Bit-exact restatement: oracle/negsample.py. */
size_t gn_negsample_table_bytes(int64_t n_edges);
int gn_negsample_build(const int64_t* src, const int64_t* dst, int64_t n_edges, int64_t n_nodes,
                       const int64_t* range_list, int32_t n_rel, void* table, size_t table_bytes, void* stream);
int gn_negsample_draw(const void* table, size_t table_bytes, int64_t n_edges, int64_t n_nodes,
                      const int64_t* range_list, int32_t n_rel, uint64_t seed, uint64_t* state,
                      int64_t* neg_src, int64_t* neg_dst, void* stream);

/* ---- K14: fused multi-tensor Adam (SURVEY.md §8f rank 2) -------------------------------------- */
/* Replaces torch.optim.Adam(model.parameters(), lr).step() of the training scripts
 * (GripNet-pose.py:104,146; GripNet-aminer.py:113,135; amsgrad = False):
 *   g' = g + weight_decay * p;  m += (g' - m)(1 - beta1);  v = v beta2 + (1 - beta2) g'^2;
 *   p -= lr / (1 - beta1^t) * m / (sqrt(v) / sqrt(1 - beta2^t) + eps),   t = step[0] + 1.
 * `tensors` is a HOST array (the descriptors travel in the kernel-parameter block, up to
 * gn_adam_max_tensors_per_launch() per launch); all pointers inside are DEVICE pointers to contiguous
 * fp32 arrays of n elements.  Hyper-parameters are doubles (torch evaluates 1 - beta and the bias corrections
 * in double before casting).  `step` is a DEVICE u64, zero-initialised by the caller, read by the
 * kernels and advanced by one at the end of the call: replays of a captured CUDA graph are successive
 * optimiser steps. */
typedef struct {
  float* param;
  const float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  int64_t n;
} gn_adam_tensor;
int gn_adam_max_tensors_per_launch(void);
int gn_adam_step(const gn_adam_tensor* tensors /*host*/, int32_t n_tensors, double lr, double beta1, double beta2,
                 double eps, double weight_decay, uint64_t* step, void* stream);

/* ---- K15: evaluation metrics on the device (SURVEY.md §8f rank 3) ------------------------------ */
/* Per-relation AUPRC / AUROC / AP of a link-prediction epoch.  Replaces the host loop of
 * GripNet-pose.py:148-164 and :188-199 around gripnet/utils.py:28-35 (sklearn roc_auc_score,
 * average_precision_score, auc(precision_recall_curve)).  Relation r scores the positives
 * pos_score[pos_range[r,0] : pos_range[r,1]] against the negatives neg_score[neg_range[r,0] :
 * neg_range[r,1]] (neg_range == NULL: the same slices, as the reference does).  Ranges are DEVICE int64
 * [n_rel,2], ascending and non-overlapping.  record: DEVICE double [3, n_rel], rows = auprc, auroc, ap
 * (the reference's `record` layout, GripNet-pose.py:148); NaN where the metric is undefined (a relation
 * without positives; AUROC also without negatives).  Tied scores form one threshold, as in sklearn. */
size_t gn_lp_metrics_workspace_bytes(int64_t n_pos, int64_t n_neg, int32_t n_rel);
int gn_lp_metrics(const float* pos_score, int64_t n_pos, const float* neg_score, int64_t n_neg,
                  const int64_t* pos_range, const int64_t* neg_range, int32_t n_rel, double* record,
                  void* ws, size_t ws_bytes, void* stream);
/* out[i] = index of the first maximum of row i (torch.argmax(score, dim=1), GripNet-aminer.py:131) */
int gn_argmax_rows(const float* x, int64_t ldx, int64_t n, int32_t C, int64_t* out, void* stream);
/* out (DEVICE double[3]) = {micro-F1, macro-F1, accuracy} of integer class predictions
 * (gripnet/utils.py:38-52: sklearn f1_score micro / macro over the classes present, accuracy_score).
 * NaN if a label lies outside [0, C). */
size_t gn_nc_metrics_workspace_bytes(int32_t C);
int gn_nc_metrics(const int64_t* target, const int64_t* pred, int64_t n, int32_t C, double* out,
                  void* ws, size_t ws_bytes, void* stream);

/* ---- K16: filtered candidate ranking and top-k of the DistMult decoder --------------------------- */
/* New capability (the reference evaluates each positive against ONE sampled negative, GripNet-pose.py:148-164).
 * Every candidate tail c in [0, n) of a query (s, r), c == s included, is scored with the PRE-sigmoid DistMult
 * score S(c) = sum_k z[s,k] w[r,k] z[c,k], evaluated as one row of S = Q . z^T with Q[g] = z[s_g] .* w[r_g]
 * (gn_rank_query_rows, then the dense product gn_sgemm / gn_tc_gemm with transB = 1).  Only tail queries
 * (s, r, ?) are ranked: lists holding both directions of every pair rank the head through the mirrored edge.
 *
 * gn_rank_csr: one-sided grouped structure of an edge list — rowptr [n_nodes*n_rel + 1] (row s*n_rel + r), entries
 *   ent_dst / ent_eid [E] (candidate, edge id) sorted by candidate inside a row (two stable counting sorts).  A
 *   FILTER (the set of directed known positives (s, r, c), e.g. train + test) is the structure of the concatenated
 *   filter lists; duplicates stay stored and are skipped where they are read.  group_row / n_groups (both or
 *   neither): the ids of the non-empty rows in ascending order ("groups", capacity n_nodes*n_rel) and their count
 *   (device int32).
 * gn_rank_query_rows: q[i, 0:D] = z[s_i] .* w[r_i], with (s_i, r_i) taken from group_row[i] = s*n_rel + r, or, when
 *   group_row is NULL, from node[i] / rel[i].
 * gn_rank_count: filtered rank of every target of groups [0, n_groups) whose score rows are S[g] (leading dimension
 *   lds >= n_nodes; group_row points at the first group of the chunk).  OGB rule: with the negatives
 *   N = {c != t : (s, r, c) not in the filter}, opt = #{c in N : S(c) > S(t)}, pess = #{c in N : S(c) >= S(t)},
 *   rank[edge id] = 1 + (opt + pess) / 2 (float32).  S(t) is read from the same row as every S(c).  f_rowptr ==
 *   NULL: no filter.
 * gn_rank_metrics: out (DEVICE double [1 + n_hits, n_rel]) = MRR = mean(1/rank) and Hits@k = mean(rank <= k) per
 *   relation over the edges rel_perm[rel_rowptr[r] : rel_rowptr[r+1]] (gn_index_prep of the edge types); NaN for a
 *   relation without edges.  hits_k is a HOST array of at most gn_rank_max_hits() entries (it travels in the
 *   kernel-parameter block: capturable).  Fixed-order float64 sums: repeated calls are bit-identical.
 * gn_rank_topk: the k (1 <= k <= 256) highest-scoring candidates c with (node[i], rel[i], c) not in the filter, for
 *   every query row i of S (overwritten: filtered entries are marked in place).  Order: descending pre-sigmoid
 *   score, ties by smaller id.  out_score / out_id [count, k]: score (sigmoid applied when `sigmoid`) and id; id -1
 *   and score NaN pad a query with fewer than k admissible candidates. */
size_t gn_rank_csr_workspace_bytes(int64_t n_edges, int32_t n_nodes, int32_t n_rel);
int gn_rank_csr(const int64_t* src, const int64_t* dst, const int64_t* etype, int64_t n_edges, int32_t n_nodes,
                int32_t n_rel, int32_t* rowptr, int32_t* ent_dst, int32_t* ent_eid, int32_t* group_row /*or NULL*/,
                int32_t* n_groups /*or NULL*/, void* ws, size_t ws_bytes, void* stream);
int gn_rank_query_rows(const float* z, int64_t ldz, int32_t D, const float* w, int32_t n_rel, const int32_t* group_row,
                       const int64_t* node, const int64_t* rel, int64_t count, float* q, int64_t ldq, void* stream);
int gn_rank_count(const float* S, int64_t lds, int32_t n_nodes, const int32_t* group_row, int32_t n_groups,
                  const int32_t* q_rowptr, const int32_t* q_dst, const int32_t* q_eid,
                  const int32_t* f_rowptr /*or NULL*/, const int32_t* f_dst, float* rank, void* stream);
int gn_rank_max_hits(void);
int gn_rank_metrics(const float* rank, const int32_t* rel_rowptr, const int32_t* rel_perm, int32_t n_rel,
                    const int32_t* hits_k /*host*/, int32_t n_hits, double* out, void* stream);
int gn_rank_topk(float* S, int64_t lds, int32_t n_nodes, int32_t n_rel, const int64_t* node, const int64_t* rel,
                 int64_t count, const int32_t* f_rowptr /*or NULL*/, const int32_t* f_dst, int32_t k, int sigmoid,
                 float* out_score, int64_t* out_id, void* stream);

/* Relation queries (s, ?, t) of a directed pair: every relation r' in [0, n_rel) is a candidate, scored with the
 * PRE-sigmoid S(r') = sum_k z[s,k] z[t,k] w[r',k], one row of S = P . W^T with P[g] = z[s_g] .* z[t_g]
 * (gn_rank_pair_rows, then gn_sgemm / gn_tc_gemm with transB = 1; W the decoder weight [n_rel, D]).  P is bitwise
 * symmetric (fp32 products commute), so (s, t) and (t, s) give identical rows when both take the same product path.
 * Filter: the same set of directed known triples (s, r', t), duplicates counted once.  For a query triple (s, r, t):
 * N = {r' != r : (s, r', t) not in the filter}, opt = #{r' in N : S(r') > S(r)}, pess = #{r' in N : S(r') >= S(r)},
 * rank = 1 + (opt + pess) / 2, S(r) read from the same row as every S(r').  Metrics: gn_index_prep of the query
 * triples' relations, then gn_rank_metrics.
 *
 * gn_rank_pair_csr: pair-grouped structure of an edge list.  Three stable counting sorts (by rel, by dst, by src)
 *   order the entries by (src, dst, rel); rows are the distinct directed pairs in (src, dst) order, compacted (not
 *   s*n + t, which does not fit int32 for general n): rowptr [capacity n_edges + 1], pair_src / pair_dst [capacity
 *   n_edges], entries ent_rel / ent_eid [n_edges] (relation, edge id) sorted by relation inside a row; n_pairs
 *   (device int32) the row count.
 * gn_rank_pair_lookup: row[i] = the row of pair (s_i, t_i) in a pair-grouped filter of n_fpairs rows (binary search
 *   over its sorted pairs), or -1 when the filter holds no triple of that pair.  (s_i, t_i) from pair_src / pair_dst
 *   (int32, e.g. a query structure's pairs) or, when pair_src is NULL, from src / dst (int64).
 * gn_rank_pair_rows: p[i, 0:D] = z[s_i] .* z[t_i], (s_i, t_i) taken as in gn_rank_pair_lookup.
 * gn_rank_pair_count: filtered relation rank of every entry of pairs [0, n_pairs) whose score rows are S[g] (lds >=
 *   n_rel; q_rowptr and f_row point at the first pair of the chunk); f_row[g] is the filter row of pair g (from
 *   gn_rank_pair_lookup), f_row == NULL: no filter.  rank[edge id] as in gn_rank_count.
 * gn_rank_pair_topk: the k (1 <= k <= 256; k > n_rel is padded) highest-scoring relations r' with (s_i, r', t_i)
 *   not in the filter, for every row i of S (overwritten: filtered entries are marked in place); f_row[i] the
 *   filter row of query i, or f_row == NULL.  Order, padding and sigmoid as in gn_rank_topk. */
size_t gn_rank_pair_csr_workspace_bytes(int64_t n_edges);
int gn_rank_pair_csr(const int64_t* src, const int64_t* dst, const int64_t* etype, int64_t n_edges, int32_t n_nodes,
                     int32_t n_rel, int32_t* rowptr, int32_t* pair_src, int32_t* pair_dst, int32_t* ent_rel,
                     int32_t* ent_eid, int32_t* n_pairs, void* ws, size_t ws_bytes, void* stream);
int gn_rank_pair_lookup(const int32_t* f_src, const int32_t* f_dst, int32_t n_fpairs,
                        const int32_t* pair_src /*or NULL*/, const int32_t* pair_dst, const int64_t* src,
                        const int64_t* dst, int64_t count, int32_t* row, void* stream);
int gn_rank_pair_rows(const float* z, int64_t ldz, int32_t D, const int32_t* pair_src /*or NULL*/,
                      const int32_t* pair_dst, const int64_t* src, const int64_t* dst, int64_t count, float* p,
                      int64_t ldp, void* stream);
int gn_rank_pair_count(const float* S, int64_t lds, int32_t n_rel, int32_t n_pairs, const int32_t* q_rowptr,
                       const int32_t* q_rel, const int32_t* q_eid, const int32_t* f_row /*or NULL*/,
                       const int32_t* f_rowptr, const int32_t* f_rel, float* rank, void* stream);
int gn_rank_pair_topk(float* S, int64_t lds, int32_t n_rel, int64_t count, const int32_t* f_row /*or NULL*/,
                      const int32_t* f_rowptr, const int32_t* f_rel, int32_t k, int sigmoid, float* out_score,
                      int64_t* out_id, void* stream);

/* Top-k new pairs of a relation, queries (?, r, ?): the candidates are the UNORDERED pairs {s, t} with s < t (the
 * DistMult score is symmetric in s and t; a self-pair is not an interaction), scored with the PRE-sigmoid
 * S = sum_k z[s,k] w[r,k] z[t,k].  {s, t} is filtered for r when (s, r, t) OR (t, r, s) is in the filter: f_rowptr /
 * f_dst is gn_rank_csr of the filter lists concatenated with their flipped copies (row s*n_rel + r holds every t of
 * either direction, sorted), or f_rowptr == NULL.  Order: descending pre-sigmoid score, ties by the smaller pair id
 * s*n + t (smaller s, then smaller t).  Requires n_nodes^2 < 2^31 (the pair id is the low word of a 64-bit key).
 * No [n, n] score matrix is written: stage 1 (one block per query and tile of 64 s rows) scores 64 x 64 tiles of
 * the triangle with FFMA and keeps the tile's top k keys; stage 2 (one block per query) merges them.
 *
 * gn_rank_rel_pairs_workspace_bytes: bytes of the keys passed from stage 1 to stage 2 (count * ceil(n/64) * k * 8).
 * gn_rank_rel_pairs_select: stage 1 for the queries rel[0 .. count) (z rows at stride ldz >= D, w [n_rel, D]
 *   contiguous, 1 <= k <= 256); writes ws.
 * gn_rank_rel_pairs_merge: stage 2, reads ws.  out_score / out_src / out_dst [count, k]: score (sigmoid applied when
 *   `sigmoid`), s and t (s < t); src = dst = -1 and score NaN pad a query with fewer than k admissible pairs. */
size_t gn_rank_rel_pairs_workspace_bytes(int64_t count, int32_t n_nodes, int32_t k);
int gn_rank_rel_pairs_select(const float* z, int64_t ldz, int32_t D, const float* w, int32_t n_rel, int32_t n_nodes,
                             const int64_t* rel, int64_t count, const int32_t* f_rowptr /*or NULL*/,
                             const int32_t* f_dst, int32_t k, void* ws, size_t ws_bytes, void* stream);
int gn_rank_rel_pairs_merge(const void* ws, size_t ws_bytes, int32_t n_nodes, int64_t count, int32_t k, int sigmoid,
                            float* out_score, int64_t* out_src, int64_t* out_dst, void* stream);

/* ---- K12: slot all-gather over NVLink peer memory (multi-GPU exchange step) ------------------ */
/* New design (the reference is single-device, SURVEY.md §8e).  Every rank of the node maps one
 * symmetric arena of identical layout; `arena_base` (HOST array, `world + 1` entries) holds every rank's
 * arena base as this process sees it (peer-mapped device pointers) and, last, the MULTICAST (NVLS) mapping of
 * the arena or 0: with it a slot leaves the GPU once (multimem.st) and the NVSwitch delivers it to every rank,
 * instead of world-1 unicast copies.  The gather buffer is
 * [world][slot_bytes] at `buf_offset` of every arena; this rank's slot is already written.  The call
 * pushes the slot to every peer (128-bit P2P stores), publishes flag (flag_index, rank) = use counter
 * in every peer's flag block (u64 [n_buffers][gn_peer_max_world()] at `flag_offset`, zero-initialised;
 * a flag counts the CTAs of its rank that have delivered, over all uses of the buffer)
 * and waits until all peers have published theirs: kernels enqueued after it on `stream` see the
 * complete buffer.  `seq` / `done`: this buffer's LOCAL use counter (u64) and CTA arrival counter
 * (u32), zero-initialised, owned by the caller; `abort_flag` (u32, zero-initialised, shared by all
 * buffers) is raised when a wait times out (~10 s: a peer died) — later calls then do not wait and the
 * host should treat the step as failed.  Every rank must issue the same sequence of calls.
 * slot_bytes and buf_offset must be multiples of 16.  world == 1 is a no-op. */
int gn_peer_max_world(void);
int gn_peer_allgather(const uint64_t* arena_base /*host*/, int32_t world, int32_t rank, int64_t buf_offset,
                      int64_t slot_bytes, int64_t flag_offset, int32_t flag_index, uint64_t* seq,
                      uint32_t* done, uint32_t* abort_flag, void* stream);


/* Halo-packed exchange (north_star: "all-gather of halo source-feature rows").  The operand buffer of a rank is
 * [its own rows | the rows of peer 0 it references | peer 1 ...] (packed, column indices remapped at graph-build time);
 * `peers[p]` (HOST array, `world` entries; entry `rank` ignored) tells this call which of ITS rows peer p needs
 * (`idx`: device int32 local row ids, `count`) and where they go in p's buffer (`dst_row`: first packed row).
 * The rows are read from `src_rows` (this rank's rows, row_floats floats each, a multiple of 4, 16-byte aligned) and
 * stored over NVLink; then the publish / wait round of gn_peer_allgather.  Every rank launches the same fixed grid
 * (gn_peer_halo_grid()).  `buf_bytes` = size of the (symmetric) operand buffer at `buf_offset`. */
typedef struct {
  const int32_t* idx;
  int64_t count;
  int64_t dst_row;
} gn_halo_peer;
int gn_peer_halo_grid(void);
int gn_peer_halo_push(const uint64_t* arena_base /*host*/, int32_t world, int32_t rank, int64_t buf_offset,
                      int64_t buf_bytes, const float* src_rows, int32_t row_floats,
                      const gn_halo_peer* peers /*host*/, int64_t flag_offset, int32_t flag_index, uint64_t* seq,
                      uint32_t* done, uint32_t* abort_flag, void* stream);

/* Segmented push + rank-ordered sum over the same arena: the small reductions of a partitioned step
 * (bucketed weight-gradient all-reduce + loss, reduce-scatter of the decoder's dz) without NCCL.
 * The exchange buffer is [world][slot_bytes] at `buf_offset` of every arena.  gn_peer_push stores every
 * segment into slot `rank` of the buffer of its target rank (`peer` >= 0) or of EVERY rank incl. this one
 * (`peer` < 0), at `slot_offset` inside the slot, then runs the publish / wait round of gn_peer_allgather
 * (same flag / seq / done / abort arguments).  `segs` is a HOST array (the descriptors travel in the
 * kernel-parameter block: capturable), at most gn_peer_max_segments() entries; bytes and offsets are
 * multiples of 4 (128-bit copies when everything is 16-byte aligned).
 * gn_slot_sum then forms dst[i] = slot_0[i] + slot_1[i] + ... + slot_{world-1}[i] IN RANK ORDER from this
 * rank's own buffer (`buf` = local arena base + buf_offset): every rank adds the same numbers in the same
 * order, so replicated gradients stay bit-identical across ranks and run to run. */
typedef struct {
  const void* src;      /* device pointer (any local memory) */
  int64_t bytes;
  int64_t slot_offset;  /* byte offset inside the slot */
  int32_t peer;         /* target rank, or < 0 for every rank */
} gn_peer_segment;
typedef struct {
  float* dst;           /* device pointer, n floats */
  int64_t n;
  int64_t slot_offset;  /* byte offset inside the slot */
} gn_sum_segment;
int gn_peer_max_segments(void);
int gn_peer_push(const uint64_t* arena_base /*host*/, int32_t world, int32_t rank, int64_t buf_offset,
                 int64_t slot_bytes, const gn_peer_segment* segs /*host*/, int32_t n_segs,
                 int64_t flag_offset, int32_t flag_index, uint64_t* seq, uint32_t* done, uint32_t* abort_flag,
                 void* stream);
int gn_slot_sum(const void* buf, int32_t world, int64_t slot_bytes, const gn_sum_segment* segs /*host*/,
                int32_t n_segs, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GRIPNET_B200_H */
