/* dcb200.h — C ABI of libdcb200.so: the sm_100a message-passing hot path of DeformContact.
 *
 * The reference (mahdi-slh/DeformContact) is pure Python and has no FFI of its own; the seam
 * this library plugs into is the PyG layer call ``conv(x, edge_index)`` at
 * models/model.py:71,77 and the edge builders at utils/graph_utils.py:7 /
 * utils/pointcloud_utils.py:7.  Every entry point below names the reference (or pinned
 * third-party) operation it replaces.  The Python binding is deformcontact_b200/_abi.py
 * (ctypes); INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Contract (all entry points):
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless stated;
 *  - the caller owns all memory (inputs, outputs, workspace); nothing is allocated, freed or
 *    retained past return;
 *  - all work is enqueued on `stream` (a cudaStream_t); no host synchronisation, no
 *    default-stream use, no mutable state shared between calls except a launch counter and per-device "function
 *    attribute set" flags (both idempotent)  => re-entrant and CUDA-graph capturable.  One entry point uploads a
 *    host-built table (dc_gemm_batched): it is capturable when the caller passes page-locked staging memory;
 *  - returns DC_OK (0) or a negative dc_status; dc_last_error() gives a thread-local message;
 *  - features / weights are fp32, indices int32 inside the ABI (int64 edge_index is converted
 *    by dc_csr_build); leading dimensions (ld*) are in elements;
 *  - reductions are deterministic: per-receiver sums run in CSR order (= original edge order,
 *    the sort is stable), split reductions use a fixed tree. No floating-point atomics.
 */
#ifndef DCB200_H
#define DCB200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define DC_API __attribute__((visibility("default")))
#else
#define DC_API
#endif

typedef void* dc_stream_t; /* cudaStream_t */

typedef enum {
  DC_OK = 0,
  DC_EINVAL = -1,     /* bad shape / alignment / null pointer */
  DC_ENOSUP = -2,     /* unsupported width or mode */
  DC_ECUDA = -3,      /* a CUDA runtime call failed; see dc_last_error() */
  DC_EWORKSPACE = -4  /* workspace too small */
} dc_status;

DC_API int dc_version(void);
DC_API const char* dc_last_error(void);
/* Total number of kernels this library has launched in the process (relaxed atomic; bench.py's
 * `gpu_launches`). */
DC_API uint64_t dc_launch_count(void);

/* ---------------------------------------------------------------- K5: CSR construction
 * Replaces the per-forward ``gcn_norm`` + scatter index handling of PyG
 * (nn/conv/gcn_conv.py:gcn_norm, called by TAGConv/GCNConv at models/model.py:71,77) and the
 * int64 -> int32 conversion.  Stable LSD radix sort of the edges by `group_by` endpoint.
 *   edge_index : int64 [2, E] row-major (row 0 = source j, row 1 = target i)
 *   group_by   : 0 = by target (forward aggregation), 1 = by source (transpose, backward)
 *   drop_self_loops : 1 removes edges with source == target (GCN/GAT "remaining self loops")
 *   rowptr [N+1], nbr [E] (the other endpoint), eid [E] (original edge id; entries at and
 *   beyond rowptr[N] are unspecified when self loops were dropped).
 */
DC_API size_t dc_csr_build_workspace_bytes(int64_t num_nodes, int64_t num_edges);
DC_API int dc_csr_build(const int64_t* edge_index, int64_t num_edges, int64_t num_nodes, int group_by,
                 int drop_self_loops, int32_t* rowptr, int32_t* nbr, int32_t* eid, void* workspace,
                 size_t workspace_bytes, dc_stream_t stream);

/* dis[i] = (deg_i + add_self_loop)^-1/2 computed as 1/sqrt (two correctly rounded ops, like
 * ATen's CPU pow(-0.5)); 0 when the degree is 0.  deg_i = rowptr[i+1] - rowptr[i] of the
 * by-target CSR.  Replaces gcn_norm's deg/pow/masked_fill. */
DC_API int dc_deg_inv_sqrt(const int32_t* rowptr_by_target, int64_t num_nodes, int add_self_loop, float* dis,
                    dc_stream_t stream);

/* ---------------------------------------------------------------- K1: gather / segmented sum
 * Replaces MessagePassing.propagate(aggr='add') with message = w_e * x_j
 * (PyG message_passing.py / tag_conv.py / gcn_conv.py; reference call sites models/model.py:71,77):
 *   out[i, :] = add[i, :] + sum_{e in rowptr[i]..rowptr[i+1]} w_e * h[nbr[e], :]  (+ self-loop term)
 *   w_e = (dis ? dis[nbr[e]] * dis[i] : 1) * (edge_w ? edge_w[edge_w_index ? edge_w_index[e] : e] : 1)
 *   self_loop = 1 appends the term dis[i]*dis[i]*h[i] (or edge_w_self[i]*h[i]) after the edges.
 * One warp (or sub-warp) per receiver, 128-bit row loads when F % 4 == 0 and rows are 16-B
 * aligned, sequential fp32 mul+add in CSR order (bit-reproducible, no atomics).
 * Epilogue: + bias[F] (row broadcast), then max(0, .) when relu = 1 (GCN/GAT `out + bias`).
 * `add`, `dis`, `edge_w`, `edge_w_index`, `self_w`, `bias` may be NULL.  out may not alias h.
 */
DC_API int dc_spmm(const int32_t* rowptr, const int32_t* nbr, const float* dis, const float* edge_w,
            const int32_t* edge_w_index, const float* self_w, const float* h, int64_t ldh, float* out, int64_t ldo, const float* add,
            int64_t ldadd, int64_t num_nodes, int32_t F, int self_loop, const float* bias, int relu,
            dc_stream_t stream);

/* K1 v2: same operation, mapped as (tile of consecutive receivers) x (128-byte feature slice)
 * per CTA so that a tile's source-row slices are reused out of L1 instead of being re-fetched
 * through L2 for every edge.  w [E] = per-edge weight in CSR order (dc_edge_weights; NULL -> 1),
 * self_w [N] = self-loop weight (required when self_loop = 1).  Tiles: tile_ptr int32
 * [n_tiles+1] of receiver offsets (e.g. graph boundaries of the block-diagonal batch, merged /
 * split to ~2k nodes), or NULL for fixed tiles of `tile_nodes` receivers.  Needs F % 4 == 0 and
 * 16-byte aligned rows (DC_ENOSUP otherwise -> use dc_spmm).  Same summation order and
 * rounding as dc_spmm: results are bit-identical.  variant: 0 = 4 lanes x 2 float4 per receiver;
 * 1 = 8 lanes x float4 with a streaming L1 prefetch pass over the tile's own rows; 2 = same, no prefetch;
 * 3 = 64-byte slices staged in shared memory with cp.async, gathers served from shared memory. */
DC_API int dc_edge_weights(const int32_t* rowptr, const int32_t* nbr, const float* dis, int64_t num_nodes, float* w,
                           float* self_w, dc_stream_t stream);
DC_API int dc_spmm_tiled(const int32_t* rowptr, const int32_t* nbr, const float* w, const float* self_w, const float* h,
                         int64_t ldh, float* out, int64_t ldo, const float* add, int64_t ldadd, int64_t num_nodes,
                         int32_t F, int self_loop, const float* bias, int relu, const int32_t* tile_ptr,
                         int64_t n_tiles, int32_t tile_nodes, int variant, dc_stream_t stream);

/* K1 v9 (hop chain): up to DC_MAX_CHAIN consecutive hops in one launch; hop k computes
 *   out_k = add_k + A in_k      (same rows, records, order and rounding as dc_spmm_lean; bit-identical)
 * where in_k may be out_{k-1} (TAGConv forward h_{k+1} = A h_k, models/model.py:71,77 via PyG tag_conv.py; backward
 * g_{k-1} = dH_{k-1} + A^T g_k on the transposed records).  add_k may equal out_k (in place).  A CTA keeps its
 * (tile, 128-byte slice) across the hops, so REQUIRES every tile to be closed under the edges (whole graphs of a
 * block-diagonal batch: tile_ptr built from Batch.ptr without splitting a graph) and F % 32 == 0. */
#define DC_MAX_CHAIN 4
typedef struct dc_hop {
  const float* in; int64_t ldin;
  const float* add; int64_t ldadd;   /* NULL: no addend */
  float* out; int64_t ldout;
} dc_hop_t;
DC_API int dc_spmm_chain(const int32_t* rowptr, const void* edges, const float* self_w, const dc_hop_t* hops, int32_t num_hops,
                  int64_t num_nodes, int32_t F, int self_loop, const int32_t* tile_ptr, int64_t n_tiles, int32_t tile_nodes,
                  dc_stream_t stream);

/* K1 v10 (TMA-staged hop chain): the contract of dc_spmm_chain, for any F % 4 == 0.  The (tile x feature slice) of each
 * hop's input is copied into shared memory once by TMA (cp.async.bulk.tensor.2d over the strided [rows, slice] view,
 * completion on an mbarrier) and the gathers are served from shared memory; the slice width adapts to the tile
 * (4..8 float4 lanes per receiver so that max_tile_rows x lanes x 16 B fits 227 KB: 2000 rows -> 112-byte slices).
 * Same rows, records, order and rounding as dc_spmm_lean / dc_spmm_chain: bit-identical.  REQUIRES closed tiles (whole
 * graphs of a block-diagonal batch) like dc_spmm_chain; max_tile_rows = the largest tile (ignored without tile_ptr).
 * dc_spmm_stage_supported() says whether tiles of that size fit (else DC_ENOSUP: use dc_spmm_chain).
 * Replaces: the K consecutive MessagePassing.propagate calls of one PyG TAGConv forward / backward
 * (models/model.py:71,77). */
DC_API int dc_spmm_stage_supported(int64_t max_tile_rows, int32_t F);
DC_API int dc_spmm_stage(const int32_t* rowptr, const void* edges, const float* self_w, const dc_hop_t* hops, int32_t num_hops,
                         int64_t num_nodes, int32_t F, int self_loop, const int32_t* tile_ptr, int64_t n_tiles,
                         int32_t tile_nodes, int64_t max_tile_rows, dc_stream_t stream);
/* K1 v11 (stream hop chain): the contract of dc_spmm_chain without self loops (TAGConv: gcn_norm(add_self_loops=False)).
 * An 8-lane group owns a contiguous, cost-balanced range of the tile's receivers, walks its edges as ONE stream of packed
 * records (prefetched into a shared-memory ring by cp.async) and keeps a rolling window of 8 row gathers in flight across
 * receiver boundaries.  Same rows, records, order and rounding as dc_spmm_lean / dc_spmm_chain: bit-identical.  REQUIRES
 * closed tiles when num_hops > 1 (like dc_spmm_chain), F % 32 == 0 and packed records (dc_pack_edges).
 * Replaces: the K consecutive MessagePassing.propagate calls of one PyG TAGConv forward / backward (models/model.py:71,77). */
DC_API int dc_spmm_stream(const int32_t* rowptr, const void* edges, const dc_hop_t* hops, int32_t num_hops, int64_t num_nodes,
                          int32_t F, const int32_t* tile_ptr, int64_t n_tiles, int32_t tile_nodes, dc_stream_t stream);
/* K1 v6 ("lean"): the same tile x 128-byte-slice mapping driven by packed 8-byte edge records
 * {int32 neighbour, fp32 weight} in CSR order (dc_pack_edges; w == NULL -> weight 1): one uniform 64-bit
 * load per edge instead of index/weight loads + shuffles, 8 row gathers in flight per lane, no predicates on
 * full 8-edge chunks.  Bit-identical to dc_spmm / dc_spmm_tiled. */
DC_API int dc_pack_edges(const int32_t* nbr, const float* w, int64_t num_edges, void* edges_out, dc_stream_t stream);
DC_API int dc_spmm_lean(const int32_t* rowptr, const void* edges, const float* self_w, const float* h, int64_t ldh,
                        float* out, int64_t ldo, const float* add, int64_t ldadd, int64_t num_nodes, int32_t F,
                        int self_loop, const float* bias, int relu, const int32_t* tile_ptr, int64_t n_tiles,
                        int32_t tile_nodes, dc_stream_t stream);

/* K1 v7 ("edge blocks"): the same operation driven by a sliced-ELL (SELL-4-sigma) copy of the CSR built once
 * per batch by dc_blocks_build and reused by every hop.  Receivers ("slots") are sorted by degree (stable,
 * descending) inside windows of 256 receivers of a tile and grouped four to a UNIT; a unit's edge records
 * {int32 neighbour, fp32 weight} are interleaved [pair of edges][slot][2] so one 128-bit load per lane fetches two
 * records and a warp reads one contiguous 64-byte segment; rows deeper than 64 edges continue from the packed CSR
 * records (`edges`, dc_pack_edges).  fp32 mul and add are issued as packed FMUL2 / FFMA2(m, 1.0, acc): separately
 * rounded, in CSR order => bit-identical to dc_spmm.
 *   tile_ptr      int32 [n_tiles+1]  receiver offsets of the tiles (graphs of the batch merged / split to ~2k)
 *   tile_unit_ptr int32 [n_tiles+1]  prefix sum of ceil(tile_size / 4); n_units = tile_unit_ptr[n_tiles]
 *   slots         int4  [n_units*4]  {node or -1, degree, record offset of the unit, depth | min_degree << 8}
 *   recs          int2  [rec_capacity], rec_capacity >= dc_blocks_record_capacity(N, E, n_tiles) (a proven bound;
 *                 `status` (int32, zero-initialised by the caller) is set to 1 if it were ever exceeded)
 * unit_size = 4 (the layout dc_spmm_blocks reads) or 8; tile_unit_ptr is the prefix sum of ceil(tile_size / unit_size)
 * and slots has n_units * unit_size entries.  Bit 16 of a slot's depth word flags units with a source outside their
 * own tile or a row deeper than 64 edges.
 * dc_spmm_blocks flags: bit 0 = persistent grid (one CTA per SM looping over tile slices), bit 1 = prefetch the
 * next unit's records into L1, bit 2 = 768-thread CTAs (80 registers) instead of 1024 (64 registers), bits 3-4 =
 * distance (in grid strides, 0 = off) of the L2 prefetch stream: while a CTA works on one tile slice it pulls the row
 * slices, edge records and slot records of the tile slice it takes that many steps later into L2.
 * tile_rec_ptr int32 [n_tiles+1] (written by dc_blocks_build) = record offsets at the tile boundaries. */
DC_API size_t dc_blocks_workspace_bytes(int64_t n_units);
DC_API int64_t dc_blocks_record_capacity(int64_t num_nodes, int64_t num_edges, int64_t n_tiles);
DC_API int dc_blocks_build(const int32_t* rowptr, const void* edges, const int32_t* tile_ptr, const int32_t* tile_unit_ptr,
                           int64_t n_tiles, int64_t n_units, int32_t unit_size, void* slots, void* recs, int64_t rec_capacity,
                           int32_t* tile_rec_ptr, int32_t* status, void* workspace, size_t workspace_bytes, dc_stream_t stream);
DC_API int dc_spmm_blocks(const void* slots, const void* recs, const int32_t* rowptr, const void* edges, const int32_t* tile_ptr,
                          const int32_t* tile_unit_ptr, const int32_t* tile_rec_ptr, int64_t n_tiles, const float* self_w, const float* h, int64_t ldh,
                          float* out, int64_t ldo, const float* add, int64_t ldadd, int32_t F, int self_loop,
                          const float* bias, int relu, int flags, dc_stream_t stream);

/* A9 — fused edge update of the edge-MLP / node-MLP residual layer (north_star; no reference symbol):
 *   mode 0: out_i = sum_{e in row i} relu(p_i + q[nbr_e])                 forward  (p = u, q = v, by-target CSR)
 *   mode 1: out_i = sum_e (p_i + q[nbr_e] > 0 ? r_i : 0)                  d/du     (r = ds, by-target CSR)
 *   mode 2: out_i = sum_e (p_i + q[nbr_e] > 0 ? r[nbr_e] : 0)             d/dv     (p = v, q = u, r = ds, by-source CSR)
 * All matrices fp32 [N, F] with leading dimension ld; F % 4 == 0, 16-byte aligned rows. */
DC_API int dc_edge_relu(const int32_t* rowptr, const int32_t* nbr, const float* p, const float* q, const float* r,
                        float* out, int64_t ld, int64_t num_nodes, int32_t F, int mode, dc_stream_t stream);

/* ---------------------------------------------------------------- K2: dense GEMMs
 * Replaces the Linear calls inside the PyG convs (nn/dense/linear.py; A3c in SURVEY.md) and, since round 1 late,
 * carries the matrix products of the cross attention and of the decoder MLP (models/model.py:7-21, 52-64).
 * C[M,N] = act( sum_{s<nseg} opA(A_s)[M,K_s] * opB(B_s)[K_s,N] + bias[N] )  (+ C if accumulate)
 *   transA = 0 : A_s stored [M, K_s] row-major (lda_s);  1 : stored [K_s, M] row-major
 *   transB = 0 : B_s stored [K_s, N] row-major (ldb_s);  1 : stored [N, K_s] row-major
 *   relu = 1 applies max(0, .) in the epilogue; bias may be NULL.
 * precision: DC_GEMM_FP32 = fp32 FFMA (SIMT, any shape / stride); DC_GEMM_TF32X3 = tcgen05 kind::tf32 with the
 * 3-term error-compensated split and fp32 round-to-nearest chain sums (fp32-class accuracy, ~1e-6 against fp64) —
 * every layout for nseg = 1, transA = 0 / transB = 1 for nseg > 1, any M, N, K; needs lda/ldb % 4 == 0 and 16-byte
 * aligned operands (DC_ENOSUP otherwise); DC_GEMM_AUTO = tensor path for M*N*K >= 1e8 where supported, else fp32;
 * DC_GEMM_PREFER_TC = tensor path whenever supported, regardless of size.
 * When M x N alone gives fewer 128 x 128 tiles than SMs the contraction is cut into parts whose partial tiles go to
 * `workspace` and are summed in fixed order by a second kernel (deterministic).
 */
enum { DC_GEMM_AUTO = 0, DC_GEMM_FP32 = 1, DC_GEMM_TF32X3 = 2, DC_GEMM_PREFER_TC = 3 };
typedef struct {
  const float* A;
  int64_t lda;
  const float* B;
  int64_t ldb;
  int64_t K;
} dc_gemm_seg;
DC_API size_t dc_gemm_workspace_bytes(int64_t M, int64_t N, int64_t K_total, int transA, int transB);
DC_API int dc_gemm(const dc_gemm_seg* segs /*host array*/, int nseg, int transA, int transB, int64_t M, int64_t N,
            float* C, int64_t ldc, const float* bias, int relu, int accumulate, int precision, void* workspace,
            size_t workspace_bytes, dc_stream_t stream);

/* `count` independent products C_i[M_i,N_i] = act(opA(A_i) opB(B_i)) (+C_i) with common transposes in ONE launch of the
 * tcgen05 3xTF32 kernel: the 128 x 128 work items of all problems are dealt to the persistent CTAs together, so
 * problems too small to fill 148 SMs alone (the per-group products of the cross attention, models/model.py:16-18) run
 * at the rate of a large one.  Every problem must satisfy the tensor-path requirements of dc_gemm (DC_ENOSUP
 * otherwise; the caller then falls back to per-problem dc_gemm).  `problems` is a host array; the problem table
 * (tensor maps) is built on the host and uploaded into `workspace` on the stream.  `host_staging` (HOST pointer,
 * page-locked, >= dc_gemm_batched_workspace_bytes(count) bytes, caller-owned) holds the host image of the table: the
 * upload is then an asynchronous copy that CUDA-graph capture records as a copy node, and the caller must keep the
 * buffer alive and unmodified until the copy has executed (for a captured graph: as long as the graph lives).  With
 * host_staging = NULL the image is a temporary pageable buffer: correct, but the call then blocks the host for the
 * staging copy and must NOT be stream-captured. */
typedef struct {
  const float* A;
  int64_t lda;
  const float* B;
  int64_t ldb;
  float* C;
  int64_t ldc;
  int64_t M, N, K;
  const float* E;    /* optional fused epilogue: C = E o (acc - rowv[row]) with E [M, N] (lde), rowv [M]; NULL = none. */
  int64_t lde;       /* With E = P (attention weights) and rowv = rowdot(dO, O) this is the softmax backward          */
  const float* rowv; /* dS = P o (dP - rowsum(dP o P)) applied to dP = dO Xr^T as it leaves the tensor core.          */
} dc_gemm_problem;   /* A batch in which any problem carries E must have relu = 0 and accumulate = 0 (DC_EINVAL otherwise). */
DC_API size_t dc_gemm_batched_workspace_bytes(int32_t count);
DC_API int dc_gemm_batched(const dc_gemm_problem* problems /*host array*/, int32_t count, int transA, int transB, int relu,
                           int accumulate, void* workspace, size_t workspace_bytes, void* host_staging /*pinned host or NULL*/,
                           size_t host_staging_bytes, dc_stream_t stream);

/* colsum[n] = sum_m X[m, n] (bias gradient), deterministic two-stage tree. */
DC_API size_t dc_colsum_workspace_bytes(int64_t M, int64_t N);
DC_API int dc_colsum(const float* X, int64_t ldx, int64_t M, int64_t N, float* out, void* workspace,
              size_t workspace_bytes, dc_stream_t stream);

/* N1 (SURVEY.md 8f) — element-wise pieces of the dense cross attention (models/model.py:7-21; the matrix products
 * run through dc_gemm): in-place row softmax  S[m,:] <- softmax(S[m,:])  and its backward, in place on dP:
 * dS[m,n] = P[m,n] * (dP[m,n] - sum_j dP[m,j] P[m,j]).  One CTA per row, fixed reduction tree (deterministic). */
DC_API int dc_softmax_rows(float* S, int64_t ld, int64_t M, int64_t N, dc_stream_t stream);
DC_API int dc_softmax_bwd_rows(const float* P, int64_t ldp, float* dP, int64_t ldd, int64_t M, int64_t N, dc_stream_t stream);

/* out[m] = sum_n A[m, n] * B[m, n]  (one warp per row, fixed order) */
DC_API int dc_rowdot(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int64_t N, float* out, dc_stream_t stream);

/* N2 (SURVEY.md 8f) — the two training losses (train.py:47-58: nn.L1Loss on the displacements, models/losses.py:12-17
 * GradientConsistencyLoss over the edges) and their gradients w.r.t. `pred` in one deterministic pass over the CSR pair
 * (by target: rowptr / nbr, by source: rowptr_t / nbr_t).  pred, tgt: fp32 [N, 3] contiguous.
 *   partial [N, 2] = { sum over edges into i of ||(tgt_i - tgt_j) - (pred_i - pred_j)||,  sum_c |pred_ic - tgt_ic| }
 *   gc [N, 3] = d(sum of edge norms)/d pred_i,   gl [N, 3] = sign(pred - tgt)
 * The caller sums the columns of `partial` (dc_colsum) and scales by 1/E and 1/(3N). */
DC_API int dc_edge_loss(const int32_t* rowptr, const int32_t* nbr, const int32_t* rowptr_t, const int32_t* nbr_t, const float* pred,
                        const float* tgt, int64_t num_nodes, float* partial, float* gc, float* gl, dc_stream_t stream);

/* dX = dY * (Y > 0)  (backward of the ReLU fused into dc_gemm's epilogue; models/model.py:71,77) */
DC_API int dc_relu_bwd(const float* Y, const float* dY, float* dX, int64_t numel, dc_stream_t stream);
/* The same with the bias gradient taken on the way: dX = dY * (Y > 0) and colsum[n] = sum_m dX[m, n] in one pass over
 * [M, N] matrices (leading dimensions ld*), summed in the order of dc_colsum (bit-identical to dc_relu_bwd + dc_colsum);
 * workspace >= dc_colsum_workspace_bytes(M, N).  Replaces relu'() followed by bias.grad of every Linear / conv + ReLU pair
 * in the backward of models/model.py:71,77,88. */
DC_API int dc_relu_bwd_colsum(const float* Y, int64_t ldy, const float* dY, int64_t lddy, float* dX, int64_t lddx, int64_t M,
                              int64_t N, float* colsum, void* workspace, size_t workspace_bytes, dc_stream_t stream);

/* ---------------------------------------------------------------- K4: kNN / radius graph
 * Replaces torch_cluster.knn_graph / radius_graph as called at utils/pointcloud_utils.py:10,12
 * (loop=False, flow source_to_target).  Brute force, tiled through shared memory, per-query
 * warp-shuffle top-k.  Distances fp32 ((dx*dx)+(dy*dy))+(dz*dz) with no FMA contraction;
 * ties -> lower index.  `ptr` (int64 [B+1], device) delimits independent point clouds
 * (Batch.ptr); pass B = 1 and ptr = {0, N} for batch=None.
 *  knn : nbr_out int32 [N, k] ascending (distance, index); -1 where fewer than k exist.
 *        With loop=0 the search is for k+1 and the self match is removed (torch_cluster rule).
 *  radius: up to max_nbr neighbours with d2 < r*r in ascending index order, self excluded
 *        per torch_cluster's "search max_nbr+1 including self, then drop self" rule;
 *        nbr_out int32 [N, max_nbr] padded with -1, count_out int32 [N].
 */
DC_API int dc_knn(const float* pos /*[N,3]*/, const int64_t* ptr, int64_t num_graphs, int64_t num_points, int32_t k,
           int loop, int32_t* nbr_out, dc_stream_t stream);
DC_API int dc_radius(const float* pos, const int64_t* ptr, int64_t num_graphs, int64_t num_points, float r,
              int32_t max_nbr, int loop, int32_t* nbr_out, int32_t* count_out, dc_stream_t stream);
/* K4g: the same searches for ONE point cloud (batch=None) on a uniform grid: bounding box, ~8 points per cell,
 * counting sort by cell, one warp per query walking rings of cells until the answer is provably complete.  Results
 * are bit-identical to dc_knn / dc_radius (same distances, keys and tie rule; radius keeps the lowest indices).  All
 * grid parameters are computed on the device (no host sync).  Worth it from a few ten thousand points up. */
DC_API size_t dc_knn_grid_workspace_bytes(int64_t num_points);
/* order_out (int32 [N], may be NULL): the points in grid-cell order, as dc_cell_order returns it. */
DC_API int dc_knn_grid(const float* pos, int64_t num_points, int32_t k, int loop, int32_t* nbr_out, int32_t* order_out,
                void* workspace, size_t workspace_bytes, dc_stream_t stream);
DC_API int dc_radius_grid(const float* pos, int64_t num_points, float r, int32_t max_nbr, int loop, int32_t* nbr_out,
                   int32_t* count_out, int32_t* order_out, void* workspace, size_t workspace_bytes, dc_stream_t stream);
/* K4g, batched (kNN): one grid per graph of a batch of large clouds (`ptr` as in dc_knn: torch_cluster.knn_graph with a `batch`
 * vector, utils/pointcloud_utils.py:10 applied per sample) in the same launches: per-graph bounding box and cell size, the graphs'
 * cells end to end in one cell array, one counting sort, every query walks its own graph's grid.  Bit-identical to dc_knn; worth
 * it from about a thousand points per graph (short brute-force scans spend their time in the top-k insertion path).  One
 * device-side decision for the whole batch: if the grids cannot split the clouds the brute-force kernel runs instead. */
DC_API size_t dc_knn_grid_batched_workspace_bytes(int64_t num_points, int64_t num_graphs);
DC_API int dc_knn_grid_batched(const float* pos, const int64_t* ptr, int64_t num_graphs, int64_t num_points, int32_t k, int loop,
                        int32_t* nbr_out, void* workspace, size_t workspace_bytes, dc_stream_t stream);
/* ... and torch_cluster.radius_graph with a `batch` vector on the same per-graph grids (workspace as dc_knn_grid_batched);
 * bit-identical to dc_radius. */
DC_API int dc_radius_grid_batched(const float* pos, const int64_t* ptr, int64_t num_graphs, int64_t num_points, float r,
                           int32_t max_nbr, int loop, int32_t* nbr_out, int32_t* count_out, void* workspace,
                           size_t workspace_bytes, dc_stream_t stream);
/* order[i] = index of the i-th point in grid-cell order (the counting sort of K4g): a spatially coherent relabelling
 * of a large point cloud.  A permutation of 0..N-1; the order inside a cell is unspecified.  Workspace as dc_knn_grid. */
DC_API int dc_cell_order(const float* pos, int64_t num_points, int32_t* order, void* workspace, size_t workspace_bytes,
                  dc_stream_t stream);
/* out[i, :] = in[perm[i], :] (fp32 rows; in != out).  Used to run the hops of a large single graph in cell order. */
DC_API int dc_permute_rows(const float* in, int64_t ldin, const int32_t* perm, float* out, int64_t ldout, int64_t num_rows,
                    int32_t F, dc_stream_t stream);
/* Compacts a padded neighbour table into edge_index int64 [2, E_cap] (row 0 = neighbour,
 * row 1 = query), queries ascending; *num_edges_out (device int64) receives E. */
DC_API size_t dc_nbr_to_edge_index_workspace_bytes(int64_t num_points);
DC_API int dc_nbr_to_edge_index(const int32_t* nbr, int64_t num_points, int32_t width, int64_t* edge_index,
                         int64_t edge_cap, int64_t* num_edges_out, void* workspace, size_t workspace_bytes,
                         dc_stream_t stream);

/* ---------------------------------------------------------------- A6: mesh -> edges, features
 * mesh_to_graph (utils/graph_utils.py:12-13): triangles int64 [T,3] -> edge_index int64 [2,3T]
 * in per-triangle order (a,b),(b,c),(c,a); `offset` is added to every index (batching). */
DC_API int dc_mesh_edges(const int64_t* triangles, int64_t num_tri, int64_t offset, int64_t* edge_index,
                  int64_t edge_stride, int64_t edge_start, dc_stream_t stream);
/* to_log_freq(pos, 3, 1) (utils/pos_encoding.py:6-44): [N,3] -> [N,21] at out[:, col0:col0+21]. */
DC_API int dc_posenc(const float* pos, int64_t num_points, float* out, int64_t ldo, int32_t col0, dc_stream_t stream);

/* ---------------------------------------------------------------- N3: on-GPU batch assembly
 * Replaces Batch.from_data_list(...).to(device) (train.py:36-44; PyG data/batch.py), the per-sample
 * mesh_to_graph loop (utils/graph_utils.py:12-16), _feature_rigid (loaders/common.py:6-19) and the
 * collider sphere instancing (loaders/common.py:25-30).  The host concatenates the per-sample arrays
 * with GRAPH-LOCAL indices into one staging buffer and copies it once; these kernels emit the batched
 * layout.  `node_ptr`, `edge_ptr`, `tri_ptr`: int64 [B+1] device arrays of cumulative counts
 * (ptr[0] = 0; empty graphs allowed).  `index_bytes` = 4 (int32) or 8 (int64) for local indices. */
/* batch[i] = graph of node i (Batch.batch), int64 [N]. */
DC_API int dc_batch_vector(const int64_t* node_ptr, int64_t num_graphs, int64_t num_nodes, int64_t* batch,
                    dc_stream_t stream);
/* edge_index[:, e] = local[:, e] + node_ptr[graph of edge e]; local is [2, E] with row stride
 * `local_stride` elements, edge_index int64 [2, E] with row stride `edge_stride`. */
DC_API int dc_edges_offset(const void* local, int32_t index_bytes, int64_t local_stride, const int64_t* edge_ptr,
                    const int64_t* node_ptr, int64_t num_graphs, int64_t num_edges, int64_t* edge_index,
                    int64_t edge_stride, dc_stream_t stream);
/* mesh_to_graph half-edges (a,b),(b,c),(c,a) for every graph of a batch in one launch.
 * Ragged form: triangles [num_tri, 3] local indices, tri_ptr / node_ptr given.
 * Instanced form (tri_ptr = NULL): the same `tri_per_graph` template triangles for each of the
 * num_graphs graphs, graph g offset by g * nodes_per_graph; num_tri = num_graphs * tri_per_graph. */
DC_API int dc_mesh_edges_batched(const void* triangles, int32_t index_bytes, const int64_t* tri_ptr,
                          const int64_t* node_ptr, int64_t num_graphs, int64_t num_tri, int64_t tri_per_graph,
                          int64_t nodes_per_graph, int64_t* edge_index, int64_t edge_stride, dc_stream_t stream);
/* out[n, :] = [head[graph(n), 0:head_width] | to_log_freq(pos[n], 3, 1)]  (head_width = 0: the 21-d soft
 * features; head_width = 4: the collider's [force_vector | force] ++ posenc, loaders/common.py:18). */
DC_API int dc_node_features(const float* pos, const float* head, int32_t head_width, const int64_t* node_ptr,
                     int64_t num_graphs, int64_t num_nodes, float* out, int64_t ldo, dc_stream_t stream);
/* pos[g*V + v, :] = float(tmpl[v, :] + centers[g, :]) with the add in fp64 (Open3D translate). */
DC_API int dc_instance_points(const double* tmpl, const double* centers, int64_t num_graphs, int64_t num_template_points,
                       float* pos, dc_stream_t stream);

/* ---------------------------------------------------------------- K6: GAT attention pieces
 * (PyG nn/conv/gat_conv.py, utils/softmax.py)  a_src[n,h] = sum_c xs[n,h,c]*att_src[h,c] etc. */
DC_API int dc_gat_scores(const float* xs, int64_t ld, int64_t num_nodes, int32_t heads, int32_t C, const float* att_src,
                  const float* att_dst, float* a_src, float* a_dst, dc_stream_t stream);
/* Per receiver i over its CSR edges plus the appended self loop:
 *   e = leaky_relu(a_src[nbr] + a_dst[i], slope); alpha = exp(e - max) / (sum + 1e-16).
 * Writes alpha_edge [E] indexed by ORIGINAL edge id (eid[p]) and alpha_self [N]; heads == 1 only (any heads: dc_gat_aggregate). */
DC_API int dc_gat_softmax(const int32_t* rowptr, const int32_t* nbr, const int32_t* eid, const float* a_src,
                   const float* a_dst, float slope, int64_t num_nodes, float* alpha_edge, float* alpha_self,
                   dc_stream_t stream);
/* Backward of the attention scalars (one warp per receiver): dalpha_e = <dout[i], xs[nbr]>,
 * softmax and leaky-relu backward; writes dz_edge [E] (by original edge id), dz_self [N] and
 * da_dst[i] = sum of dz over i's edges and self loop. */
DC_API int dc_gat_bwd_edge(const int32_t* rowptr, const int32_t* nbr, const int32_t* eid, const float* a_src,
                    const float* a_dst, float slope, const float* alpha_edge, const float* alpha_self,
                    const float* xs, int64_t ldx, const float* dout, int64_t ldd, int32_t C, int64_t num_nodes,
                    float* dz_edge, float* dz_self, float* da_dst, dc_stream_t stream);
/* out[i] = (init ? init[i] : 0) + sum_{p in row i} val[eid[p]]  (CSR order; e.g. da_src over the by-source CSR) */
DC_API int dc_segment_sum(const int32_t* rowptr, const int32_t* eid, const float* val, const float* init,
                   int64_t num_nodes, float* out, dc_stream_t stream);

/* ---------------------------------------------------------------- K6 multi-head (csrc/gat.cu)
 * PyG 2.5.x GATConv with any heads >= 1, concat or mean (add_self_loops=True, dropout=0).  Structure: the "gat" CSR pair
 * (self loops removed; one appended per node by the kernels).  Per-(node, head) arrays are [N, H] row-major, per-edge ones
 * [E, H] indexed by ORIGINAL edge id.  Sums per (node, head) in CSR order, then the self loop; no atomics.
 * All return DC_EINVAL for heads < 1, C < 1, a leading dimension shorter than the row, or a null pointer. */
/* Replaces GATConv's softmax (utils/softmax.py) + propagate(aggr='add') + concat / mean(dim=1) + bias (nn/conv/gat_conv.py):
 *   z[e,h] = leaky_relu(a_src[src,h] + a_dst[i,h], slope); alpha = exp(z - max_i) / (sum_i exp(z - max_i) + 1e-16);
 *   out_h[i] = sum_e alpha[e,h] xs[src_e, h*C : (h+1)*C] (+ self loop);
 *   out[i] = concat ? [out_0 | ... | out_{H-1}] : (out_0 + ... + out_{H-1}) / H;  then + bias (H*C or C), ReLU if relu.
 * xs [N, H*C] (ld ldx), a_src / a_dst [N, H] from dc_gat_scores.  Writes out (width H*C or C, ld ldo), alpha_edge [E, H],
 * alpha_self [N, H]. */
DC_API int dc_gat_aggregate(const int32_t* rowptr, const int32_t* nbr, const int32_t* eid, const float* xs, int64_t ldx,
                     const float* a_src, const float* a_dst, float slope, int32_t heads, int32_t C, int32_t concat,
                     const float* bias, int32_t relu, int64_t num_nodes, float* out, int64_t ldo, float* alpha_edge,
                     float* alpha_self, dc_stream_t stream);
/* Replaces the autograd of GATConv's attention (softmax and leaky-ReLU backward), by receiver:
 *   dalpha[e,h] = dout_scale * <dout[i, h*dout_head_stride : +C], xs[src_e, h*C : (h+1)*C]>
 * (concat: head stride C, scale 1; mean: head stride 0, scale 1/H), then dz = alpha (dalpha - sum alpha dalpha) leaky'(z).
 * Writes dz_edge [E, H] (by original edge id), dz_self [N, H], da_dst[i,h] = sum of dz over i's edges and self loop. */
DC_API int dc_gat_bwd_edge_heads(const int32_t* rowptr, const int32_t* nbr, const int32_t* eid, const float* a_src,
                          const float* a_dst, float slope, const float* alpha_edge, const float* alpha_self, const float* xs,
                          int64_t ldx, const float* dout, int64_t ldd, int64_t dout_head_stride, float dout_scale,
                          int32_t heads, int32_t C, int64_t num_nodes, float* dz_edge, float* dz_self, float* da_dst,
                          dc_stream_t stream);
/* dc_gat_bwd_edge_heads for a loss that also reads the attention coefficients (GATConv's return_attention_weights):
 *   dalpha[e,h] = dout_scale * <dout_h[i], xs_h[src_e]> + dalpha_edge[e,h]  (self loop: + dalpha_self[i,h]),
 * then the same softmax and leaky-ReLU backward.  dalpha_edge [E, H] by original edge id, dalpha_self [N, H], both row-major
 * with row stride heads and nullable (null adds nothing; both null runs dc_gat_bwd_edge_heads' kernel, same bits).  dout is
 * required: a loss on alpha alone passes zeros.  Same checks and outputs as dc_gat_bwd_edge_heads. */
DC_API int dc_gat_bwd_edge_heads_ext(const int32_t* rowptr, const int32_t* nbr, const int32_t* eid, const float* a_src,
                              const float* a_dst, float slope, const float* alpha_edge, const float* alpha_self, const float* xs,
                              int64_t ldx, const float* dout, int64_t ldd, int64_t dout_head_stride, float dout_scale,
                              int32_t heads, int32_t C, int64_t num_nodes, const float* dalpha_edge, const float* dalpha_self,
                              float* dz_edge, float* dz_self, float* da_dst, dc_stream_t stream);
/* Replaces the autograd of the aggregation and of the scores (the transposed propagate and the att products), by source, on the
 * by-source CSR (nbr_t = receivers):  da_src[j,h] = sum_{e: src=j} dz[e,h] + dz_self[j,h];
 *   dxs[j,h,:] = dout_scale (sum_e alpha[e,h] dout_h[dst_e] + alpha_self[j,h] dout_h[j]) + da_src[j,h] att_src[h,:]
 *                + da_dst[j,h] att_dst[h,:],  dout_h as in dc_gat_bwd_edge_heads.  Writes dxs [N, H*C] (ld lddx), da_src [N, H]. */
DC_API int dc_gat_scatter_heads(const int32_t* rowptr_t, const int32_t* nbr_t, const int32_t* eid_t, const float* alpha_edge,
                         const float* alpha_self, const float* dz_edge, const float* dz_self, const float* da_dst,
                         const float* att_src, const float* att_dst, const float* dout, int64_t ldd, int64_t dout_head_stride,
                         float dout_scale, int32_t heads, int32_t C, int64_t num_nodes, float* dxs, int64_t lddx, float* da_src,
                         dc_stream_t stream);
/* Replaces the autograd of (xs * att_src).sum(-1) / (xs * att_dst).sum(-1) wrt att:
 *   datt_src[h,c] = sum_n da_src[n,h] xs[n, h*C + c], datt_dst likewise; fixed two-stage column reduction (as dc_colsum). */
DC_API size_t dc_gat_att_grad_workspace_bytes(int64_t num_nodes, int32_t heads, int32_t C);
DC_API int dc_gat_att_grad(const float* xs, int64_t ldx, const float* da_src, const float* da_dst, int64_t num_nodes,
                    int32_t heads, int32_t C, float* datt_src, float* datt_dst, void* workspace, size_t workspace_bytes,
                    dc_stream_t stream);

/* ---------------------------------------------------------------- edge weights for TAGConv / GCNConv (csrc/gcn_norm.cu)
 * edge_weight: fp32 [E] in edge_index order.  Structures: the "tag" CSR pair (loops kept as ordinary edges) or the "gcn"
 * pair (self loops dropped, one appended per node).  Per-node sums in CSR order, then the loop; no floating-point atomics. */
/* Replaces PyG 2.5.2's weighted gcn_norm (nn/conv/gcn_conv.py:gcn_norm; loop_mode 1 = utils/loop.py:add_remaining_self_loops
 * with fill_value):
 *   loop_eid[n] = last edge id e with src = dst = n, else -1; loop_w[n] = edge_weight[loop_eid[n]], else fill_value;
 *   deg_i = sum_{CSR row i} edge_weight[eid] (+ loop_w[i]);  dis = deg^-1/2 (0 where deg == 0, NaN where deg < 0);
 *   norm_e = (dis[src] * w_e) * dis[dst]  (normalize = 0: norm_e = w_e);  self_w[i] = (dis[i] * loop_w[i]) * dis[i].
 * Writes dis (normalize), loop_w / loop_eid / self_w (loop_mode 1), and norm_e at every CSR position of the by-target
 * structure (w_fwd [E] and / or packed {nbr, norm} records edges_fwd [E] for dc_spmm_lean / dc_spmm_chain) and, when
 * w_src or edges_src is given, of the by-source structure.  edge_index (int64 [2, E]) is read in loop_mode 1 only. */
DC_API int dc_gcn_norm_weighted(const int64_t* edge_index, int64_t num_edges, int64_t num_nodes, const int32_t* rowptr,
                                const int32_t* nbr, const int32_t* eid, const int32_t* rowptr_t, const int32_t* nbr_t,
                                const int32_t* eid_t, const float* edge_weight, float fill_value, int normalize, int loop_mode,
                                float* dis, float* loop_w, int32_t* loop_eid, float* self_w, float* w_fwd, void* edges_fwd,
                                float* w_src, void* edges_src, dc_stream_t stream);
/* Sampled dense-dense products over the edges (the autograd of the hops of MessagePassing.propagate wrt the edge weights):
 *   s_edge[eid[p]] (+)= sum_k <g_k[i, :F], h_k[nbr[p], :F]>  for every by-target CSR position p of receiver i,
 *   s_self[i]      (+)= sum_k <g_k[i, :F], h_k[i, :F]>        (when s_self is not NULL),
 * for 1..DC_MAX_CHAIN pairs in one launch (accumulate = 1 adds to the values already there).  One warp per receiver; per pair
 * a lane sums its columns in fp32, the pairs and the lanes are added in fp64 (fixed shuffle tree), rounded once.
 * DC_EINVAL for F < 1, a bad pair count, ld < F or a null pointer (rowptr, nbr, eid, pairs, s_edge and every g_k / h_k are
 * required; nbr and eid are not read when every row is empty). */
typedef struct dc_sddmm_pair {
  const float* g; int64_t ldg;
  const float* h; int64_t ldh;
} dc_sddmm_pair_t;
DC_API int dc_edge_sddmm(const int32_t* rowptr, const int32_t* nbr, const int32_t* eid, const dc_sddmm_pair_t* pairs,
                         int32_t num_pairs, int64_t num_nodes, int32_t F, int accumulate, float* s_edge, float* s_self,
                         dc_stream_t stream);
/* Backward of dc_gcn_norm_weighted (normalize = 1) from s = dL/dnorm (dc_edge_sddmm), in fp64, rounded once:
 *   dL/ddis_n = sum_{e: dst=n} s_e dis[src] w_e + sum_{e: src=n} s_e w_e dis[dst] + 2 s_self[n] loop_w[n] dis[n];
 *   dL/ddeg_n = -dis_n^3 / 2 * dL/ddis_n (0 where deg_n == 0);  dw[e] = s_e dis[src] dis[dst] + dL/ddeg[dst];
 *   dw[loop_eid[n]] = s_self[n] dis[n]^2 + dL/ddeg_n; every other edge (superseded loops, dropped edges) gets 0.
 * s_self / loop_w / loop_eid NULL: no appended loops (the "tag" structure).  dw [E] by original edge id. */
DC_API int dc_gcn_norm_weighted_backward(const int32_t* rowptr, const int32_t* nbr, const int32_t* eid, const int32_t* rowptr_t,
                                         const int32_t* nbr_t, const int32_t* eid_t, const float* edge_weight, const float* dis,
                                         const float* loop_w, const int32_t* loop_eid, const float* s_edge, const float* s_self,
                                         int64_t num_nodes, int64_t num_edges, float* dw, dc_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DCB200_H */
