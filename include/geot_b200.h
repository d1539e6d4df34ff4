/*
 * geot_b200.h -- C ABI of the B200-native (sm_100a) segment-reduction library.
 *
 * This is the drop-in boundary for GeoT's hot path: every entry point replaces one host entry point
 * of the reference's CUDA layer (declared in /root/reference/csrc/cuda/header_cuda.h:4-38) and is
 * what the reference's torch bindings (csrc/<op>.cpp) bind after the swap -- see INTEGRATION.md.
 *
 *   - plain pointers and sizes only: no ATen / torch types cross this boundary;
 *   - every function returns a geot_status_t and never throws;
 *   - all device pointers must belong to the current CUDA device; work is enqueued on `stream`
 *     (the reference launches on the legacy default stream, gather_scatter_base.h:33; callers
 *     pass at::cuda::getCurrentCUDAStream());
 *   - no allocation inside the device entry points: scratch is caller-provided
 *     (geot_b200_workspace_bytes / geot_b200_plan_bytes);
 *   - index tensors are int64, as at the reference API (wrapper/gather_scatter_base.h:20-21).
 *
 * Semantics (SURVEY.md 8a / Appendix B):
 *     dst[dst_index[e], h, :]  (op)=  weight[e, h] * src[src_index[e], h, :]      e = 0 .. E-1
 * dst has S rows and is fully overwritten; rows that receive no edge are 0.  op in
 * {sum, mean, max, min, prod}; mean = sum / count; max/min propagate NaN (torch amax/amin).
 * fp32 and fp64 accumulate in their own type, bf16/fp16 accumulate in fp32 and round once.
 * The reduction is deterministic (fixed tree, no atomics) for sorted dst_index, and for unsorted input unless the
 * fp32-sum vector-atomic path is in use (geot_b200_set_unsorted_mode).
 */
#ifndef GEOT_B200_H_
#define GEOT_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __DRIVER_TYPES_H__
typedef struct CUstream_st *cudaStream_t;
#endif

#define GEOT_B200_VERSION 200 /* 0.2.0 */

#if defined(__GNUC__)
#define GEOT_API __attribute__((visibility("default")))
#else
#define GEOT_API
#endif

typedef enum {
  GEOT_OK = 0,
  GEOT_ERR_INVALID_ARG = 1,  /* null pointer, negative size, bad enum ... */
  GEOT_ERR_UNSUPPORTED = 2,  /* valid request this build does not implement */
  GEOT_ERR_WORKSPACE = 3,    /* workspace / plan buffer too small or misaligned */
  GEOT_ERR_CUDA = 4,         /* a CUDA call failed: see geot_b200_last_cuda_error() */
  GEOT_ERR_EMPTY = 5         /* E == 0 (the reference raises on index[-1] of an empty tensor) */
} geot_status_t;

typedef enum { GEOT_F32 = 0, GEOT_F64 = 1, GEOT_BF16 = 2, GEOT_F16 = 3 } geot_dtype_t;

/* Same members as the reference's ReductionType (csrc/reducetype.h:3). */
typedef enum { GEOT_SUM = 0, GEOT_MEAN = 1, GEOT_MAX = 2, GEOT_MIN = 3, GEOT_PROD = 4 } geot_reduce_t;

/* Where weight element (e, h) lives.  EDGE: weight[e] (gather_weight_scatter_base.h:25);
 * EDGE_HEAD: weight[e*H + h] (mh_spmm_kernel.cuh:66); HEAD_EDGE: weight[h*E + e] (:168). */
typedef enum { GEOT_W_NONE = 0, GEOT_W_EDGE = 1, GEOT_W_EDGE_HEAD = 2, GEOT_W_HEAD_EDGE = 3 } geot_weight_layout_t;

/* ---- library queries ------------------------------------------------------------------------ */

GEOT_API int geot_b200_version(void);                 /* GEOT_B200_VERSION */
GEOT_API int geot_b200_arch(void);                    /* 100: the SASS in this library is sm_100a only */
GEOT_API const char *geot_b200_status_string(int status);
GEOT_API const char *geot_b200_last_cuda_error(void); /* text of the last CUDA failure on this thread */

/* ---- format_preprocess: segment pointers + edge-count partition ------------------------------ */

/* Result of geot_b200_format_preprocess.  Host POD; `rowptr` points into the caller's device
 * plan buffer.  Replaces the reference's per-call `index[-1].item()` (csrc/gather_scatter.cpp:27)
 * and its decision-tree features (wrapper/gather_scatter_rule.h:9-12) with facts about the graph
 * that are computed once and cached by the caller. */
typedef struct geot_plan {
  int64_t E;              /* edges */
  int64_t S;              /* dst rows = dst_index[E-1] + 1 (or the caller's dim_size) */
  int64_t num_segments;   /* non-empty dst rows (index_scatter_cpu.cpp:51 num_nonzero_rows) */
  int64_t max_degree;     /* longest segment */
  int32_t is_sorted;      /* 1 iff dst_index is non-decreasing */
  int32_t has_gaps;       /* 1 iff some row in [0,S) has no edge (num_segments < S) */
  const int64_t *rowptr;  /* device, S+1 entries: CSR row pointer == geot::coo_to_csr
                             (geot/match_replace/format_transform.py:5-18); segment r covers edges
                             [rowptr[r], rowptr[r+1]) */
  int64_t max_row;        /* largest value in dst_index (== dst_index[E-1] when sorted) */
} geot_plan_t;

/* Highest index: reads dst_index[E-1] (sorted input) -- one 8-byte D2H copy, synchronises `stream`. */
GEOT_API int geot_b200_index_last(const int64_t *dst_index, int64_t E, int64_t *last, cudaStream_t stream);

/* Bytes of device memory a plan for (E, S) needs (256-byte aligned buffer). */
GEOT_API size_t geot_b200_plan_bytes(int64_t E, int64_t S);

/* Builds the plan in plan_buf and fills *plan.  Synchronises `stream` once (to return the
 * statistics).  dst_index must be sorted for rowptr to be meaningful; is_sorted reports it. */
GEOT_API int geot_b200_format_preprocess(const int64_t *dst_index, int64_t E, int64_t S, void *plan_buf,
                                size_t plan_bytes, geot_plan_t *plan, cudaStream_t stream);

/* Edge-balanced contiguous dst-row shards for `parts` GPUs (SURVEY.md 8e): row_bounds[parts+1]
 * and edge_bounds[parts+1] (host arrays); shard g owns rows [row_bounds[g], row_bounds[g+1]) and
 * edges [edge_bounds[g], edge_bounds[g+1]), cut at segment boundaries nearest to g*E/parts.
 * Synchronises `stream`. */
GEOT_API int geot_b200_plan_shards(const geot_plan_t *plan, int parts, int64_t *row_bounds,
                          int64_t *edge_bounds, cudaStream_t stream);

/* ---- the hot path ---------------------------------------------------------------------------- */

/* Scratch bytes for one call on E edges with rows of W = H*F elements (256-byte aligned buffer).
 * sorted == 0 adds the buffers of the edge sort that the unsorted path runs first. */
GEOT_API size_t geot_b200_workspace_bytes(int64_t E, int64_t W, int dtype, int sorted);

/* Generic entry: all four ops are this call with different operands.
 *   src        [N_src, H*F]   device, dtype
 *   src_index  [E] int64 or NULL (NULL: src row = e)
 *   dst_index  [E] int64, non-decreasing when sorted != 0
 *   weight     per weight_layout, dtype; NULL iff GEOT_W_NONE
 *   dst        [S, H*F]       device, dtype; fully overwritten
 *   plan       optional (NULL allowed): lets the call skip zero-filling when the graph has no
 *              empty rows, and zero exactly the empty ones up front when it has (without a plan the
 *              main kernel fills the gaps it sees); results are identical with and without it. */
GEOT_API int geot_b200_segment_reduce(const void *src, const int64_t *src_index, const int64_t *dst_index,
                             const void *weight, void *dst, int64_t E, int64_t S, int64_t H,
                             int64_t F, int dtype, int reduce, int weight_layout, int sorted,
                             const geot_plan_t *plan, void *workspace, size_t workspace_bytes,
                             cudaStream_t stream);

/* Options of geot_b200_segment_reduce_ex (zero-initialise, set struct_size = sizeof(geot_reduce_opts_t)).
 * They serve reductions that run as several passes over disjoint edge buckets of ONE graph -- the multi-GPU
 * two-bucket exchange (edges whose src row is local are reduced while the remote rows are in flight, the rest
 * afterwards: geot_b200/dist.py) -- without a combine pass and without re-ordering the caller's weights:
 *   accumulate   != 0: dst[r] += result for the rows this pass touches, other rows untouched (sum, or mean with
 *                mean_rowptr); the first pass runs with accumulate == 0 and writes every row of dst.
 *   edge_perm    [E] int32, device: the weight of edge e of THIS pass is weight[edge_perm[e]] (the bucket keeps the
 *                caller's weight order).  GEOT_W_EDGE weights, sorted input, sum / mean only.
 *   mean_rowptr  [S+1] int64, device: reduce == GEOT_MEAN divides by mean_rowptr[r+1] - mean_rowptr[r] (the row's
 *                degree in the complete edge list) instead of by this pass's own count, so partial means add up. */
typedef struct geot_src_blocks geot_src_blocks_t;
typedef struct geot_reduce_opts {
  size_t struct_size;
  int32_t accumulate;
  int32_t reserved;
  const int32_t *edge_perm;
  const int64_t *mean_rowptr;
  const geot_src_blocks_t *src_blocks;  /* the graph regrouped by src-row block (below): the call reduces block
                                           after block; src_index / dst_index must be the arrays it was built from */
} geot_reduce_opts_t;

GEOT_API int geot_b200_segment_reduce_ex(const void *src, const int64_t *src_index, const int64_t *dst_index,
                                const void *weight, void *dst, int64_t E, int64_t S, int64_t H,
                                int64_t F, int dtype, int reduce, int weight_layout, int sorted,
                                const geot_plan_t *plan, void *workspace, size_t workspace_bytes,
                                cudaStream_t stream, const geot_reduce_opts_t *opts);

/* ---- src-row blocking for the L2 (format_preprocess family; once per graph) ------------------------------------
 * A gather op re-reads src rows E / N_src times; a src matrix beyond what the L2 keeps of a read-shared working set
 * (~60 MB measured on B200) turns those re-reads into DRAM traffic (Reddit-shape F=128: 17 GB per call instead of
 * 2.5).  The edge list is regrouped once, stably, by src-row block; every block is still dst-sorted, and
 * geot_b200_segment_reduce_ex (opts.src_blocks) reduces block after block, the later ones accumulating into dst.
 * Results equal the one-pass results within the sum tolerance (the summation order inside a row changes); sum / mean
 * with at most one weight per edge.  The passes accumulate INTO dst, so a bf16 / fp16 dst is rounded once per pass:
 * callers that hold the 1e-2 bound of 16-bit types keep the block count small (the torch bindings block fp32 / fp64
 * automatically and 16-bit types only on request).
 *   suggest   number of blocks worth using for this shape (1: do not block)
 *   bytes / scratch_bytes   device buffer that holds the regrouped list / scratch for building it (256-byte aligned)
 *   build     fills buf and *blocks; synchronises `stream` once. */
#define GEOT_MAX_SRC_BLOCKS 16
struct geot_src_blocks {
  int64_t E;
  int32_t n_blocks;
  int32_t reserved;
  int64_t bounds[GEOT_MAX_SRC_BLOCKS + 1];  /* edge offsets of the blocks in the arrays below */
  const int64_t *dst_index;                 /* [E] device: the regrouped list */
  const int64_t *src_index;                 /* [E] */
  const int32_t *edge_perm;                 /* [E]: position of regrouped edge e in the caller's list (weights) */
};
GEOT_API int geot_b200_src_blocks_suggest(int64_t E, int64_t S, int64_t N_src, int64_t row_bytes);
GEOT_API size_t geot_b200_src_blocks_bytes(int64_t E);
GEOT_API size_t geot_b200_src_blocks_scratch_bytes(int64_t E);
GEOT_API int geot_b200_src_blocks_build(const int64_t *src_index, const int64_t *dst_index, int64_t E, int64_t N_src,
                               int n_blocks, void *buf, size_t buf_bytes, void *scratch, size_t scratch_bytes,
                               geot_src_blocks_t *blocks, cudaStream_t stream);
/* Scratch for geot_b200_segment_reduce_ex with opts.src_blocks (every block partitions on its own). */
GEOT_API size_t geot_b200_src_blocks_workspace_bytes(const geot_src_blocks_t *blocks, int64_t W, int dtype);

/* Replaces index_scatter_cuda (header_cuda.h:4-6; csrc/cuda/index_scatter_cuda.cu:86-105), dim = 0:
 * src viewed as [E, F] (wrapper/index_scatter_base.h:15-17).  sorted == 0 replaces the reference's all-atomic
 * scatter_reduce_kernel (index_scatter_cuda.cu:75-84, index_scatter_kernel.cuh:204-263): fp32 sum clears dst and adds
 * 16-byte pieces with vector atomics (red.global.add.v4.f32; summation order = the hardware's, as in the reference);
 * every other dtype / reduce op -- and fp32 sum after geot_b200_set_unsorted_mode(1) -- sorts the edge ids by row
 * (stable) and runs the deterministic sorted kernels. */
GEOT_API int geot_b200_index_scatter(const void *src, const int64_t *index, void *dst, int64_t E, int64_t S,
                            int64_t F, int dtype, int reduce, int sorted, const geot_plan_t *plan,
                            void *workspace, size_t workspace_bytes, cudaStream_t stream);

/* Replaces gather_scatter_cuda (header_cuda.h:8-10; csrc/cuda/gather_scatter_cuda.cu:15-28). */
GEOT_API int geot_b200_gather_scatter(const void *src, const int64_t *src_index, const int64_t *dst_index,
                             void *dst, int64_t E, int64_t S, int64_t F, int dtype, int reduce,
                             const geot_plan_t *plan, void *workspace, size_t workspace_bytes,
                             cudaStream_t stream);

/* Replaces gather_weight_scatter_cuda (header_cuda.h:12-17; gather_weight_scatter_cuda.cu:22-39). */
GEOT_API int geot_b200_gather_weight_scatter(const void *src, const int64_t *src_index,
                                    const int64_t *dst_index, const void *weight, void *dst,
                                    int64_t E, int64_t S, int64_t F, int dtype, int reduce,
                                    const geot_plan_t *plan, void *workspace,
                                    size_t workspace_bytes, cudaStream_t stream);

/* Replaces mh_spmm_cuda (header_cuda.h:23-26; csrc/cuda/mh_spmm_cuda.cu:20-38): src [N,H,F],
 * weight_layout GEOT_W_EDGE_HEAD ([E,H]) or GEOT_W_HEAD_EDGE ([H,E]) (wrapper/mh_spmm_base.h:38-49). */
GEOT_API int geot_b200_mh_spmm(const void *src, const int64_t *src_index, const int64_t *dst_index,
                      const void *weight, void *dst, int64_t E, int64_t S, int64_t H, int64_t F,
                      int dtype, int reduce, int weight_layout, const geot_plan_t *plan,
                      void *workspace, size_t workspace_bytes, cudaStream_t stream);

/* Replaces sddmm_coo_cuda (header_cuda.h:19-21; gather_weight_scatter_cuda.cu:41-62), the weight gradient
 * of gather_weight_scatter (geot/gather_weight_scatter.py:47):
 *     out[e] = < mat1[row_index[e], :], mat2[col_index[e], :] >        mat1 [N1,F], mat2 [N2,F], out [E]
 * all of `dtype` (the reference is fp32 + int32 indices only); bf16/fp16 accumulate in fp32.  No scratch,
 * no sortedness requirement; a sorted row_index lets the kernel keep the mat1 row in registers. */
GEOT_API int geot_b200_sddmm_coo(const void *mat1, const int64_t *row_index, const void *mat2,
                        const int64_t *col_index, void *out, int64_t E, int64_t F, int dtype,
                        cudaStream_t stream);

/* Multi-head SDDMM, the weight gradient of mh_spmm (one dot product per edge and head):
 *     out[e, h] = < mat1[row_index[e], h, :], mat2[col_index[e], h, :] >   mat1 [N1,H,F], mat2 [N2,H,F]
 * out is [E,H] (out_layout GEOT_W_EDGE_HEAD) or [H,E] (GEOT_W_HEAD_EDGE), the weight layouts of geot_b200_mh_spmm.
 * All of `dtype`; bf16/fp16 accumulate in fp32 and round once.  No scratch, no sortedness requirement; a sorted
 * row_index lets the kernel keep the mat1 row in registers.  H = 1 computes what geot_b200_sddmm_coo does. */
GEOT_API int geot_b200_sddmm_mh(const void *mat1, const int64_t *row_index, const void *mat2, const int64_t *col_index,
                       void *out, int64_t E, int64_t H, int64_t F, int dtype, int out_layout, cudaStream_t stream);

/* Segment softmax over the edges of each dst row -- the attention weights of a GAT layer:
 *     out[e, h] = exp(src[e, h] - m[r, h]) / sum_{e' : dst_index[e'] = r} exp(src[e', h] - m[r, h]),   r = dst_index[e]
 * with m[r, h] the row's largest logit.  src / out [E, H] row-major, of `dtype`; dst_index [E] int64, non-decreasing
 * (plan->is_sorted; the plan of dst_index from geot_b200_format_preprocess).  bf16/fp16/fp32 accumulate in fp32, fp64 in
 * fp64, with the accurate exp and one IEEE division per element; special values per (row, head) as torch.softmax: a NaN
 * or a +inf logit makes the row NaN, a row of -inf is NaN.  Edge-balanced (a hub row is cut over many CTAs), no
 * atomics: the result is bit-reproducible.  Returns GEOT_ERR_EMPTY for E == 0 and GEOT_ERR_INVALID_ARG for an unsorted
 * plan; workspace: geot_b200_segment_softmax_workspace_bytes (256-byte aligned). */
GEOT_API size_t geot_b200_segment_softmax_workspace_bytes(int64_t E, int64_t H, int dtype);
GEOT_API int geot_b200_segment_softmax(const void *src, const int64_t *dst_index, void *out, int64_t E, int64_t H,
                              int dtype, const geot_plan_t *plan, void *workspace, size_t workspace_bytes,
                              cudaStream_t stream);
/* Its backward, from the forward's output:
 *     grad_src[e, h] = out[e, h] * (grad_out[e, h] - sum_{e' : dst_index[e'] = r} out[e', h] * grad_out[e', h])
 * Same operands, precision, partition, determinism, status codes and workspace as geot_b200_segment_softmax. */
GEOT_API int geot_b200_segment_softmax_backward(const void *out, const void *grad_out, const int64_t *dst_index,
                                       void *grad_src, int64_t E, int64_t H, int dtype, const geot_plan_t *plan,
                                       void *workspace, size_t workspace_bytes, cudaStream_t stream);

/* GATv2 attention score (PyG GATv2Conv, share_weights = False) of every edge and head:
 *     score[e, h] = sum_f att[h, f] * leaky_relu(x_l[src_index[e], h, f] + x_r[dst_index[e], h, f])
 * leaky_relu(u) = u > 0 ? u : slope * u, slope = *negative_slope (host memory, read before the call returns; only
 * integers, sizes and pointers cross this ABI).  x_l [N_l, H, F], x_r [N_r, H, F], att [H, F], out [E, H], all of
 * `dtype`; bf16/fp16/fp32 accumulate in fp32, fp64 in fp64: the sum x_l + x_r is formed in the accumulator, then the
 * slope, then the product with att; one rounding on the store.  No scratch; a sorted dst_index lets the kernel keep the
 * x_r row in registers while dst repeats.  Returns GEOT_ERR_EMPTY for E == 0. */
GEOT_API int geot_b200_gatv2_score(const void *x_l, const void *x_r, const void *att, const int64_t *src_index,
                          const int64_t *dst_index, void *out, int64_t E, int64_t H, int64_t F, int dtype,
                          const double *negative_slope, cudaStream_t stream);
/* Its backward, one pass per node operand.  For g = grad_score [E, H] in the edge order of row_index:
 *     grad_row[r, h, f] = att[h, f] * sum_{e : row_index[e] = r} g[e, h] * leaky'(x_row[r, h, f] + x_gat[gat_index[e], h, f])
 *     grad_att[h, f]    = sum_e g[e, h] * leaky_relu(x_row[row_index[e], h, f] + x_gat[gat_index[e], h, f])
 * with leaky'(u) = u > 0 ? 1 : slope (torch's leaky_relu_backward).  The dst pass is row = x_r, row_index =
 * dst_index, gat = x_l by src_index; the src pass runs on the src-sorted (transposed) edge list with row = x_l and the
 * grads carried into that order (geot_b200_permute_edges).  row_index is non-decreasing: plan is its plan
 * (geot_b200_format_preprocess), with plan->max_row < S_out.  grad_row [S_out, H, F] is fully written (rows without
 * edges are 0); grad_att [H, F] may be NULL.  Same precision as the score; edge-balanced, no atomics: bit-reproducible.
 * Returns GEOT_ERR_EMPTY for E == 0, GEOT_ERR_INVALID_ARG for an unsorted plan, a plan of another index or a plan
 * whose largest index is >= S_out; workspace: geot_b200_gatv2_grad_workspace_bytes (256-byte aligned). */
GEOT_API size_t geot_b200_gatv2_grad_workspace_bytes(int64_t E, int64_t H, int64_t F, int dtype);
GEOT_API int geot_b200_gatv2_grad(const void *x_row, const void *x_gat, const void *att, const void *grad_score,
                         const int64_t *row_index, const int64_t *gat_index, const geot_plan_t *plan, int64_t S_out,
                         void *grad_row, void *grad_att, int64_t E, int64_t H, int64_t F, int dtype,
                         const double *negative_slope, void *workspace, size_t workspace_bytes, cudaStream_t stream);

/* Dot-product graph attention, fused (PyG TransformerConv's attention, without beta, edge features or dropout):
 *     score[e, h]  = scale * < q[dst_index[e], h, :], k[src_index[e], h, :] >          scale = *scale (host memory)
 *     out[i, h, :] = sum_{e : dst_index[e] = i} alpha[e, h] * v[src_index[e], h, :],   alpha = softmax of score over row i
 *     lse[i, h]    = log sum_{e : dst_index[e] = i} exp(score[e, h])
 * q [N_dst, H, F], k / v [N_src, H, F], out [N_dst, H, F] of `dtype`; lse [N_dst, H] in the accumulator type (fp32, or
 * fp64 for fp64).  One edge-balanced pass with an online softmax: no [E, H] score or alpha is stored.  dst_index is
 * non-decreasing: plan is its plan (geot_b200_format_preprocess) with plan->max_row < N_dst.  Every row of out and lse
 * is written; rows without edges get out = 0 and lse = -inf.  bf16/fp16/fp32 accumulate in fp32, fp64 in fp64, with the
 * accurate exp / log and IEEE division, one rounding on every store; a NaN score makes its row NaN.  No atomics: the
 * result is bit-reproducible.  A launch covers whole heads of at most 256 columns (128 for fp64): a head wider than that
 * returns GEOT_ERR_UNSUPPORTED.  Returns GEOT_ERR_EMPTY for E == 0, GEOT_ERR_INVALID_ARG for an unsorted plan, a plan of
 * another index or a plan whose largest index is >= N_dst; workspace: geot_b200_graph_attention_workspace_bytes
 * (256-byte aligned). */
GEOT_API size_t geot_b200_graph_attention_workspace_bytes(int64_t E, int64_t H, int64_t F, int dtype);
GEOT_API int geot_b200_graph_attention(const void *q, const void *k, const void *v, const int64_t *src_index,
                              const int64_t *dst_index, const geot_plan_t *plan, int64_t N_dst, void *out, void *lse,
                              int64_t E, int64_t H, int64_t F, int dtype, const double *scale, void *workspace,
                              size_t workspace_bytes, cudaStream_t stream);
/* The dst pass of its backward, recomputing alpha from lse (FlashAttention-2).  With g = grad_out [N_dst, H, F]:
 *     D[i, h] = < g[i, h], out[i, h] >,   p[e, h] = exp(score[e, h] - lse[dst, h]),
 *     ds[e, h] = scale * p[e, h] * (< g[dst, h], v[src, h] > - D[dst, h]),
 *     grad_q[i] = sum_{e : dst_index[e] = i} ds[e, h] * k[src, h, :]
 * grad_q [N_dst, H, F] is fully written (rows without edges are 0); p and ds [E, H] (`dtype`) are the weights of the
 * src-side gradients grad_k = sum_{e : src = j} ds q[dst] and grad_v = sum_{e : src = j} p g[dst], which
 * geot_b200_mh_spmm computes on the transposed edge list.  Same operands, precision, determinism and status codes as
 * the forward; workspace: geot_b200_graph_attention_grad_workspace_bytes (256-byte aligned). */
GEOT_API size_t geot_b200_graph_attention_grad_workspace_bytes(int64_t E, int64_t H, int64_t F, int dtype);
GEOT_API int geot_b200_graph_attention_grad(const void *q, const void *k, const void *v, const void *out,
                                   const void *lse, const void *grad_out, const int64_t *src_index,
                                   const int64_t *dst_index, const geot_plan_t *plan, int64_t N_dst, void *grad_q,
                                   void *p, void *ds, int64_t E, int64_t H, int64_t F, int dtype, const double *scale,
                                   void *workspace, size_t workspace_bytes, cudaStream_t stream);

/* CSR row pointer -> sorted COO row index (the inverse of geot::coo_to_csr): row_index[e] = r for
 * rowptr[r] <= e < rowptr[r+1].  rowptr has S+1 entries of 32 or 64 bits (rowptr_bits).  Lets the CSR entry
 * point csr_gws (csrc/csr_gws.cpp:24-35, csr_gws_cuda.cu) run on the same kernels. */
GEOT_API int geot_b200_csr_to_coo(const void *rowptr, int rowptr_bits, int64_t S, int64_t E, int64_t *row_index,
                         cudaStream_t stream);

/* ---- multi-GPU helpers (dst-row shards, SURVEY.md 8e; new -- the reference has no distributed code) ---------- */

/* out[e] = in[perm[e]] for records of bytes_per_edge bytes (even): carries per-head edge weights [E, H] into bucket
 * order (one weight per edge needs no pass: geot_reduce_opts_t.edge_perm), or packs feature rows (perm = row ids,
 * bytes_per_edge = the row size; moved as 16-byte vectors when size and pointers allow). */
GEOT_API int geot_b200_permute_edges(const void *in, const int64_t *perm, void *out, int64_t E, int64_t bytes_per_edge,
                            cudaStream_t stream);

/* Fused pack + transfer over peer memory (NVLink P2P stores; no NCCL call, no staging buffer):
 *     peer_bases[dest_peer[e]][dest_row[e], :] = x[rows[e], :]          e = 0 .. n-1,  rows of row_bytes bytes
 * peer_bases: DEVICE array of base pointers, one per GPU of the group, each the receive buffer of that GPU mapped
 * into this process (torch symmetric memory: _SymmetricMemory.buffer_ptrs_dev; cudaIpc / cuMem mappings work the
 * same); peers_aligned16 != 0 promises those bases are 16-byte aligned.  row_bytes must be even.  The
 * stores are complete when the kernel is; the caller orders them against the consumers with a cross-GPU barrier on
 * `stream` (geot_b200/dist.py BucketedGather, transport "push").  rows / dest_peer / dest_row are built once per graph. */
GEOT_API int geot_b200_push_rows(const void *x, const int64_t *rows, const int32_t *dest_peer, const int64_t *dest_row,
                        void *const *peer_bases, int64_t n, int64_t row_bytes, int peers_aligned16,
                        cudaStream_t stream);
/* The same transfer on a grid of at most max_ctas CTAs (128 threads, <= 48 registers each), for a push that runs BESIDE
 * a reduction on another stream: 2 CTAs per SM (296) keep an NVLink direction ~85 % busy and still fit next to the
 * resident CTAs of the reduction kernel.  max_ctas <= 0: the whole GPU (= geot_b200_push_rows). */
GEOT_API int geot_b200_push_rows_ex(const void *x, const int64_t *rows, const int32_t *dest_peer, const int64_t *dest_row,
                           void *const *peer_bases, int64_t n, int64_t row_bytes, int peers_aligned16, int max_ctas,
                           cudaStream_t stream);

/* ---- host-buffer entry (end-to-end path) ----------------------------------------------------- */

/* Same operation with every operand in HOST memory (pinned memory makes the copies asynchronous).
 * src is copied first, then the sorted edge list in slices cut at segment boundaries: slice k+1 is
 * copied while slice k is reduced and the finished dst rows of slice k-1 travel back.  Device buffers
 * come from a per-process arena that is reused across calls (geot_b200_host_arena_release frees it).
 * Returns after dst is complete in host memory.  dst_index must be sorted; S must be given.  Not
 * thread-safe (one arena).  This is the call a non-torch host (cgo / JNI / ctypes) makes. */
GEOT_API int geot_b200_segment_reduce_host(const void *src, int64_t N_src, const int64_t *src_index,
                                  const int64_t *dst_index, const void *weight, void *dst,
                                  int64_t E, int64_t S, int64_t H, int64_t F, int dtype, int reduce,
                                  int weight_layout);
GEOT_API int geot_b200_host_arena_release(void);

/* Resident host graph: the index arrays of a graph are uploaded ONCE; every reduce call then moves only what
 * changes from call to call (src rows and edge weights in, dst rows out).  A GNN's graph is static across layers and
 * epochs, so this is the host-buffer call a training / serving loop makes after the first step.
 *   create   src_index [E] (or NULL: src row = edge id, index_scatter) and dst_index [E] (sorted) in HOST memory;
 *            S dst rows, N_src src rows.  Synchronous; the handle belongs to the current device.
 *   reduce   src [N_src, H*F] (or [E, H*F] when created without src_index), weight per weight_layout (or NULL), dst
 *            [S, H*F], all in HOST memory (pinned memory makes the copies asynchronous).  The edge list is processed
 *            in slices cut at segment boundaries: the weights (and edge-aligned src rows) of slice k+1 travel while
 *            slice k is reduced and the finished dst rows of slice k-1 go home.  Returns when dst is complete.
 *   last_transfer  bytes the last reduce moved over the link per direction, and the bytes made resident by create.
 * One call at a time per handle. */
typedef struct geot_host_graph geot_host_graph_t;
GEOT_API int geot_b200_host_graph_create(const int64_t *src_index, const int64_t *dst_index, int64_t E, int64_t S,
                                int64_t N_src, geot_host_graph_t **graph);
GEOT_API int geot_b200_host_graph_reduce(geot_host_graph_t *graph, const void *src, const void *weight, void *dst,
                                int64_t H, int64_t F, int dtype, int reduce, int weight_layout);
GEOT_API int geot_b200_host_graph_last_transfer(const geot_host_graph_t *graph, unsigned long long *h2d_bytes,
                                       unsigned long long *d2h_bytes, unsigned long long *resident_bytes);
GEOT_API int geot_b200_host_graph_destroy(geot_host_graph_t *graph);

/* Row-pointer transport of the host-buffer entry (default; environment GEOT_B200_HOST_COMPACT=0 turns it off): each
 * slice sends its CSR row pointer (rows + 1 values, computed by the host threads below) instead of its dst_index (one
 * value per edge); the device expands it (the inverse of geot::coo_to_csr).  Results are identical; the bytes over
 * the link drop (Reddit-shape gather_weight_scatter: 2.41 -> 1.49 GB, 44.5 -> 28.1 ms).
 * GEOT_B200_HOST_THREADS bounds the host threads (default: hardware concurrency, at most 32).
 * geot_b200_host_last_transfer reports the bytes the last host call really moved in each direction. */
GEOT_API int geot_b200_host_last_transfer(unsigned long long *h2d_bytes, unsigned long long *d2h_bytes);

/* Host-side CSR row pointer of a sorted index slice (pure CPU, no CUDA call):
 *     rowptr[i] = first position p in index[0, n) with index[p] >= row0 + i,      i = 0 .. rows
 * == geot::coo_to_csr (geot/match_replace/format_transform.py:5-18) for row0 = 0, rows = index[n-1] + 1, and the
 * segment-pointer pass of the reference's CPU kernel (csrc/cpu/index_scatter_cpu.cpp:36-75).  threads <= 0: all. */
GEOT_API int geot_b200_host_row_pointers(const int64_t *index, int64_t n, int64_t row0, int64_t rows, int64_t *rowptr,
                                int threads);

/* sorted == 0 policy, process-wide: 0 (default) = vector atomics where they apply (fp32 sum: fastest, not
 * bit-reproducible run to run); 1 = always the deterministic sort-based path.  The torch bindings select 1 while
 * torch.use_deterministic_algorithms(True) is in force. */
GEOT_API int geot_b200_set_unsorted_mode(int mode);

/* ---- instrumentation -------------------------------------------------------------------------- */

/* geot_b200_profile_enable(n > 0): every following segment-reduce call on this host thread records a
 * CUDA event pair around its MAIN kernel (the fixup pass and any memset stay outside), cycling through
 * n pairs; n = 0 disables and frees them.  geot_b200_profile_read copies the durations (ms) of the
 * last min(n, calls) recorded kernels, oldest first, into ms[] and returns their count in *count
 * (synchronises on the events).  Used by bench.py for the roofline figure; off by default. */
GEOT_API int geot_b200_profile_enable(int n);
GEOT_API int geot_b200_profile_read(float *ms, int capacity, int *count);

#ifdef __cplusplus
}
#endif
#endif /* GEOT_B200_H_ */
