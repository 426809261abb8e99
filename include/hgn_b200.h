/* libhgn_b200.so -- C ABI of the B200 (sm_100a) message-passing processor kernels.
 *
 * The reference (CemOezcan/hyper-graph-nets) has no FFI: its hot path is Python calling ATen and
 * torch_scatter.  The drop-in boundary is therefore the Python module API of src/migration + src/util
 * (mirrored by hyper-graph-nets_b200/hgn_b200), and THIS header is what that mirror binds through
 * ctypes.  Every entry point names the reference code it replaces (paths relative to the reference
 * root).  Conventions:
 *   - plain pointers and sizes only; all data pointers are DEVICE pointers unless named host_*;
 *   - the caller owns every buffer; nothing is allocated or freed inside; scratch memory is passed in
 *     and its size is queried with the matching *_workspace_bytes function;
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on that stream and
 *     re-entrant across streams (no global mutable state besides the per-thread error string);
 *   - return value: HGN_OK (0) or a negative hgn_status; hgn_last_error() gives the message;
 *   - feature rows are row-major contiguous [rows, D]; index arrays are int32 unless stated;
 *   - dtype: HGN_F32 = fp32 storage and fp32 FFMA arithmetic (parity mode, 1e-5 relative);
 *            HGN_BF16 = bf16 storage, bf16 tcgen05 tensor-core GEMMs with fp32 TMEM accumulators,
 *            fp32 bias/ReLU/LayerNorm/residual arithmetic (throughput mode, 2e-2 relative);
 *   - all reductions are order-deterministic: no floating-point atomics anywhere.
 */
#ifndef HGN_B200_H_
#define HGN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HGN_B200_ABI_VERSION 6

typedef enum {
  HGN_OK = 0,
  HGN_ERR_INVALID_ARGUMENT = -1,
  HGN_ERR_CUDA = -2,
  HGN_ERR_UNSUPPORTED = -3,
  HGN_ERR_WORKSPACE = -4
} hgn_status;

typedef enum { HGN_F32 = 0, HGN_BF16 = 1 } hgn_dtype;

/* bit flags selecting segment reductions; 'pna' = all four (src/migration/graphnet.py:52-64) */
enum { HGN_AGG_SUM = 1, HGN_AGG_MEAN = 2, HGN_AGG_MAX = 4, HGN_AGG_MIN = 8 };

#define HGN_MAX_CHUNKS 24   /* 1 + 4 aggregates x 5 edge sets = 21 for hetero/plate (SURVEY.md s8 a10) */

int hgn_abi_version(void);
const char* hgn_last_error(void);
/* 1 if the current device is an sm_100-class GPU that can run the tcgen05 kernels */
int hgn_device_supported(void);

/* ---- plan: receiver-sorted CSR --------------------------------------------------------------
 * Replaces the per-call index expansion of src/util.py:105-110 (repeat_interleave of the int64 ids to
 * [E,128]) by a one-off stable counting sort.  `segment_ids` are the reference's int64 receivers (or
 * senders).  Outputs: perm[E] = edge ids grouped by segment, ascending edge id inside a segment
 * (stable -> "first edge wins" for max/min ties, like torch_scatter's CPU reducer); rowptr[S+1];
 * ids32[E] = the ids narrowed to int32 (may be NULL).  Ids outside [0,S) are an error reported
 * through *host_status_flag semantics: the call returns HGN_ERR_INVALID_ARGUMENT after a sync. */
size_t hgn_csr_workspace_bytes(int64_t num_edges, int64_t num_segments);
int hgn_csr_build(const int64_t* segment_ids, int64_t num_edges, int64_t num_segments,
                  int32_t* perm, int32_t* rowptr, int32_t* ids32,
                  void* workspace, size_t workspace_bytes, void* stream);

/* ---- edge -> node aggregation -----------------------------------------------------------------
 * Replaces util.unsorted_segment_operation / torch_scatter.scatter_{add,mean,max,min}
 * (src/util.py:92-134) as used by GraphNet.aggregation (src/migration/graphnet.py:50-70).
 * One pass over the receiver-sorted edges produces every requested reduction of data[E,D] into
 * out_*[S,D] (NULL = not requested).  Empty segments give 0; mean = sum / max(count,1);
 * argmax/argmin[S,D] (int32, -1 for empty segments) record the winning edge id and are required when
 * max/min are requested with need_arg != 0.  D must be a multiple of 4 for the vector path; any D
 * >= 1 is accepted (scalar path).  accumulate_sum != 0 adds into out_sum instead of overwriting (used
 * for the gather backward: dv += segment_sum(dX)). */
int hgn_segment_reduce(int dtype, const void* data, int64_t num_edges, int32_t D,
                       const int32_t* perm, const int32_t* rowptr, int64_t num_segments,
                       void* out_sum, void* out_mean, void* out_max, void* out_min,
                       int32_t* argmax, int32_t* argmin, int accumulate_sum, void* stream);

/* 'sum' of the same rows under two groupings in one pass (out_a[S_a,D] by (perm_a,rowptr_a), out_b[S_b,D] by (perm_b,rowptr_b)):
 * the autograd of the two row gathers v[senders], v[receivers] of one edge set (src/migration/graphnet.py:24-25: index_select ->
 * two index_add_) applied to the same per-edge gradient.  Same arithmetic and summation order as two hgn_segment_reduce calls; for
 * bf16 / D = 128 the two groupings are interleaved block by block so that, on a mesh with local node numbering, each row is read
 * from HBM once. */
int hgn_segment_sum_pair(int dtype, const void* data, int64_t num_edges, int32_t D,
                         const int32_t* perm_a, const int32_t* rowptr_a, int64_t num_segments_a, void* out_a,
                         const int32_t* perm_b, const int32_t* rowptr_b, int64_t num_segments_b, void* out_b, void* stream);

/* Backward of the above (autograd of scatter_add / scatter_mean / scatter_max / scatter_min):
 * grad_data[e,:] (+)= g_sum[r_e,:] + g_mean[r_e,:]/max(cnt_r,1) + [argmax[r_e,:]==e] g_max[r_e,:]
 *                    + [argmin[r_e,:]==e] g_min[r_e,:]        (NULL gradients are skipped). */
/* perm (the plan's grouping of element ids by segment, may be NULL) lets the bf16 / D = 128 case run segment-wise: each
 * segment's gradient rows are read once instead of once per element. */
int hgn_segment_reduce_bwd(int dtype, int64_t num_edges, int32_t D,
                           const int32_t* ids32, const int32_t* perm, const int32_t* rowptr, int64_t num_segments,
                           const void* g_sum, const void* g_mean, const void* g_max, const void* g_min,
                           const int32_t* argmax, const int32_t* argmin,
                           void* grad_data, int accumulate, void* stream);

/* Incoming gradient of e' in a GraphNet layer with a 'mean' / 'max' / 'min' / 'pna' aggregator (HGN_BF16, D = 128 only; HGN_F32
 * returns HGN_ERR_UNSUPPORTED), in one pass over the receiver CSR (perm, rowptr[S+1]) of the num_edges elements:
 *     agg_grad[r,:]  = g_sum[r,:] + g_mean[r,:] * (1 / max(cnt_r, 1))                                 [S,128], every segment
 *     edge_grad[e,:] = base[e,:] + [argmax[r_e,:] == e] g_max[r_e,:] + [argmin[r_e,:] == e] g_min[r_e,:]    [E,128]
 * agg_grad is what hgn_edge_update_backward gathers through the receivers as grad_agg, edge_grad its grad_out; base is the dense
 * gradient of e' (next layer / loss).  NULL inputs are skipped.  Arithmetic: fp32 starting from +0, terms added in the order above,
 * g_mean * inv rounded before the addition (no fused multiply-add), each output rounded to bf16 once.  agg_grad may be NULL when
 * g_sum and g_mean are; edge_grad may be NULL when g_max, g_min and base are; edge_grad must not alias base, nor agg_grad a
 * gradient input. */
int hgn_segment_layer_grad(int dtype, int64_t num_edges, int32_t D, const int32_t* perm, const int32_t* rowptr, int64_t num_segments,
                           const void* g_sum, const void* g_mean, const void* g_max, const void* g_min,
                           const int32_t* argmax, const int32_t* argmin, const void* base, void* agg_grad, void* edge_grad,
                           void* stream);

/* ---- long segments: the split plan and its entry points (HGN_BF16, D = 128 only) -------------------------------------------
 * The four calls above give one segment to half a warp or one warp.  A HyperGraphNet's cluster pooling (intra_cluster_to_cluster,
 * receivers = the C hyper nodes) and broadcast (intra_cluster_to_mesh, senders = the hyper nodes) turn every cluster into one
 * segment of ~N/C elements, which one thread group then walks one latency round at a time.  A segment is LONG when it has more than
 * HGN_SEGMENT_SPLIT_THRESHOLD elements; it is cut into PIECES of HGN_SEGMENT_SPLIT_PIECE consecutive positions of perm (the last
 * piece may be shorter), and every piece of a call is worked at once.  The short segments go through the calls above, unchanged,
 * on the split's SHORT CSR (perm_short, rowptr_short): the plan's CSR with every long segment emptied and every short one keeping
 * its elements in order.  So short segments get exactly the bits of the calls above.
 *
 * Arithmetic of a long segment (fp32, no atomics, bitwise reproducible):
 *   piece partial p_k = sum from +0 of the piece's rows in perm order;  total = (((0 + p_0) + p_1) + ...) in ascending k;
 *   sum  = bf16_rn(total), or bf16_rn(total + prior) with accumulate_sum (the prior added after the sum, as above);
 *   mean = bf16_rn(total * (1.0f / cnt));
 *   max / min and their winners = the sequential first-in-order result of hgn_segment_reduce, bit for bit (piece winners
 *   combined in ascending order with strict comparisons);
 *   the backward terms (hgn_segment_reduce_bwd_split, hgn_segment_layer_grad_split) are per element, with the arithmetic of the
 *   calls they mirror, so they are bit-identical to them. */
#define HGN_SEGMENT_SPLIT_THRESHOLD 2048
#define HGN_SEGMENT_SPLIT_PIECE 256
/* the two constants above, as built into the library */
int32_t hgn_segment_split_threshold(void);
int32_t hgn_segment_split_piece(void);

typedef struct {
  int64_t num_segments, num_elements;   /* S and E of the CSR it was built from */
  int64_t n_long, n_pieces, n_short;
  const int32_t* long_ids;              /* [n_long] ascending segment ids */
  const int32_t* piece_ptr;             /* [n_long + 1]: the pieces of long_ids[i] are piece_ptr[i] .. piece_ptr[i+1]-1 */
  const int32_t* pieces;                /* [n_pieces][3]: segment, begin, end (positions in perm), grouped by segment ascending */
  const int32_t* perm_short;            /* [n_short] (a valid pointer even when n_short = 0) */
  const int32_t* rowptr_short;          /* [S+1] */
} hgn_segment_split;

/* Builds a split from a CSR (perm[E], rowptr[S+1]) into caller buffers sized from bounds:
 *   long_ids   >= hgn_segment_split_max_long(E, S) int32,      piece_ptr >= that + 1 int32,
 *   pieces     >= 3 * hgn_segment_split_max_pieces(E) int32,    perm_short >= max(E, 1) int32,    rowptr_short = S + 1 int32.
 * host_counts[3] receives n_long, n_pieces, n_short: the call reads them with one small device-to-host copy and synchronises the
 * stream.  Everything is written whether or not a segment is long (with n_long = 0 the short CSR is the plan's own). */
size_t hgn_segment_split_build_workspace_bytes(int64_t num_edges, int64_t num_segments);
int64_t hgn_segment_split_max_long(int64_t num_edges, int64_t num_segments);
int64_t hgn_segment_split_max_pieces(int64_t num_edges);
int hgn_segment_split_build(const int32_t* perm, const int32_t* rowptr, int64_t num_edges, int64_t num_segments,
                            int32_t* long_ids, int32_t* piece_ptr, int32_t* pieces, int32_t* perm_short, int32_t* rowptr_short,
                            int64_t* host_counts, void* workspace, size_t workspace_bytes, void* stream);

/* fp32 partials of the long pieces: the workspace of hgn_segment_reduce_split and hgn_segment_sum_pair_split (for the pair: the
 * larger of the two sides' sizes; a NULL split needs none). */
size_t hgn_segment_split_reduce_workspace_bytes(const hgn_segment_split* split);

/* hgn_segment_reduce over a split plan: the short segments through hgn_segment_reduce on the short CSR, the long ones by pieces.
 * Same outputs and conventions; (perm, rowptr) are the plan's own CSR. */
int hgn_segment_reduce_split(int dtype, const void* data, int64_t num_edges, int32_t D,
                             const int32_t* perm, const int32_t* rowptr, int64_t num_segments, const hgn_segment_split* split,
                             void* out_sum, void* out_mean, void* out_max, void* out_min,
                             int32_t* argmax, int32_t* argmin, int accumulate_sum,
                             void* workspace, size_t workspace_bytes, void* stream);

/* hgn_segment_sum_pair with a split on either side (NULL = that side has no long segment). */
int hgn_segment_sum_pair_split(int dtype, const void* data, int64_t num_edges, int32_t D,
                               const int32_t* perm_a, const int32_t* rowptr_a, int64_t num_segments_a,
                               const hgn_segment_split* split_a, void* out_a,
                               const int32_t* perm_b, const int32_t* rowptr_b, int64_t num_segments_b,
                               const hgn_segment_split* split_b, void* out_b,
                               void* workspace, size_t workspace_bytes, void* stream);

/* hgn_segment_reduce_bwd over a split plan, segment-wise (perm required, grad_data overwritten). */
int hgn_segment_reduce_bwd_split(int dtype, int64_t num_edges, int32_t D,
                                 const int32_t* ids32, const int32_t* perm, const int32_t* rowptr, int64_t num_segments,
                                 const hgn_segment_split* split,
                                 const void* g_sum, const void* g_mean, const void* g_max, const void* g_min,
                                 const int32_t* argmax, const int32_t* argmin, void* grad_data, void* stream);

/* hgn_segment_layer_grad over a split plan; the agg_grad row of a long segment is written once. */
int hgn_segment_layer_grad_split(int dtype, int64_t num_edges, int32_t D, const int32_t* perm, const int32_t* rowptr,
                                 int64_t num_segments, const hgn_segment_split* split,
                                 const void* g_sum, const void* g_mean, const void* g_max, const void* g_min,
                                 const int32_t* argmax, const int32_t* argmin, const void* base, void* agg_grad, void* edge_grad,
                                 void* stream);

/* fp32 partials of a segment reduction (the cluster pooling of a partitioned HyperGraphNet, combined across ranks before rounding):
 * row s of out ([S, HGN_SEGMENT_PARTIAL_WIDTH] fp32) is [sum 0..127 | max 128..255 | min 256..383 | count (int32 bits) | 3 x 0],
 * holding the values hgn_segment_reduce / hgn_segment_reduce_split would round to bf16 -- the same summation order, on the short
 * CSR and by pieces for the long segments -- and the segment's element count.  max / min and the winners are written only with
 * minmax; an empty segment leaves sum 0, max -inf, min +inf, winners -1, count 0.  bf16 rows of width 128; split may be NULL (no long
 * segment); the workspace is hgn_segment_split_reduce_workspace_bytes(split). */
#define HGN_SEGMENT_PARTIAL_WIDTH 388
int hgn_segment_partials(int dtype, const void* data, int64_t num_edges, int32_t D, const int32_t* perm, const int32_t* rowptr,
                         int64_t num_segments, const hgn_segment_split* split, int minmax, float* out, int32_t* argmax, int32_t* argmin,
                         void* workspace, size_t workspace_bytes, void* stream);

/* Backward of the row gathers v[senders], v[receivers] (torch.index_select -> index_add_ with float
 * atomics in the reference, src/migration/graphnet.py:28-29): out[n,:] = base[n,:] (if base != NULL)
 * + sum_k sum_{j in segment_k(n)} data_k[perm_k[j], :], accumulated in fp32 in a fixed order
 * (source k ascending, then ascending element id) and rounded once.  n_sources <= 4; out may alias base. */
typedef struct {
  int32_t n_sources;
  const void* data[4];          /* [E_k, D] rows of dtype */
  const int32_t* perm[4];       /* CSR permutation of source k */
  const int32_t* rowptr[4];     /* [S+1] */
} hgn_segment_sources;
int hgn_multi_segment_sum(int dtype, const hgn_segment_sources* sources, int64_t num_segments, int32_t D,
                          const void* base, void* out, void* stream);

/* ---- fused gather + MLP + LayerNorm + residual ("MLP tile") -----------------------------------
 * One call = one edge update (src/migration/graphnet.py:22-32) or one node update
 * (graphnet.py:34-48, 94-108, 110-124; heterographnet.py:17-33):
 *     x_row   = [ chunk_0[row] | chunk_1[row] | ... ]          each chunk 128 wide; chunk_c[row] =
 *               src_c[idx_c[row]] when idx_c != NULL (gathered sender / receiver latents) else
 *               src_c[row + row_offset_c]
 *     out_row = resid[row] + LayerNorm(W2 relu(W1 relu(W0 x + b0) + b1) + b2) * gamma + beta
 * The concatenation is never materialised (it replaces index_select x2 + cat + 3 addmm + 2 relu +
 * layer_norm + add = 9 launches).  Weights are the reference's nn.Linear tensors: W0[128, 128*n_chunks],
 * W1[128,128], W2[128,128] row-major fp32, biases/gamma/beta fp32[128] (meshgraphnet.py:53-60,93-108);
 * hgn_mlp_pack converts them once per optimiser step into the layout/precision the kernels stage. */
typedef struct {
  int32_t n_chunks;
  const void* src[HGN_MAX_CHUNKS];       /* [*,128] rows of dtype */
  const int32_t* idx[HGN_MAX_CHUNKS];    /* [rows] gather indices or NULL */
  int64_t row_offset[HGN_MAX_CHUNKS];    /* used when idx == NULL */
} hgn_chunks;

size_t hgn_mlp_packed_bytes(int dtype, int32_t n_chunks);
int hgn_mlp_pack(int dtype, int32_t n_chunks,
                 const float* W0, const float* b0, const float* W1, const float* b1,
                 const float* W2, const float* b2, const float* gamma, const float* beta,
                 void* packed, void* stream);

/* resid may alias one of the chunk sources (edge update: the edge latents; node update: the node
 * latents); out[rows,128] must not alias any input. */
int hgn_mlp_forward(int dtype, int64_t rows, const hgn_chunks* chunks, const void* packed,
                    const void* resid, int64_t resid_row_offset, void* out, void* stream);

/* Backward.  Activations are recomputed from the inputs (nothing but the inputs is saved by the
 * forward).  Outputs:
 *   grad_chunk[c][rows,128] : d loss / d chunk_c rows (before the scatter back through idx_c);
 *                             NULL = not needed.  resid_chunk >= 0 additionally adds grad_out (the
 *                             gradient of the residual branch, graphnet.py:32,48) into
 *                             grad_chunk[resid_chunk]; -1 leaves it to the caller.
 *   grad_W0[128,128*n_chunks], grad_b0, grad_W1, grad_b1, grad_W2, grad_b2, grad_gamma, grad_beta :
 *                             fp32, overwritten (deterministic two-stage reduction over row tiles). */
size_t hgn_mlp_backward_workspace_bytes(int dtype, int64_t rows, int32_t n_chunks);
int hgn_mlp_backward(int dtype, int64_t rows, const hgn_chunks* chunks, const void* packed,
                     const void* grad_out, int32_t resid_chunk, void* const* grad_chunk,
                     float* grad_W0, float* grad_b0, float* grad_W1, float* grad_b1,
                     float* grad_W2, float* grad_b2, float* grad_gamma, float* grad_beta,
                     void* workspace, size_t workspace_bytes, void* stream);

/* ---- encoder / decoder MLPs (bf16 tcgen05, fp32 TMEM accumulators; opt-in in the Python layer) ---------------
 * The reference's _make_mlp with num_layers = 2 (src/migration/meshgraphnet.py:93-108) on either side of the processor
 * (encoder.py, decoder.py):
 *   encoder  out[R,128] bf16 = LayerNorm(W2 relu(W1 relu(W0 x + b0) + b1) + b2) * gamma + beta,  x fp32 [R,K], 1 <= K <= 128
 *   decoder  out[N,n_out] fp32 = W2 relu(W1 relu(W0 x + b0) + b1) + b2,                          x bf16 [N,128], 1 <= n_out <= 16
 * No residual.  Weights are the nn.Linear tensors: encoder W0[128,K], decoder W2[n_out,128] and b2[n_out], the rest [128,128] /
 * [128]; hgn_io_mlp_pack stages them (bf16, zero-padded; `width` = K for the encoder, n_out for the decoder; gamma / beta may be
 * NULL for the decoder).  The forward / backward calls take the same `width` the blob was packed with.
 * Rounding points: x (encoder) and the weights are rounded to bf16; each hidden layer is fp32 sum + bias + ReLU rounded to bf16;
 * the encoder's LayerNorm runs in fp32 on acc + b2 and its output is rounded once to bf16; the decoder's output is acc + b2 in
 * fp32.  Backward: the decoder's upstream gradient is rounded to bf16 (it becomes an MMA operand); the chain follows the MLP tile's
 * rounding points; the encoder's grad_x[R,K] is fp32 (NULL = not requested), the decoder's grad_x[N,128] bf16 is required.  Weight,
 * bias, gamma and beta gradients are fp32 in the parameter shapes, overwritten, reduced in a fixed order (bitwise reproducible).
 * rows == 0 is valid: nothing is written by the forward and the backward writes exactly zero parameter gradients. */
enum { HGN_IO_ENCODER = 0, HGN_IO_DECODER = 1 };
#define HGN_IO_MAX_OUT 16
size_t hgn_io_mlp_packed_bytes(void);
int hgn_io_mlp_pack(int32_t kind, int32_t width,
                    const float* W0, const float* b0, const float* W1, const float* b1,
                    const float* W2, const float* b2, const float* gamma, const float* beta,
                    void* packed, void* stream);
int hgn_encoder_forward(int64_t rows, int32_t k_in, const float* x, const void* packed, void* out, void* stream);
size_t hgn_encoder_backward_workspace_bytes(int64_t rows, int32_t k_in);
int hgn_encoder_backward(int64_t rows, int32_t k_in, const float* x, const void* packed, const void* grad_out, float* grad_x,
                         float* grad_W0, float* grad_b0, float* grad_W1, float* grad_b1,
                         float* grad_W2, float* grad_b2, float* grad_gamma, float* grad_beta,
                         void* workspace, size_t workspace_bytes, void* stream);
int hgn_decoder_forward(int64_t rows, int32_t n_out, const void* x, const void* packed, float* out, void* stream);
size_t hgn_decoder_backward_workspace_bytes(int64_t rows, int32_t n_out);
int hgn_decoder_backward(int64_t rows, int32_t n_out, const void* x, const void* packed, const float* grad_out, void* grad_x,
                         float* grad_W0, float* grad_b0, float* grad_W1, float* grad_b1, float* grad_W2, float* grad_b2,
                         void* workspace, size_t workspace_bytes, void* stream);

/* ---- projected edge update (HGN_BF16 only; HGN_F32 returns HGN_ERR_UNSUPPORTED: use hgn_mlp_* there) --------
 * The edge update of src/migration/graphnet.py:22-32 with the first linear split by input block,
 * W0 = [Ws | Wr | We] (columns 0:128 | 128:256 | 256:384 of edge_models.<set>.0.layers.linear_0.weight):
 *     proj_s = v Ws^T, proj_r = v Wr^T                     once per NODE  (hgn_edge_project_forward)
 *     e'     = e + LN(W2 relu(W1 relu(proj_s[s] + proj_r[r] + We e + b0) + b1) + b2)     per edge
 * which replaces index_select x2 + cat + the K=384 addmm by two 128-wide row gathers and a K=128 GEMM.
 * `packed` is the hgn_mlp_pack blob of the edge MLP with n_chunks = 3.  senders/receivers: int32 [E]. */
int hgn_edge_project_forward(int dtype, int64_t num_nodes, const void* v, const void* packed,
                             void* proj_s, void* proj_r, void* stream);
/* grad_v[N,128] = grad_s Ws + grad_r Wr (+ grad_v_add when not NULL: the other consumers' share of d loss / d v, e.g. the node
 * update's, added in the kernel's epilogue instead of by a separate pass); grad_W0[128,384] columns 0:256 =
 * [grad_s^T v | grad_r^T v] (columns 256:384 are left untouched), where grad_s / grad_r are the sender- / receiver-keyed segment
 * sums of grad_pre0. */
size_t hgn_edge_project_backward_workspace_bytes(int dtype, int64_t num_nodes);
int hgn_edge_project_backward(int dtype, int64_t num_nodes, const void* v, const void* packed,
                              const void* grad_s, const void* grad_r, const void* grad_v_add, void* grad_v, float* grad_W0,
                              void* workspace, size_t workspace_bytes, void* stream);
int hgn_edge_update_forward(int dtype, int64_t num_edges, const void* edge, const void* proj_s, const void* proj_r,
                            const int32_t* senders, const int32_t* receivers, const void* packed, void* out, void* stream);
/* Backward (activations recomputed).  The incoming gradient of e' is  grad_out[e] + grad_agg[receivers[e]] :
 * grad_out[E,128] (may be NULL) is the dense part (next layer / loss), grad_agg[N,128] (may be NULL) the gradient
 * of the 'sum' aggregate of e' over receivers (graphnet.py:50-70), gathered here instead of being expanded to
 * [E,128] by a separate kernel.  Outputs: grad_edge[E,128] = d loss / d e (residual branch included);
 * grad_pre0[E,128] = d loss / d (first-layer pre-activation), whose sender- and receiver-keyed segment sums are
 * the inputs of hgn_edge_project_backward; grad_W0 columns 256:384 (= We) only; all other parameter gradients
 * complete (fp32, overwritten, fixed-order reductions). */
size_t hgn_edge_update_backward_workspace_bytes(int dtype, int64_t num_edges);
int hgn_edge_update_backward(int dtype, int64_t num_edges, const void* edge, const void* proj_s, const void* proj_r,
                             const int32_t* senders, const int32_t* receivers, const void* packed,
                             const void* grad_out, const void* grad_agg, void* grad_edge, void* grad_pre0,
                             float* grad_W0, float* grad_b0, float* grad_W1, float* grad_b1,
                             float* grad_W2, float* grad_b2, float* grad_gamma, float* grad_beta,
                             void* workspace, size_t workspace_bytes, void* stream);

/* ---- node update with 1..4 aggregates (HGN_BF16 only) -- src/migration/graphnet.py:34-48 with one edge set -----------------
 *     v' = v + LN(W2 relu(W1 relu(Wv v + sum_j Wa_j agg_j + b0) + b1) + b2),   W0 = [Wv | Wa_1 | ... | Wa_n] = node_model_cross.0.layers.linear_0.weight
 * n_agg = 1 ('sum', 'mean', 'max' or 'min') or 4 ('pna': sum, mean, max, min in the order of graphnet.py:53-64); aggs[j] is [N,128] bf16.
 * `packed` is the hgn_mlp_pack blob of the node MLP with n_chunks = 1 + n_agg.  q1 (and q2 when n_agg > 2; caller-owned [N,128] bf16)
 * receive agg_1 Wa_1^T + agg_2 Wa_2^T and agg_3 Wa_3^T + agg_4 Wa_4^T; the recompute backward reads them again.  Runs on the projected
 * edge kernels: the q tables play the roles of the node tables, gathered through the identity.
 * Backward: grad_v = d loss / d v (residual branch included), grad_aggs[j] = d loss / d agg_j, and every parameter gradient (fp32,
 * overwritten, fixed-order reductions).  num_nodes must be > 0 for the backward. */
int hgn_node_update_forward(int dtype, int64_t num_nodes, const void* v, int32_t n_agg, const void* const* aggs, const void* packed,
                            void* q1, void* q2, void* out, void* stream);
size_t hgn_node_update_backward_workspace_bytes(int dtype, int64_t num_nodes);
int hgn_node_update_backward(int dtype, int64_t num_nodes, const void* v, int32_t n_agg, const void* const* aggs,
                             const void* q1, const void* q2, const void* packed,
                             const void* grad_out, void* grad_v, void* const* grad_aggs,
                             float* grad_W0, float* grad_b0, float* grad_W1, float* grad_b1,
                             float* grad_W2, float* grad_b2, float* grad_gamma, float* grad_beta,
                             void* workspace, size_t workspace_bytes, void* stream);

/* ---- column sums ------------------------------------------------------------------------------
 * out[D] (fp32) = sum over rows of x[rows, D]; two-stage fixed-order reduction (LayerNorm beta / bias
 * gradients).  D must be a multiple of 4, at most 256 and a divisor of 1024 (4, 8, 16, 32, 64, 128 or 256: one block's 256
 * threads cover the D / 4 column groups); any other D returns HGN_ERR_INVALID_ARGUMENT. */
size_t hgn_colsum_workspace_bytes(int64_t rows, int32_t D);
int hgn_colsum(int dtype, const void* x, int64_t rows, int32_t D, float* out,
               void* workspace, size_t workspace_bytes, void* stream);

/* ---- halo exchange helpers (edge-cut partitioning, SURVEY.md s8e) -------------------------------
 * pack:   dst[i,:] = src[idx[i],:]            boundary rows -> contiguous send buffer
 * unpack: dst[idx[i],:] = src[i,:]            received ghost rows -> local ghost slots
 * unpack_add (backward): dst[idx[i],:] += src[i,:], idx unique per call (one peer at a time, peers in
 *         rank order -> deterministic). */
int hgn_rows_gather(int dtype, const void* src, const int32_t* idx, int64_t n, int32_t D, void* dst, void* stream);
int hgn_rows_scatter(int dtype, const void* src, const int32_t* idx, int64_t n, int32_t D, void* dst,
                     int accumulate, void* stream);

/* ---- halo exchange over NVLink peer memory (one process per GPU) ----------------------------------------------------
 * hgn_peer_alloc: cudaMalloc'ed, zero-filled exchange pool of this rank + its 64-byte CUDA IPC handle (send it to the peers,
 * e.g. with torch.distributed.all_gather); hgn_peer_open maps a peer's pool into this process (peer access over NVLink is enabled
 * lazily); _close / _free undo them.
 * hgn_halo_push: for every peer q, rows send_index[row_begin[q] .. row_begin[q+1]) of `table` ([*, D]) are stored into dst[q]
 * (a pointer INTO the peer's mapped pool: where its ghost rows / gradient inbox for this rank start), then flag[q] (a uint32 in
 * the peer's pool) is set to `epoch` -- after all rows of all peers have been written and fenced.  `counter` is a zero-initialised
 * uint32 in this rank's memory used by the kernel to find its last CTA (re-armed by the kernel).
 * hgn_halo_wait: makes `stream` wait until every flag[q] (uint32s in THIS rank's pool, written by the peers) has reached `epoch`
 * (wrap-safe comparison).  Epochs are the running number of the exchange, the same on all ranks; flags are never reset. */
#define HGN_MAX_PEERS 16
typedef struct {
  void* dst[HGN_MAX_PEERS];
  void* flag[HGN_MAX_PEERS];
  int64_t row_begin[HGN_MAX_PEERS + 1];
} hgn_halo_peers;
typedef struct {
  const void* flag[HGN_MAX_PEERS];
} hgn_halo_flags;
int hgn_peer_alloc(size_t bytes, void** ptr, unsigned char* handle64);
int hgn_peer_open(const unsigned char* handle64, void** ptr);
int hgn_peer_close(void* ptr);
int hgn_peer_free(void* ptr);
int hgn_halo_push(int dtype, const void* table, const int32_t* send_index, int32_t D, const hgn_halo_peers* peers, int32_t n_peers,
                  uint32_t epoch, void* counter, void* stream);
int hgn_halo_wait(const hgn_halo_flags* flags, int32_t n_flags, uint32_t epoch, void* stream);

/* ---- cluster pooling across ranks (partitioned HyperGraphNet; the rows travel with hgn_halo_push / hgn_halo_wait) -------------
 * hgn_cluster_combine: slots = [world][C][HGN_SEGMENT_PARTIAL_WIDTH] fp32, every rank's hgn_segment_partials rows in rank order.
 * Per cluster and feature, in rank order: sum = bf16_rn((((0 + s_0) + s_1) + ...)), mean = bf16_rn(total * (1.0f / max(cnt, 1))),
 * max / min over the ranks with a nonzero count (strict comparisons: the lowest rank wins a tie; 0 when every count is 0).  Any output
 * may be NULL.  argmax / argmin are this rank's local winners: cleared to -1 where another rank won.  count (may be NULL) receives
 * the total counts.  Every rank runs this on the same bytes, so the outputs are bit-identical on every rank.
 * hgn_cluster_grad_sum: out[C, D] = bf16_rn(sum over r in rank order of slots[r]) from +0 in fp32; slots = [world][C][D] bf16.
 * hgn_cluster_mean_grad: out = bf16_rn(fma(g_mean, 1.0f / max(count, 1), 0 + g_sum)) per [C, 128] bf16 row (g_sum may be NULL):
 * the 'sum' and 'mean' gradient of a pooled cluster as one sum term for hgn_segment_reduce_bwd on the local elements. */
int hgn_cluster_combine(const float* slots, int32_t world, int32_t rank, int64_t num_clusters, void* out_sum, void* out_mean,
                        void* out_max, void* out_min, int32_t* argmax, int32_t* argmin, int32_t* count, void* stream);
int hgn_cluster_grad_sum(int dtype, const void* slots, int32_t world, int64_t num_clusters, int32_t D, void* out, void* stream);
int hgn_cluster_mean_grad(const void* g_sum, const void* g_mean, const int32_t* count, int64_t num_clusters, void* out, void* stream);

/* ---- world edges: fixed-radius neighbour search ----------------------------------------------------
 * Replaces the dense search of PlateModel.build_graph (src/model/plate.py:86-110): torch.cdist over all
 * node pairs, `< radius`, diagonal and existing mesh edges removed, senders restricted to sender_type
 * (OBSTACLE) and receivers to receiver_type (NORMAL), then torch.nonzero.  A uniform-grid cell list gives
 * the identical (sender, receiver) list in torch.nonzero's row-major order, int64, with the distance
 * evaluated in torch.cdist's own fp32 arithmetic (see csrc/world_edges.cu).  world_pos is [N,3] fp32,
 * node_type [N] int32, mesh_senders / mesh_receivers the reference's int64 two-way mesh edges.
 * Two calls because the output size is data dependent (torch.nonzero synchronises for the same reason):
 * _count fills the workspace, synchronises the stream and returns the number of pairs in *host_num_pairs;
 * _emit writes them from the same (unmodified) workspace and inputs. */
size_t hgn_world_edges_workspace_bytes(int64_t num_nodes, int64_t num_mesh_edges);
int hgn_world_edges_count(const float* world_pos, const int32_t* node_type, int64_t num_nodes,
                          const int64_t* mesh_senders, const int64_t* mesh_receivers, int64_t num_mesh_edges,
                          float radius, int32_t sender_type, int32_t receiver_type,
                          void* workspace, size_t workspace_bytes, int64_t* host_num_pairs, void* stream);
int hgn_world_edges_emit(const float* world_pos, const int32_t* node_type, int64_t num_nodes, int64_t num_mesh_edges,
                         float radius, int32_t sender_type, const void* workspace, size_t workspace_bytes,
                         int64_t* senders_out, int64_t* receivers_out, int64_t capacity, void* stream);

/* ---- kernel timing (tracing hook; the reference only has wall-clock time.time() around a batch,
 * src/algorithms/MeshSimulator.py:135-155) ----------------------------------------------------------
 * When enabled, every kernel launch inside the library is bracketed by CUDA events on the launching
 * stream.  hgn_profile_report synchronises the device and writes a JSON array
 * [{"name": "...", "launches": n, "ms": total_ms}, ...] into buf (truncated to buf_bytes, always
 * NUL-terminated) and returns the number of bytes needed. */
int hgn_profile_enable(int on);
int hgn_profile_reset(void);
size_t hgn_profile_report(char* buf, size_t buf_bytes);

/* ---- host-buffer convenience (the end-to-end path timed by bench.py "e2e") ---------------------
 * Not part of the reference API; copies pinned host rows to the device and back on `stream`. */
int hgn_copy_h2d(void* dst_device, const void* src_host, size_t bytes, void* stream);
int hgn_copy_d2h(void* dst_host, const void* src_device, size_t bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HGN_B200_H_ */
