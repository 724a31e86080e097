/* fgnn_b200.h -- C ABI of libfgnn_b200.so: the B200 (sm_100a) implementation of the
 * 2-FGNN siamese hot path of mlelarge/graph_neural_net.
 *
 * The reference has no FFI: its boundary is the Python API (SURVEY.md section 8b).  Each entry point
 * below states which reference call site it replaces (paths relative to the reference tree).
 * The Python mirror of the reference interface (graph_neural_net_b200/models, maskedtensors,
 * toolbox) binds these symbols with ctypes; see INTEGRATION.md for the stub a reference
 * maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - tensors are dense row-major fp32 with the reference's shapes: activations (G,C,N,N),
 *     node vectors (G,C,N), scores (G,N,N); N is the padded size (Nmax of the batch);
 *   - n_per_graph: int32[G] true vertex counts (prefix masks of maskedtensor.from_list,
 *     maskedtensors/maskedtensor.py:40-46), or NULL when every graph has exactly N vertices;
 *     padded positions of every output are written as exact zeros (maskedtensor.py:87-90);
 *   - graph pairs of unequal sizes: the *_pair_* entry points take graph 1 (rows i) padded to N1 with sizes n1 and
 *     graph 2 (columns j) padded to N2 with sizes n2 (either NULL when every graph has its padded size): e1 (G,C,N1),
 *     e2 (G,C,N2), scores (G,N1,N2), zero outside the n1 x n2 block.  The loss keeps the reference's ground truth,
 *     row i <-> column i: rows i >= n2[g] carry no target and add nothing to ce_sum, correct or the gradient (the
 *     loss is meant for n1 <= n2, where CrossEntropyLoss(out, arange(n1)) is defined).  Each square entry point is
 *     its pair form with N1 = N2 = N and n1 = n2 = n_per_graph;
 *   - stream: a cudaStream_t passed as void*; all work is enqueued there, no hidden syncs;
 *   - the library never allocates device memory: callers size scratch with the *_workspace_bytes
 *     query and own every buffer;
 *   - return value: FGNN_OK or an fgnn_status error code; fgnn_last_error() gives text.
 */
#ifndef FGNN_B200_H
#define FGNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  FGNN_OK = 0,
  FGNN_ERR_INVALID = 1,      /* bad argument (shape, null pointer, alignment)            */
  FGNN_ERR_UNSUPPORTED = 2,  /* valid request this build cannot serve (e.g. C > 128)     */
  FGNN_ERR_CUDA = 3,         /* a CUDA runtime / driver call failed                      */
  FGNN_ERR_WORKSPACE = 4     /* workspace too small                                      */
} fgnn_status;

typedef enum {
  FGNN_FP32 = 0,  /* CUDA-core fp32 everywhere: parity mode (<= 1e-4 rel. on embeddings)        */
  FGNN_BF16 = 1,  /* tcgen05 kind::f16 with bf16 operands, fp32 accumulate / statistics        */
  FGNN_FP16 = 2   /* same kernels and speed with fp16 operands (8x smaller rounding error)     */
} fgnn_precision;

/* Deterministic mode: ORed into the `precision` argument of the embedder entry points (fgnn_embed_workspace_bytes,
 * fgnn_embed_fwd, fgnn_embed_fwd_adjacency_u8, fgnn_embed_train_workspace_bytes, fgnn_embed_fwd_train, fgnn_embed_bwd)
 * and passed as `flags` to fgnn_mlp_workspace_bytes_ex / fgnn_mlp_bwd_f32_ex.  Every sum whose partials come from
 * several CTAs (GraphNorm statistics, bias and weight gradients) is then formed from per-CTA records added in a fixed
 * order instead of floating-point atomics, so that, for the same build, device model, inputs, batch composition,
 * FGNN_TC_* variables and parameters, the embeddings and parameter gradients are bit-identical from run to run.  Not
 * covered: a graph alone vs inside a batch, keep-all vs recompute plans (the reduction partitions differ), multi-GPU
 * all-reduce order.  The workspaces are larger (they hold the records): the workspace query, the forward and the
 * backward of one training call must all take the same flag, as they must see the same FGNN_TC_* variables.  The fused
 * head (fgnn_head_*) accepts the bit and ignores it: it is deterministic in both modes.  Any other bit outside the
 * precision's low byte is rejected (FGNN_ERR_INVALID; workspace queries return 0). */
#define FGNN_DETERMINISTIC 0x100

#define FGNN_MAX_DEPTH 8
#define FGNN_MAX_BLOCKS 16

/* One MlpBlock_Real: depth x Conv2d(k=1) + GraphNorm  (models/layers.py:109-131).
 * w[k]: (c_out, c_in_k) row-major (== Conv2d weight (Co,Ci,1,1)), b[k]: (c_out).
 * gn_w/gn_b: (c_out) (== GraphNorm (1,C,1,1), models/layers.py:47-69). */
typedef struct {
  int32_t c_in;
  int32_t c_out;
  int32_t depth;
  const float* w[FGNN_MAX_DEPTH];
  const float* b[FGNN_MAX_DEPTH];
  const float* gn_w;
  const float* gn_b;
  float eps; /* 1e-5 in the reference */
  /* GraphNorm's n (models/layers.py:76-79): 1 = constant_n_vertices=True, n = the padded size N even for a ragged
   * batch (the reference's default; mean / variance still run over each graph's own n_g x n_g block);
   * 0 = constant_n_vertices=False, n = the graph's own vertex count n_g.  Irrelevant when n_per_graph is NULL. */
  int32_t constant_n;
} fgnn_mlp_params;

/* Gradients of the above, same shapes; accumulated into (+=), caller zeroes them. */
typedef struct {
  float* w[FGNN_MAX_DEPTH];
  float* b[FGNN_MAX_DEPTH];
  float* gn_w;
  float* gn_b;
} fgnn_mlp_grads;

/* One `block` of models/blocks_emb.py:16-27: mlp3(cat[mlp1(x) @ mlp2(x), x]). */
typedef struct {
  fgnn_mlp_params mlp1, mlp2, mlp3;
} fgnn_block_params;

/* node_embedding: num_blocks blocks + ColumnMaxPooling (models/blocks_emb.py:29-43). */
typedef struct {
  int32_t num_blocks;
  fgnn_block_params block[FGNN_MAX_BLOCKS];
} fgnn_embed_params;

/* Parameter gradients of the above (same shapes, accumulated into: the caller zeroes them). */
typedef struct {
  fgnn_mlp_grads mlp1, mlp2, mlp3;
} fgnn_block_grads;
typedef struct {
  int32_t num_blocks;
  fgnn_block_grads block[FGNN_MAX_BLOCKS];
} fgnn_embed_grads;

/* ---- library ---------------------------------------------------------------------------- */
const char* fgnn_version(void);
const char* fgnn_last_error(void); /* thread-local text of the last failure */
/* 1 if the current device is sm_100 (tcgen05 paths usable), 0 otherwise */
int fgnn_device_supports_tcgen05(void);

/* ---- fp32 per-operator entry points (each mirrors one reference module) ------------------ */

/* MlpBlock_Real.forward (models/layers.py:126-131), also its MaskedTensor form
 * (maskedtensor.py:230-238 conv2d override + layers.py:76-79 per-graph n).
 * x (G,c_in,N,N) -> y (G,c_out,N,N).  stats (G,c_out,2) receives {mean, 1/(2*sqrt(n*(var+eps)))}
 * of the pre-norm activations (kept for backward).  workspace: fgnn_mlp_workspace_bytes. */
size_t fgnn_mlp_workspace_bytes(int32_t G, int32_t c_in, int32_t c_out, int32_t depth, int32_t N);
int fgnn_mlp_fwd_f32(const fgnn_mlp_params* p, const float* x, float* y, float* stats, int32_t G,
                     int32_t N, const int32_t* n_per_graph, void* workspace, size_t workspace_bytes,
                     void* stream);
/* Backward of the above.  Hidden activations are recomputed from x (nothing but x and stats is
 * saved).  dy (G,c_out,N,N) -> dx (G,c_in,N,N) (may be NULL), parameter grads accumulated. */
int fgnn_mlp_bwd_f32(const fgnn_mlp_params* p, const fgnn_mlp_grads* g, const float* x,
                     const float* stats, const float* dy, float* dx, int32_t G, int32_t N,
                     const int32_t* n_per_graph, void* workspace, size_t workspace_bytes,
                     void* stream);
/* The same with flags: 0 or FGNN_DETERMINISTIC (fixed-order parameter-gradient sums; the backward's workspace must be
 * sized by fgnn_mlp_workspace_bytes_ex with the same flags).  The two functions above are these with flags 0. */
size_t fgnn_mlp_workspace_bytes_ex(int32_t G, int32_t c_in, int32_t c_out, int32_t depth, int32_t N, int32_t flags);
int fgnn_mlp_bwd_f32_ex(const fgnn_mlp_params* p, const fgnn_mlp_grads* g, const float* x, const float* stats,
                        const float* dy, float* dx, int32_t G, int32_t N, const int32_t* n_per_graph, void* workspace,
                        size_t workspace_bytes, void* stream, int32_t flags);

/* GraphNorm.forward / normalize (models/layers.py:68-80).  gn_w/gn_b may be NULL (plain
 * normalize).  stats (G,C,2) as above, required: the normalisation reads it back.  constant_n: see fgnn_mlp_params. */
int fgnn_graphnorm_fwd_f32(const float* x, float* y, float* stats, const float* gn_w,
                           const float* gn_b, float eps, int32_t constant_n, int32_t G, int32_t C, int32_t N,
                           const int32_t* n_per_graph, void* stream);

/* Matmul.forward: torch.matmul over the last two dims (models/layers.py:161-162).
 * a,b,out (G,C,N,N); padded rows/cols ignored and written as zero. */
int fgnn_matmul_fwd_f32(const float* a, const float* b, float* out, int32_t G, int32_t C, int32_t N,
                        const int32_t* n_per_graph, void* stream);
/* da = dout @ b^T, db = a^T @ dout (either may be NULL). */
int fgnn_matmul_bwd_f32(const float* a, const float* b, const float* dout, float* da, float* db,
                        int32_t G, int32_t C, int32_t N, const int32_t* n_per_graph, void* stream);

/* ColumnMaxPooling.forward: max over the last dim (models/layers.py:194-203; masked form
 * maskedtensor.py:213-228).  x (G,C,N,N) -> out (G,C,N); argmax (G,C,N) int32 may be NULL. */
int fgnn_colmax_fwd_f32(const float* x, float* out, int32_t* argmax, int32_t G, int32_t C, int32_t N,
                        const int32_t* n_per_graph, void* stream);
int fgnn_colmax_bwd_f32(const float* dout, const int32_t* argmax, float* dx, int32_t G, int32_t C,
                        int32_t N, const int32_t* n_per_graph, void* stream);

/* Input construction on the device (SURVEY 8(f) row 2): adjacency_matrix_to_tensor_representation
 * (loaders/data_generator.py:118-125) followed by the zero padding of maskedtensor.from_list
 * (maskedtensors/maskedtensor.py:8-48) for a whole batch.  adj (G,N,N) uint8 in {0,1}, row-major, only the
 * leading n_g x n_g block of graph g is read; out (G,2,N,N) float32: out[g,0] = W, out[g,1] = diag(W.sum(1)),
 * zero outside the n_g x n_g block.  Ships 1 byte per entry over PCIe instead of 8. */
int fgnn_features_from_adjacency_u8(const uint8_t* adj, float* out, int32_t G, int32_t N,
                                    const int32_t* n_per_graph, void* stream);

/* Synthetic graph pairs on the device (loaders/data_generator.py:39-87): adj1[g] ~ generator(edge_density, n_g) with
 * generator 0 = "ErdosRenyi" (:39-44), 1 = "Regular" (:58-68: d = int(edge_density n), +1 if n d is odd; sampled by the
 * switch chain from a relabelled circulant graph), and adj2[g] = noise_erdos_renyi(adj1[g]) = W (1 - N1) + (1 - W) N2,
 * N1 ~ ER(noise), N2 ~ ER(edge_density noise / (1 - edge_density)) (:79-87).  uint8 (G,N,N), zero outside n_g x n_g;
 * counter-based generator: the same seed gives the same graphs.  Parity with networkx is distributional.
 * 2 <= N <= 4096.  "Regular" runs its switch chain on one thread per graph (10 |E| proposals, time grows with |E|);
 * its workspace holds the edge lists and, above N = 1264, the adjacency bitmaps (G N ceil(N/32) words). */
size_t fgnn_generate_workspace_bytes(int32_t G, int32_t N, int32_t generator);
int fgnn_generate_pairs_u8(uint8_t* adj1, uint8_t* adj2, int32_t G, int32_t N, const int32_t* n_per_graph,
                           int32_t generator, float edge_density, float noise, uint64_t seed, void* workspace,
                           size_t workspace_bytes, void* stream);

/* Siamese head: scores[g] = e1[g]^T e2[g]  (models/trainers.py:67).  e1,e2 (G,C,N) -> (G,N,N). */
int fgnn_scores_fwd_f32(const float* e1, const float* e2, float* scores, int32_t G, int32_t C,
                        int32_t N, const int32_t* n_per_graph, void* stream);
int fgnn_scores_bwd_f32(const float* e1, const float* e2, const float* dscores, float* de1,
                        float* de2, int32_t G, int32_t C, int32_t N, const int32_t* n_per_graph,
                        void* stream);
/* Pair forms: e1 (G,C,N1), e2 (G,C,N2) -> scores (G,N1,N2); de1 (G,C,N1), de2 (G,C,N2). */
int fgnn_scores_pair_fwd_f32(const float* e1, const float* e2, float* scores, int32_t G, int32_t C, int32_t N1,
                             int32_t N2, const int32_t* n1, const int32_t* n2, void* stream);
int fgnn_scores_pair_bwd_f32(const float* e1, const float* e2, const float* dscores, float* de1, float* de2, int32_t G,
                             int32_t C, int32_t N1, int32_t N2, const int32_t* n1, const int32_t* n2, void* stream);

/* Row-softmax cross-entropy against the identity matching + row argmax, one pass
 * (toolbox/losses.py:20-34 and toolbox/metrics.py:118-141 without the per-graph host loop).
 * scores (G,N,N) -> ce_sum[G] (sum_i lse_i - s_ii), correct[G] (#rows with argmax == i),
 * row_lse (G,N) may be NULL (kept for backward).  One warp per row + a fixed-order per-graph reduction
 * (deterministic); workspace: fgnn_ce_workspace_bytes. */
size_t fgnn_ce_workspace_bytes(int32_t G, int32_t N);
int fgnn_ce_argmax_fwd_f32(const float* scores, float* ce_sum, int32_t* correct, float* row_lse,
                           int32_t G, int32_t N, const int32_t* n_per_graph, void* workspace,
                           size_t workspace_bytes, void* stream);
/* dscores[g,i,j] = coef[g] * (softmax(scores[g,i,:])[j] - [i==j]); coef folds the loss
 * reduction and the upstream gradient. */
int fgnn_ce_bwd_f32(const float* scores, const float* row_lse, const float* coef, float* dscores,
                    int32_t G, int32_t N, const int32_t* n_per_graph, void* stream);
/* Pair forms: scores (G,N1,N2), the softmax of row i over its n2[g] valid columns; row_lse (G,N1); workspace:
 * fgnn_ce_workspace_bytes(G, N1).  row_argmax (G,N1) int32 may be NULL: the arg-max column of every row i < n1[g]
 * (ties: the lowest column), -1 on padded rows. */
int fgnn_ce_pair_argmax_fwd_f32(const float* scores, float* ce_sum, int32_t* correct, float* row_lse, int32_t* row_argmax,
                                int32_t G, int32_t N1, int32_t N2, const int32_t* n1, const int32_t* n2, void* workspace,
                                size_t workspace_bytes, void* stream);
int fgnn_ce_pair_bwd_f32(const float* scores, const float* row_lse, const float* coef, float* dscores, int32_t G,
                         int32_t N1, int32_t N2, const int32_t* n1, const int32_t* n2, void* stream);

/* Fused siamese head on tensor cores (FGNN_BF16 / FGNN_FP16): scores = e1^T e2 (models/trainers.py:67) with the
 * row-softmax cross-entropy against the identity matching (toolbox/losses.py:27-33) and the row argmax
 * (toolbox/metrics.py:125-134) in the epilogue of the tcgen05 GEMM, flash style: online row max / sum of exponentials
 * over 256-column tiles.  e1,e2 (G,C,N) fp32 are split into 16-bit (hi, lo) operand pairs in shared memory
 * (Ahi Bhi + Alo Bhi + Ahi Blo: fp32-level accuracy), C a multiple of 16, at most 128.  ce_sum[G], correct[G] as
 * fgnn_ce_argmax_fwd_f32; scores (G,N,N) is written only when non-NULL (zero outside the n_g x n_g block).  N <= 4096,
 * G <= 65535.  Training goes through fgnn_head_fwd_train / fgnn_head_bwd below. */
size_t fgnn_head_workspace_bytes(int32_t G, int32_t N);
int fgnn_head_fwd(int32_t precision, const float* e1, const float* e2, float* scores, float* ce_sum, int32_t* correct,
                  int32_t G, int32_t C, int32_t N, const int32_t* n_per_graph, void* workspace, size_t workspace_bytes,
                  void* stream);
/* Training form of the fused head: the scores (models/trainers.py:67) and the summed cross-entropy against the identity
 * matching (toolbox/losses.py:27-34) with autograd's backward through both, without ever forming the (G,N,N) scores
 * or their gradient (fgnn_scores_* + fgnn_ce_* keep two such tensors per step).
 * fgnn_head_fwd_train: ce_sum, correct bit-identical to fgnn_head_fwd, plus row_lse (G,N) fp32 = log sum_j exp(s_ij)
 * of every valid row (0 for i >= n_g), kept for the backward; workspace as fgnn_head_workspace_bytes.
 * fgnn_head_bwd: coef[G] = d loss / d ce_sum[g] (device);  with dS_ij = coef[g] (softmax(s_i)_j - [i == j]) it
 * OVERWRITES de1[g,:,i] = sum_j dS_ij e2[g,:,j] and de2[g,:,j] = sum_i dS_ij e1[g,:,i] (G,C,N), zero at positions
 * >= n_g -- what fgnn_ce_bwd_f32 followed by fgnn_scores_bwd_f32 compute.  S is recomputed from the (hi, lo) operands
 * and dS is split into (hi, lo) operands too (fp32-level gradients); coef scales the fp32 accumulator.  Deterministic
 * (every output written once, no atomics).  The backward needs no workspace (NULL, 0 are accepted).  Both calls take
 * FGNN_BF16 / FGNN_FP16, C a multiple of 16 at most 128, N <= 4096, G <= 65535. */
int fgnn_head_fwd_train(int32_t precision, const float* e1, const float* e2, float* ce_sum, int32_t* correct, float* row_lse,
                        int32_t G, int32_t C, int32_t N, const int32_t* n_per_graph, void* workspace, size_t workspace_bytes,
                        void* stream);
int fgnn_head_bwd(int32_t precision, const float* e1, const float* e2, const float* row_lse, const float* coef, float* de1,
                  float* de2, int32_t G, int32_t C, int32_t N, const int32_t* n_per_graph, void* workspace,
                  size_t workspace_bytes, void* stream);
/* Pair forms of the fused head: e1 (G,C,N1), e2 (G,C,N2), scores (G,N1,N2), row_lse (G,N1), de1 (G,C,N1), de2 (G,C,N2);
 * N1, N2 <= 4096.  The workspace depends on N1 only: fgnn_head_pair_workspace_bytes(G, N1) ==
 * fgnn_head_workspace_bytes(G, N1). */
size_t fgnn_head_pair_workspace_bytes(int32_t G, int32_t N1);
int fgnn_head_pair_fwd(int32_t precision, const float* e1, const float* e2, float* scores, float* ce_sum, int32_t* correct,
                       int32_t G, int32_t C, int32_t N1, int32_t N2, const int32_t* n1, const int32_t* n2, void* workspace,
                       size_t workspace_bytes, void* stream);
int fgnn_head_pair_fwd_train(int32_t precision, const float* e1, const float* e2, float* ce_sum, int32_t* correct,
                             float* row_lse, int32_t G, int32_t C, int32_t N1, int32_t N2, const int32_t* n1,
                             const int32_t* n2, void* workspace, size_t workspace_bytes, void* stream);
int fgnn_head_pair_bwd(int32_t precision, const float* e1, const float* e2, const float* row_lse, const float* coef,
                       float* de1, float* de2, int32_t G, int32_t C, int32_t N1, int32_t N2, const int32_t* n1,
                       const int32_t* n2, void* workspace, size_t workspace_bytes, void* stream);

/* accuracy_linear_assignment (toolbox/metrics.py:92-116), the metric training_step / validation_step call
 * (models/trainers.py:53,74): per graph the assignment scipy.optimize.linear_sum_assignment returns on
 * cost = -log_softmax(scores, -1) (fp32 weights formed in the kernel), found on the device by shortest augmenting
 * paths in double precision with scipy's operation order and tie rule, one CTA per graph.  scores (G,N,N);
 * col_of_row (G,N) int32 (rows >= n_g get -1; may be NULL); correct[G] = #rows with col(i) == i;
 * total_cost[G] = sum_i cost[i, col(i)] (may be NULL).  The working arrays take 53 N bytes of shared memory, so N is
 * limited by the device's opt-in shared memory per block: N <= 4380 on sm_100 (227 KB); beyond it the call fails
 * with FGNN_ERR_UNSUPPORTED and states the limit. */
int fgnn_lap_fwd(const float* scores, int32_t* col_of_row, int32_t* correct, double* total_cost, int32_t G,
                 int32_t N, const int32_t* n_per_graph, void* stream);
/* Rectangular form, as scipy's rectangular_lsap: scores (G,N1,N2), cost = -log_softmax over each row's n2[g] valid
 * columns; min(n1, n2) pairs are matched (the problem is solved transposed when n1 > n2).  col_of_row (G,N1): -1 on
 * padded rows and on rows left without a column.  The shared-memory limit above applies to max(N1, N2). */
int fgnn_lap_pair_fwd(const float* scores, int32_t* col_of_row, int32_t* correct, double* total_cost, int32_t G,
                      int32_t N1, int32_t N2, const int32_t* n1, const int32_t* n2, void* stream);

/* ---- fused embedder (the hot path proper) ------------------------------------------------ */

/* node_embedding forward for G graphs: x (G,c_in0,N,N) fp32 -> emb (G,C,N) fp32, C = the last block's c_out.
 * Replaces Network.forward over the 4-block DAG + ColumnMaxPooling
 * (models/utils.py:63-69, models/blocks_emb.py:16-43, models/trainers.py:64-65).
 *   precision FGNN_FP32 : composition of the fp32 operators above.
 *   precision FGNN_BF16 / FGNN_FP16 : TMA + tcgen05/TMEM kernels; activations live in HBM as
 *     16-bit pre-normalisation planes, GraphNorm is folded into the consumers (DESIGN.md).  N <= 4096; the
 *     batch is cut into passes of equal size, each within FGNN_TC_WS_GB (default 16) GB of planes when a graph
 *     fits (one graph takes 11.6 GB at N = 4096, C = 64, a pass is never less than one graph).
 *     Widths: every block's c_out (shared by its three MLPs) is 1 .. 64 and c_in0 <= 64, with the parameters in
 *     their real shapes.  The kernels run at width 32 when every c_out is <= 32, else 64, with the padded channels
 *     exactly zero (the library pads the parameters itself); the workspace is that of the uniform model of that
 *     width.  A c_out above 64 fails with FGNN_ERR_UNSUPPORTED.
 * workspace: fgnn_embed_workspace_bytes(...) bytes, 1024-byte aligned (0 when the shape is unsupported). */
size_t fgnn_embed_workspace_bytes(const fgnn_embed_params* p, int32_t precision, int32_t G, int32_t N);
int fgnn_embed_fwd(const fgnn_embed_params* p, int32_t precision, const float* x, float* emb,
                   int32_t G, int32_t N, const int32_t* n_per_graph, void* workspace, size_t workspace_bytes,
                   void* stream);

/* Same embedder fed from a uint8 adjacency batch (G,N,N) instead of the fp32 (G,2,N,N) features: the two
 * input planes W and diag(W.sum(1)) (loaders/data_generator.py:118-125) are built on the device straight into
 * the 16-bit plane layout.  FGNN_BF16 / FGNN_FP16 only; workspace as for fgnn_embed_fwd. */
int fgnn_embed_fwd_adjacency_u8(const fgnn_embed_params* p, int32_t precision, const uint8_t* adj, float* emb,
                                int32_t G, int32_t N, const int32_t* n_per_graph, void* workspace,
                                size_t workspace_bytes, void* stream);

/* 16-bit TRAINING of the embedder: what autograd does to Network.forward under Lightning's precision=16
 * (models/trainers.py:70-76, commander_explore.py:120-123), with every contraction of both passes on tcgen05.
 * fgnn_embed_fwd_train computes the same embeddings as fgnn_embed_fwd (FGNN_BF16 / FGNN_FP16) and leaves in
 * `workspace` what backward needs (hidden activations, pre-norm planes, GraphNorm statistics, pooling arg-max);
 * fgnn_embed_bwd takes d loss / d emb (G,C,N) fp32 (C = the last block's c_out) and ACCUMULATES d loss / d parameter
 * into `grads` (fp32, the real shapes of the parameters: widths as for fgnn_embed_fwd, padded entries are never written; the last conv bias of every MLP receives its exact gradient, zero up to rounding, as
 * in the reference).  16-bit gradient planes carry a power-of-two loss scale: the one that brings max |d emb| into
 * [2^(grad_scale_log2 - 1), 2^grad_scale_log2), chosen on the device; the parameter gradients come back un-scaled.
 * As with the reference's AMP GradScaler, fp16 gradient planes can overflow for a given scale: the parameter
 * gradients are then non-finite and the caller skips the step and lowers grad_scale_log2 (training.py does; 9 is
 * the default, -24 .. 15 accepted; bf16 never overflows).  The workspace must be the one the forward call filled
 * (same G, N, parameters), fgnn_embed_train_workspace_bytes(...) bytes, 1024-byte aligned.  N <= 1024, and every
 * MLP has the same depth.
 * Two plans, picked from the shapes by all three calls alike:
 *   keep-all   the workspace keeps every activation of the batch from forward to backward (about 51 plane sets per
 *              graph at depth 3, 4 blocks: 107 GB for 64 graphs of N = 500, C = 64).  Used while that size is <= T.
 *   recompute  the workspace keeps the 16-bit input planes of the batch plus the activations of one pass of graphs;
 *              the forward runs pass by pass and keeps only emb, the backward re-runs each pass's forward before its
 *              backward (about one more forward per step; the loss scale is still chosen once over all of d emb).
 *              Passes are equal and as large as fit FGNN_TC_WS_GB (default 16) GiB, never less than one graph
 *              (FGNN_TC_CHUNK graphs when set, as for fgnn_embed_fwd).
 * T is FGNN_TC_TRAIN_WS_GB GiB when set (0 always picks recompute); otherwise half the current device's memory, because
 * a siamese step holds two workspaces (x1 and x2) until backward; unlimited when no device can be queried.  The plan
 * must not change between fgnn_embed_fwd_train and fgnn_embed_bwd: keep these variables and the current device as
 * they were for the workspace query. */
size_t fgnn_embed_train_workspace_bytes(const fgnn_embed_params* p, int32_t precision, int32_t G, int32_t N);
int fgnn_embed_fwd_train(const fgnn_embed_params* p, int32_t precision, const float* x, float* emb, int32_t G,
                         int32_t N, const int32_t* n_per_graph, void* workspace, size_t workspace_bytes,
                         void* stream);
int fgnn_embed_bwd(const fgnn_embed_params* p, const fgnn_embed_grads* grads, int32_t precision, const float* demb,
                   int32_t grad_scale_log2, int32_t G, int32_t N, const int32_t* n_per_graph, void* workspace,
                   size_t workspace_bytes, void* stream);

/* Fused multi-tensor Adam on one flat fp32 buffer: torch.optim.Adam(lr) of configure_optimizers
 * (models/trainers.py:92-104; betas, eps, weight_decay as given, no amsgrad) for all n entries in one launch.
 * p, g, m, v: parameters, gradients, first / second moments (n floats each, device); step >= 1 is the bias-correction
 * step.  grad_div (device scalar or NULL): gradients are divided by max(*grad_div, 1) -- the global row count of the
 * loss after the data-parallel all-reduce (toolbox/losses.py:32-34); skip_flag (device scalar or NULL): if
 * *skip_flag > 0 nothing is updated (a rank's 16-bit gradients overflowed: AMP's skipped step). */
int fgnn_adam_step_f32(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                       float eps, float weight_decay, int32_t step, const float* grad_div, const float* skip_flag,
                       void* stream);

/* Number of kernels the last call on this thread launched (bench.py's gpu_launches). */
int64_t fgnn_launch_count(void);
void fgnn_reset_launch_count(void);

/* Per-kernel-class device timing for bench.py's roofline: when enabled, every launch of the class
 * is bracketed by CUDA events on the launching stream.  kind: 0 = tensor-core conv-chain (MLP)
 * kernel, 1 = tensor-core N x N matmul kernel, 2 = plane statistics, 3 = other glue kernels.
 * fgnn_profile_read synchronises on the recorded events and returns their summed duration. */
void fgnn_profile_enable(int on);
void fgnn_profile_reset(void);
int fgnn_profile_read(int32_t kind, double* total_ms, int64_t* launches);

/* Diagnostics for the tensor-core building blocks (tests call these to check each kernel in
 * isolation against the fp32 operators): 16-bit planes are (G*C) planes of pitch_rows x pitch_cols. */
int fgnn_debug_tc_matmul(int32_t precision, const float* a, const float* b, float* out, int32_t G,
                         int32_t C, int32_t N, const int32_t* n_per_graph, void* workspace,
                         size_t workspace_bytes, void* stream);
size_t fgnn_debug_tc_matmul_workspace_bytes(int32_t G, int32_t C, int32_t N);
/* One MlpBlock_Real through the tensor-core conv-chain kernel (fold -> chain -> statistics ->
 * normalise): x (G,c_in,N,N) fp32 -> y (G,c_out,N,N) fp32, comparable with fgnn_mlp_fwd_f32. */
size_t fgnn_debug_tc_mlp_workspace_bytes(int32_t G, int32_t c_in, int32_t c_out, int32_t depth, int32_t N);
int fgnn_debug_tc_mlp(int32_t precision, const fgnn_mlp_params* p, const float* x, float* y, int32_t G,
                      int32_t N, const int32_t* n_per_graph, void* workspace, size_t workspace_bytes,
                      void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FGNN_B200_H */
