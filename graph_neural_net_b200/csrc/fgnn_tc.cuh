// Internal interface of the tensor-core (tcgen05 / TMEM / TMA) path (fgnn_tc.cu).
#pragma once
#include "fgnn_common.cuh"

namespace fgnn {
namespace tc {

// det: deterministic mode (FGNN_DETERMINISTIC): OrderedSum kernels, and a workspace with room for their records
size_t embed_workspace_bytes(const fgnn_embed_params& p, int G, int N, bool det);
int embed_fwd(const fgnn_embed_params& p, int precision, bool det, const float* x, float* emb, int G, int N,
              const int32_t* n_per_graph, void* ws, size_t ws_bytes, cudaStream_t st);

int embed_fwd_adjacency(const fgnn_embed_params& p, int precision, bool det, const uint8_t* adj, float* emb, int G, int N,
                        const int32_t* n_per_graph, void* ws, size_t ws_bytes, cudaStream_t st);

// 16-bit training path (fgnn_tc_train.cuh): forward keeping what backward needs in `ws`, and the backward of the stack.
// ckpt: block-level checkpoints (FGNN_CHECKPOINT_BLOCKS), the plan that trains up to N = 4096
size_t embed_train_workspace_bytes(const fgnn_embed_params& p, int G, int N, bool det, bool ckpt);
int embed_fwd_train(const fgnn_embed_params& p, int precision, bool det, bool ckpt, const float* x, float* emb, int G, int N,
                    const int32_t* n_per_graph, void* ws, size_t ws_bytes, cudaStream_t st);
int embed_bwd(const fgnn_embed_params& p, const fgnn_embed_grads& g, int precision, bool det, bool ckpt, const float* demb,
              int grad_scale_log2, int G, int N, const int32_t* n_per_graph, void* ws, size_t ws_bytes, cudaStream_t st);

// fused head: scores (optional) + row-softmax CE + row argmax on tensor cores.  Graph 1 (rows) is padded to N1 with
// sizes n1, graph 2 (columns) to N2 with sizes n2 (null: every graph has the padded size); the workspace follows N1.
size_t head_workspace_bytes(int G, int N1);
int head_fwd(int precision, const float* e1, const float* e2, float* scores, float* ce_sum, int32_t* correct, int G, int C,
             int N1, int N2, const int32_t* n1, const int32_t* n2, void* ws, size_t ws_bytes, cudaStream_t st);
// training: the same forward keeping each row's log-sum-exp, and its backward (d E1, d E2 without the (G,N1,N2) scores)
int head_fwd_train(int precision, const float* e1, const float* e2, float* ce_sum, int32_t* correct, float* row_lse, int G,
                   int C, int N1, int N2, const int32_t* n1, const int32_t* n2, void* ws, size_t ws_bytes, cudaStream_t st);
int head_bwd(int precision, const float* e1, const float* e2, const float* row_lse, const float* coef, float* de1, float* de2,
             int G, int C, int N1, int N2, const int32_t* n1, const int32_t* n2, cudaStream_t st);

size_t debug_matmul_workspace_bytes(int G, int C, int N);
int debug_matmul(int precision, const float* a, const float* b, float* out, int G, int C, int N,
                 const int32_t* n_per_graph, void* ws, size_t ws_bytes, cudaStream_t st);

size_t debug_mlp_workspace_bytes(int G, int c_in, int c_out, int depth, int N);
int debug_mlp(int precision, const fgnn_mlp_params& mp, const float* x, float* y, int G, int N,
              const int32_t* n_per_graph, void* ws, size_t ws_bytes, cudaStream_t st);

}  // namespace tc

namespace lap {
int lap_fwd(const float* scores, int32_t* col_of_row, int32_t* correct, double* total_cost, int G, int N1, int N2,
            const int32_t* n1, const int32_t* n2, cudaStream_t st);
}  // namespace lap
}  // namespace fgnn
