// Internal interface of the fp32 CUDA-core operators (fgnn_f32.cu).  These are the parity-mode
// kernels: plain FP32 FMA arithmetic with double-precision GraphNorm statistics.
#pragma once
#include "fgnn_common.cuh"

namespace fgnn {
namespace f32 {

// single 1x1 conv layer (shared by forward recomputation and backward-data in fgnn_f32_bwd.cu)
int run_conv1x1(const float* w, const float* b, int c_in, int c_out, bool transpose_w, bool relu, const float* x,
                float* y, float* wt_scratch, int G, int N, const int32_t* n_per_graph, cudaStream_t st);

// OrderedSum records of the fp32 MLP backward (deterministic mode): the GraphNorm affine-gradient terms of every
// (graph, channel) [2][G][c_out], and the weight / bias gradient of every pixel split [kMaxWgradSplits][c_out][cmax] /
// [kMaxWgradSplits][c_out]
constexpr int kMaxWgradSplits = 64;
struct MlpBwdRecords {
  float *gn, *w, *b;
};
inline MlpBwdRecords mlp_bwd_records(Arena& ar, int G, int c_out, int cmax) {
  MlpBwdRecords r;
  r.gn = ar.take<float>((size_t)2 * G * c_out);
  r.w = ar.take<float>((size_t)kMaxWgradSplits * c_out * cmax);
  r.b = ar.take<float>((size_t)kMaxWgradSplits * c_out);
  return r;
}

// workspace layout helper for one MLP call (det: room for the backward's OrderedSum records)
size_t mlp_workspace_bytes(int G, int c_in, int c_out, int depth, int N, bool det = false);

int mlp_fwd(const fgnn_mlp_params& p, const float* x, float* y, float* stats, int G, int N,
            const int32_t* n_per_graph, void* ws, size_t ws_bytes, cudaStream_t st);
int mlp_bwd(const fgnn_mlp_params& p, const fgnn_mlp_grads& g, const float* x, const float* stats,
            const float* dy, float* dx, int G, int N, const int32_t* n_per_graph, void* ws,
            size_t ws_bytes, cudaStream_t st, bool det = false);
int graphnorm_fwd(const float* x, float* y, float* stats, const float* gw, const float* gb, float eps,
                  int constant_n, int G, int C, int N, const int32_t* n_per_graph, cudaStream_t st);
int matmul_fwd(const float* a, const float* b, float* out, int G, int C, int N,
               const int32_t* n_per_graph, cudaStream_t st, bool trans_a = false, bool trans_b = false);
int colmax_fwd(const float* x, float* out, int32_t* argmax, int G, int C, int N,
               const int32_t* n_per_graph, cudaStream_t st);
int colmax_bwd(const float* dout, const int32_t* argmax, float* dx, int G, int C, int N,
               const int32_t* n_per_graph, cudaStream_t st);
// siamese head, graph 1 padded to N1 with sizes n1, graph 2 to N2 with sizes n2 (null: the padded size)
int scores_fwd(const float* e1, const float* e2, float* scores, int G, int C, int N1, int N2,
               const int32_t* n1, const int32_t* n2, cudaStream_t st);
int scores_bwd(const float* e1, const float* e2, const float* ds, float* de1, float* de2, int G, int C,
               int N1, int N2, const int32_t* n1, const int32_t* n2, cudaStream_t st);
int ce_argmax_fwd(const float* scores, float* ce_sum, int32_t* correct, float* row_lse, int32_t* row_argmax, int G,
                  int N1, int N2, const int32_t* n1, const int32_t* n2, void* ws, size_t ws_bytes, cudaStream_t st);
int ce_bwd(const float* scores, const float* row_lse, const float* coef, float* ds, int G, int N1, int N2,
           const int32_t* n1, const int32_t* n2, cudaStream_t st);
// out (G,Ca+Cb,N,N) = cat(a (G,Ca,N,N), b (G,Cb,N,N)) along channels  (models/layers.py:145-146)
int concat_channels(const float* a, const float* b, float* out, int G, int Ca, int Cb, int N,
                    cudaStream_t st);

// (G,N,N) uint8 adjacency -> (G,2,N,N) features W, diag(deg)  (loaders/data_generator.py:118-125)
int features_from_adjacency(const uint8_t* adj, float* out, int G, int N, const int32_t* n_per_graph, cudaStream_t st);

}  // namespace f32
}  // namespace fgnn
