// extern "C" surface of libfgnn_b200.so (declared in include/fgnn_b200.h).
#include "fgnn_common.cuh"
#include "fgnn_f32.cuh"
#include "fgnn_tc.cuh"

#include <mutex>
#include <utility>
#include <vector>

namespace fgnn {
thread_local char g_last_error[512] = "";
thread_local int64_t g_launches = 0;

namespace prof {
namespace {
struct Pool {
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev;
  size_t used = 0;
};
Pool g_pool[kNumKinds];
bool g_enabled = false;
std::mutex g_mu;
constexpr size_t kMaxEvents = 1 << 16;
}  // namespace
void begin(Kind k, cudaStream_t st) {
  if (!g_enabled) return;
  std::lock_guard<std::mutex> lk(g_mu);
  Pool& p = g_pool[k];
  if (p.used >= kMaxEvents) return;
  if (p.used == p.ev.size()) {
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    p.ev.emplace_back(a, b);
  }
  cudaEventRecord(p.ev[p.used].first, st);
}
void end(Kind k, cudaStream_t st) {
  if (!g_enabled) return;
  std::lock_guard<std::mutex> lk(g_mu);
  Pool& p = g_pool[k];
  if (p.used >= p.ev.size()) return;
  cudaEventRecord(p.ev[p.used].second, st);
  ++p.used;
}
}  // namespace prof

namespace {

// ---- fp32 fused embedder: composition of the per-operator kernels, chunked over graphs so the
// ---- scratch stays bounded (a (G,C,N,N) fp32 tensor is 8 GB at the headline config).
struct F32Plan {
  int chunk;        // graphs per pass
  int cmax, cinmax; // widest block output / widest concat input
  size_t act;       // floats per (chunk, cmax, N, N) tensor
};

F32Plan f32_plan(const fgnn_embed_params& p, int G, int N) {
  F32Plan pl{};
  pl.cmax = 0;
  pl.cinmax = 0;
  for (int b = 0; b < p.num_blocks; ++b) {
    pl.cmax = max(pl.cmax, p.block[b].mlp1.c_out);
    pl.cinmax = max(pl.cinmax, p.block[b].mlp3.c_in);
  }
  const size_t per_graph = (size_t)(5 * pl.cmax + pl.cinmax) * N * N * sizeof(float);
  const size_t budget = (size_t)3 << 30;
  long chunk = (long)(budget / (per_graph ? per_graph : 1));
  pl.chunk = (int)min((long)G, max(1L, chunk));
  pl.act = (size_t)pl.chunk * pl.cmax * N * N;
  return pl;
}

size_t f32_embed_ws(const fgnn_embed_params& p, int G, int N, F32Plan* out = nullptr) {
  F32Plan pl = f32_plan(p, G, N);
  if (out) *out = pl;
  Arena ar(nullptr, 0);
  for (int i = 0; i < 5; ++i) ar.take<float>(pl.act);                    // y1,y2,mult,ping,pong
  ar.take<float>((size_t)pl.chunk * pl.cinmax * N * N);                 // cat
  ar.take<float>((size_t)pl.chunk * pl.cmax * 2);                       // stats
  size_t mlpws = 0;
  for (int b = 0; b < p.num_blocks; ++b)
    mlpws = max(mlpws, f32::mlp_workspace_bytes(pl.chunk, p.block[b].mlp3.c_in, p.block[b].mlp3.c_out,
                                                p.block[b].mlp3.depth, N));
  ar.take<char>(mlpws);
  return align_up(ar.off, 1024);
}

int f32_embed_fwd(const fgnn_embed_params& p, const float* x, float* emb, int G, int N,
                  const int32_t* npg, void* ws, size_t ws_bytes, cudaStream_t st) {
  F32Plan pl;
  size_t need = f32_embed_ws(p, G, N, &pl);
  if (ws_bytes < need) return fail(FGNN_ERR_WORKSPACE, "embed workspace too small: %zu < %zu", ws_bytes, need);
  Arena ar(ws, ws_bytes);
  float* y1 = ar.take<float>(pl.act);
  float* y2 = ar.take<float>(pl.act);
  float* mult = ar.take<float>(pl.act);
  float* ping = ar.take<float>(pl.act);
  float* pong = ar.take<float>(pl.act);
  float* cat = ar.take<float>((size_t)pl.chunk * pl.cinmax * N * N);
  float* stats = ar.take<float>((size_t)pl.chunk * pl.cmax * 2);
  size_t mlpws_bytes = ws_bytes - align_up(ar.off, 256);
  char* mlpws = ar.take<char>(0);
  const long P = (long)N * N;
  const int c_in0 = p.block[0].mlp1.c_in;
  const int c_last = p.block[p.num_blocks - 1].mlp3.c_out;
  for (int g0 = 0; g0 < G; g0 += pl.chunk) {
    const int gc = min(pl.chunk, G - g0);
    const int32_t* n_c = npg ? npg + g0 : nullptr;
    const float* cur = x + (long)g0 * c_in0 * P;
    int cur_c = c_in0;
    float* nxt = ping;
    for (int b = 0; b < p.num_blocks; ++b) {
      const fgnn_block_params& bp = p.block[b];
      FGNN_CHECK_ARG(bp.mlp1.c_in == cur_c && bp.mlp2.c_in == cur_c, "block %d: c_in mismatch", b);
      FGNN_CHECK_ARG(bp.mlp3.c_in == cur_c + bp.mlp1.c_out && bp.mlp2.c_out == bp.mlp1.c_out,
                     "block %d: mlp3 must take c_in + c_out channels", b);
      if (int e = f32::mlp_fwd(bp.mlp1, cur, y1, stats, gc, N, n_c, mlpws, mlpws_bytes, st)) return e;
      if (int e = f32::mlp_fwd(bp.mlp2, cur, y2, stats, gc, N, n_c, mlpws, mlpws_bytes, st)) return e;
      if (int e = f32::matmul_fwd(y1, y2, mult, gc, bp.mlp1.c_out, N, n_c, st)) return e;
      if (int e = f32::concat_channels(mult, cur, cat, gc, bp.mlp1.c_out, cur_c, N, st)) return e;
      if (int e = f32::mlp_fwd(bp.mlp3, cat, nxt, stats, gc, N, n_c, mlpws, mlpws_bytes, st)) return e;
      cur = nxt;
      cur_c = bp.mlp3.c_out;
      nxt = (nxt == ping) ? pong : ping;
    }
    if (int e = f32::colmax_fwd(cur, emb + (long)g0 * c_last * N, nullptr, gc, c_last, N, n_c, st)) return e;
  }
  return FGNN_OK;
}

// `precision` argument of the embedder entry points: an fgnn_precision in the low byte, optionally | FGNN_DETERMINISTIC.
// false for any other bit.
bool split_precision(int32_t arg, int* precision, bool* det) {
  *precision = arg & 0xFF;
  *det = (arg & FGNN_DETERMINISTIC) != 0;
  return (arg & ~(0xFF | FGNN_DETERMINISTIC)) == 0;
}

int check_embed(const fgnn_embed_params* p, int G, int N) {
  FGNN_CHECK_ARG(p != nullptr, "null params");
  FGNN_CHECK_ARG(p->num_blocks >= 1 && p->num_blocks <= FGNN_MAX_BLOCKS, "num_blocks %d out of range", p->num_blocks);
  FGNN_CHECK_ARG(G >= 1 && N >= 1, "bad G=%d N=%d", G, N);
  return FGNN_OK;
}

}  // namespace
}  // namespace fgnn

using namespace fgnn;

extern "C" {

const char* fgnn_version(void) { return "fgnn_b200 0.1 (sm_100a)"; }
const char* fgnn_last_error(void) { return g_last_error; }
int64_t fgnn_launch_count(void) { return g_launches; }
void fgnn_reset_launch_count(void) { g_launches = 0; }

int fgnn_device_supports_tcgen05(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  int major = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
  return major == 10 ? 1 : 0;
}

size_t fgnn_mlp_workspace_bytes(int32_t G, int32_t c_in, int32_t c_out, int32_t depth, int32_t N) {
  return fgnn_mlp_workspace_bytes_ex(G, c_in, c_out, depth, N, 0);
}

size_t fgnn_mlp_workspace_bytes_ex(int32_t G, int32_t c_in, int32_t c_out, int32_t depth, int32_t N, int32_t flags) {
  if (flags & ~FGNN_DETERMINISTIC) return 0;
  return f32::mlp_workspace_bytes(G, c_in, c_out, depth, N, flags != 0);
}

int fgnn_mlp_fwd_f32(const fgnn_mlp_params* p, const float* x, float* y, float* stats, int32_t G,
                     int32_t N, const int32_t* n_per_graph, void* workspace, size_t workspace_bytes,
                     void* stream) {
  FGNN_CHECK_ARG(p != nullptr, "null params");
  return f32::mlp_fwd(*p, x, y, stats, G, N, n_per_graph, workspace, workspace_bytes, (cudaStream_t)stream);
}

int fgnn_mlp_bwd_f32(const fgnn_mlp_params* p, const fgnn_mlp_grads* g, const float* x,
                     const float* stats, const float* dy, float* dx, int32_t G, int32_t N,
                     const int32_t* n_per_graph, void* workspace, size_t workspace_bytes,
                     void* stream) {
  return fgnn_mlp_bwd_f32_ex(p, g, x, stats, dy, dx, G, N, n_per_graph, workspace, workspace_bytes, stream, 0);
}

int fgnn_mlp_bwd_f32_ex(const fgnn_mlp_params* p, const fgnn_mlp_grads* g, const float* x, const float* stats,
                        const float* dy, float* dx, int32_t G, int32_t N, const int32_t* n_per_graph, void* workspace,
                        size_t workspace_bytes, void* stream, int32_t flags) {
  FGNN_CHECK_ARG(p != nullptr && g != nullptr, "null params");
  FGNN_CHECK_ARG((flags & ~FGNN_DETERMINISTIC) == 0, "unknown flags 0x%x", (unsigned)flags);
  return f32::mlp_bwd(*p, *g, x, stats, dy, dx, G, N, n_per_graph, workspace, workspace_bytes, (cudaStream_t)stream,
                      flags != 0);
}

int fgnn_graphnorm_fwd_f32(const float* x, float* y, float* stats, const float* gn_w,
                           const float* gn_b, float eps, int32_t constant_n, int32_t G, int32_t C, int32_t N,
                           const int32_t* n_per_graph, void* stream) {
  return f32::graphnorm_fwd(x, y, stats, gn_w, gn_b, eps, constant_n, G, C, N, n_per_graph, (cudaStream_t)stream);
}

int fgnn_matmul_fwd_f32(const float* a, const float* b, float* out, int32_t G, int32_t C, int32_t N,
                        const int32_t* n_per_graph, void* stream) {
  return f32::matmul_fwd(a, b, out, G, C, N, n_per_graph, (cudaStream_t)stream);
}

int fgnn_matmul_bwd_f32(const float* a, const float* b, const float* dout, float* da, float* db,
                        int32_t G, int32_t C, int32_t N, const int32_t* n_per_graph, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (da)  // da = dout @ b^T
    if (int e = f32::matmul_fwd(dout, b, da, G, C, N, n_per_graph, st, false, true)) return e;
  if (db)  // db = a^T @ dout
    if (int e = f32::matmul_fwd(a, dout, db, G, C, N, n_per_graph, st, true, false)) return e;
  return FGNN_OK;
}

size_t fgnn_head_workspace_bytes(int32_t G, int32_t N) { return fgnn_head_pair_workspace_bytes(G, N); }
size_t fgnn_head_pair_workspace_bytes(int32_t G, int32_t N1) { return tc::head_workspace_bytes(G, N1); }

int fgnn_head_fwd(int32_t precision, const float* e1, const float* e2, float* scores, float* ce_sum, int32_t* correct,
                  int32_t G, int32_t C, int32_t N, const int32_t* n_per_graph, void* workspace, size_t workspace_bytes,
                  void* stream) {
  return fgnn_head_pair_fwd(precision, e1, e2, scores, ce_sum, correct, G, C, N, N, n_per_graph, n_per_graph, workspace,
                            workspace_bytes, stream);
}

int fgnn_head_pair_fwd(int32_t precision, const float* e1, const float* e2, float* scores, float* ce_sum, int32_t* correct,
                       int32_t G, int32_t C, int32_t N1, int32_t N2, const int32_t* n1, const int32_t* n2, void* workspace,
                       size_t workspace_bytes, void* stream) {
  return tc::head_fwd(precision & ~FGNN_DETERMINISTIC, e1, e2, scores, ce_sum, correct, G, C, N1, N2, n1, n2, workspace, workspace_bytes,
                      (cudaStream_t)stream);
}

int fgnn_head_fwd_train(int32_t precision, const float* e1, const float* e2, float* ce_sum, int32_t* correct, float* row_lse,
                        int32_t G, int32_t C, int32_t N, const int32_t* n_per_graph, void* workspace, size_t workspace_bytes,
                        void* stream) {
  return fgnn_head_pair_fwd_train(precision, e1, e2, ce_sum, correct, row_lse, G, C, N, N, n_per_graph, n_per_graph,
                                  workspace, workspace_bytes, stream);
}

int fgnn_head_pair_fwd_train(int32_t precision, const float* e1, const float* e2, float* ce_sum, int32_t* correct,
                             float* row_lse, int32_t G, int32_t C, int32_t N1, int32_t N2, const int32_t* n1,
                             const int32_t* n2, void* workspace, size_t workspace_bytes, void* stream) {
  return tc::head_fwd_train(precision & ~FGNN_DETERMINISTIC, e1, e2, ce_sum, correct, row_lse, G, C, N1, N2, n1, n2, workspace, workspace_bytes,
                            (cudaStream_t)stream);
}

int fgnn_head_bwd(int32_t precision, const float* e1, const float* e2, const float* row_lse, const float* coef, float* de1,
                  float* de2, int32_t G, int32_t C, int32_t N, const int32_t* n_per_graph, void* workspace,
                  size_t workspace_bytes, void* stream) {
  return fgnn_head_pair_bwd(precision, e1, e2, row_lse, coef, de1, de2, G, C, N, N, n_per_graph, n_per_graph, workspace,
                            workspace_bytes, stream);
}

int fgnn_head_pair_bwd(int32_t precision, const float* e1, const float* e2, const float* row_lse, const float* coef,
                       float* de1, float* de2, int32_t G, int32_t C, int32_t N1, int32_t N2, const int32_t* n1,
                       const int32_t* n2, void* workspace, size_t workspace_bytes, void* stream) {
  (void)workspace;
  (void)workspace_bytes;
  return tc::head_bwd(precision & ~FGNN_DETERMINISTIC, e1, e2, row_lse, coef, de1, de2, G, C, N1, N2, n1, n2, (cudaStream_t)stream);
}

int fgnn_lap_fwd(const float* scores, int32_t* col_of_row, int32_t* correct, double* total_cost, int32_t G,
                 int32_t N, const int32_t* n_per_graph, void* stream) {
  return fgnn_lap_pair_fwd(scores, col_of_row, correct, total_cost, G, N, N, n_per_graph, n_per_graph, stream);
}

int fgnn_lap_pair_fwd(const float* scores, int32_t* col_of_row, int32_t* correct, double* total_cost, int32_t G,
                      int32_t N1, int32_t N2, const int32_t* n1, const int32_t* n2, void* stream) {
  return lap::lap_fwd(scores, col_of_row, correct, total_cost, G, N1, N2, n1, n2, (cudaStream_t)stream);
}

int fgnn_features_from_adjacency_u8(const uint8_t* adj, float* out, int32_t G, int32_t N, const int32_t* n_per_graph,
                                    void* stream) {
  FGNN_CHECK_ARG(adj && out, "null pointer");
  FGNN_CHECK_ARG(G >= 0 && N > 0, "bad shape G=%d N=%d", G, N);
  return f32::features_from_adjacency(adj, out, G, N, n_per_graph, (cudaStream_t)stream);
}

int fgnn_colmax_fwd_f32(const float* x, float* out, int32_t* argmax, int32_t G, int32_t C, int32_t N,
                        const int32_t* n_per_graph, void* stream) {
  return f32::colmax_fwd(x, out, argmax, G, C, N, n_per_graph, (cudaStream_t)stream);
}

int fgnn_colmax_bwd_f32(const float* dout, const int32_t* argmax, float* dx, int32_t G, int32_t C,
                        int32_t N, const int32_t* n_per_graph, void* stream) {
  return f32::colmax_bwd(dout, argmax, dx, G, C, N, n_per_graph, (cudaStream_t)stream);
}

int fgnn_scores_fwd_f32(const float* e1, const float* e2, float* scores, int32_t G, int32_t C,
                        int32_t N, const int32_t* n_per_graph, void* stream) {
  return fgnn_scores_pair_fwd_f32(e1, e2, scores, G, C, N, N, n_per_graph, n_per_graph, stream);
}

int fgnn_scores_pair_fwd_f32(const float* e1, const float* e2, float* scores, int32_t G, int32_t C, int32_t N1,
                             int32_t N2, const int32_t* n1, const int32_t* n2, void* stream) {
  return f32::scores_fwd(e1, e2, scores, G, C, N1, N2, n1, n2, (cudaStream_t)stream);
}

int fgnn_scores_bwd_f32(const float* e1, const float* e2, const float* dscores, float* de1,
                        float* de2, int32_t G, int32_t C, int32_t N, const int32_t* n_per_graph,
                        void* stream) {
  return fgnn_scores_pair_bwd_f32(e1, e2, dscores, de1, de2, G, C, N, N, n_per_graph, n_per_graph, stream);
}

int fgnn_scores_pair_bwd_f32(const float* e1, const float* e2, const float* dscores, float* de1, float* de2, int32_t G,
                             int32_t C, int32_t N1, int32_t N2, const int32_t* n1, const int32_t* n2, void* stream) {
  return f32::scores_bwd(e1, e2, dscores, de1, de2, G, C, N1, N2, n1, n2, (cudaStream_t)stream);
}

size_t fgnn_ce_workspace_bytes(int32_t G, int32_t N) { return (size_t)G * N * 8 + 1024; }

int fgnn_ce_argmax_fwd_f32(const float* scores, float* ce_sum, int32_t* correct, float* row_lse,
                           int32_t G, int32_t N, const int32_t* n_per_graph, void* workspace,
                           size_t workspace_bytes, void* stream) {
  return fgnn_ce_pair_argmax_fwd_f32(scores, ce_sum, correct, row_lse, nullptr, G, N, N, n_per_graph, n_per_graph,
                                     workspace, workspace_bytes, stream);
}

int fgnn_ce_pair_argmax_fwd_f32(const float* scores, float* ce_sum, int32_t* correct, float* row_lse, int32_t* row_argmax,
                                int32_t G, int32_t N1, int32_t N2, const int32_t* n1, const int32_t* n2, void* workspace,
                                size_t workspace_bytes, void* stream) {
  return f32::ce_argmax_fwd(scores, ce_sum, correct, row_lse, row_argmax, G, N1, N2, n1, n2, workspace, workspace_bytes,
                            (cudaStream_t)stream);
}

int fgnn_ce_bwd_f32(const float* scores, const float* row_lse, const float* coef, float* dscores,
                    int32_t G, int32_t N, const int32_t* n_per_graph, void* stream) {
  return fgnn_ce_pair_bwd_f32(scores, row_lse, coef, dscores, G, N, N, n_per_graph, n_per_graph, stream);
}

int fgnn_ce_pair_bwd_f32(const float* scores, const float* row_lse, const float* coef, float* dscores, int32_t G,
                         int32_t N1, int32_t N2, const int32_t* n1, const int32_t* n2, void* stream) {
  return f32::ce_bwd(scores, row_lse, coef, dscores, G, N1, N2, n1, n2, (cudaStream_t)stream);
}

size_t fgnn_embed_workspace_bytes(const fgnn_embed_params* p, int32_t precision_flags, int32_t G, int32_t N) {
  int precision;
  bool det;
  if (!split_precision(precision_flags, &precision, &det)) return 0;
  if (!p || p->num_blocks < 1 || p->num_blocks > FGNN_MAX_BLOCKS || G < 1 || N < 1) return 0;
  if (precision == FGNN_FP32) return f32_embed_ws(*p, G, N);   // the fp32 forward has no cross-CTA sums
  return tc::embed_workspace_bytes(*p, G, N, det);
}

int fgnn_embed_fwd(const fgnn_embed_params* p, int32_t precision_flags, const float* x, float* emb,
                   int32_t G, int32_t N, const int32_t* n_per_graph, void* workspace, size_t workspace_bytes,
                   void* stream) {
  int precision;
  bool det;
  FGNN_CHECK_ARG(split_precision(precision_flags, &precision, &det), "unknown precision flags 0x%x", (unsigned)precision_flags);
  if (int e = check_embed(p, G, N)) return e;
  FGNN_CHECK_ARG(x && emb && workspace, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (precision == FGNN_FP32)
    return f32_embed_fwd(*p, x, emb, G, N, n_per_graph, workspace, workspace_bytes, st);
  if (precision == FGNN_BF16 || precision == FGNN_FP16)
    return tc::embed_fwd(*p, precision, det, x, emb, G, N, n_per_graph, workspace, workspace_bytes, st);
  return fail(FGNN_ERR_INVALID, "unknown precision %d", precision);
}

int fgnn_embed_fwd_adjacency_u8(const fgnn_embed_params* p, int32_t precision_flags, const uint8_t* adj, float* emb,
                                int32_t G, int32_t N, const int32_t* n_per_graph, void* workspace,
                                size_t workspace_bytes, void* stream) {
  int precision;
  bool det;
  FGNN_CHECK_ARG(split_precision(precision_flags, &precision, &det), "unknown precision flags 0x%x", (unsigned)precision_flags);
  if (int e = check_embed(p, G, N)) return e;
  FGNN_CHECK_ARG(adj && emb && workspace, "null pointer");
  return tc::embed_fwd_adjacency(*p, precision, det, adj, emb, G, N, n_per_graph, workspace, workspace_bytes,
                                 (cudaStream_t)stream);
}

size_t fgnn_embed_train_workspace_bytes(const fgnn_embed_params* p, int32_t precision_flags, int32_t G, int32_t N) {
  int precision;
  bool det;
  if (!split_precision(precision_flags, &precision, &det)) return 0;
  if (!p || p->num_blocks < 1 || p->num_blocks > FGNN_MAX_BLOCKS || G < 1 || N < 1) return 0;
  if (precision != FGNN_BF16 && precision != FGNN_FP16) return 0;
  return tc::embed_train_workspace_bytes(*p, G, N, det);
}

int fgnn_embed_fwd_train(const fgnn_embed_params* p, int32_t precision_flags, const float* x, float* emb, int32_t G,
                         int32_t N, const int32_t* n_per_graph, void* workspace, size_t workspace_bytes,
                         void* stream) {
  int precision;
  bool det;
  FGNN_CHECK_ARG(split_precision(precision_flags, &precision, &det), "unknown precision flags 0x%x", (unsigned)precision_flags);
  if (int e = check_embed(p, G, N)) return e;
  FGNN_CHECK_ARG(x && emb && workspace, "null pointer");
  return tc::embed_fwd_train(*p, precision, det, x, emb, G, N, n_per_graph, workspace, workspace_bytes, (cudaStream_t)stream);
}

int fgnn_embed_bwd(const fgnn_embed_params* p, const fgnn_embed_grads* grads, int32_t precision_flags, const float* demb,
                   int32_t grad_scale_log2, int32_t G, int32_t N, const int32_t* n_per_graph, void* workspace,
                   size_t workspace_bytes, void* stream) {
  int precision;
  bool det;
  FGNN_CHECK_ARG(split_precision(precision_flags, &precision, &det), "unknown precision flags 0x%x", (unsigned)precision_flags);
  if (int e = check_embed(p, G, N)) return e;
  FGNN_CHECK_ARG(grads && demb && workspace, "null pointer");
  FGNN_CHECK_ARG(grads->num_blocks == p->num_blocks, "grads describe %d blocks, params %d", grads->num_blocks, p->num_blocks);
  for (int b = 0; b < p->num_blocks; ++b) {
    const fgnn_mlp_params* mp[3] = {&p->block[b].mlp1, &p->block[b].mlp2, &p->block[b].mlp3};
    const fgnn_mlp_grads* mg[3] = {&grads->block[b].mlp1, &grads->block[b].mlp2, &grads->block[b].mlp3};
    for (int m = 0; m < 3; ++m)
      for (int l = 0; l < mp[m]->depth; ++l)
        FGNN_CHECK_ARG(mg[m]->w[l] != nullptr, "block %d mlp%d: missing weight-gradient buffer of layer %d", b, m + 1, l);
  }
  return tc::embed_bwd(*p, *grads, precision, det, demb, grad_scale_log2, G, N, n_per_graph, workspace, workspace_bytes,
                       (cudaStream_t)stream);
}

size_t fgnn_debug_tc_matmul_workspace_bytes(int32_t G, int32_t C, int32_t N) {
  return tc::debug_matmul_workspace_bytes(G, C, N);
}

int fgnn_debug_tc_matmul(int32_t precision, const float* a, const float* b, float* out, int32_t G,
                         int32_t C, int32_t N, const int32_t* n_per_graph, void* workspace,
                         size_t workspace_bytes, void* stream) {
  return tc::debug_matmul(precision, a, b, out, G, C, N, n_per_graph, workspace, workspace_bytes,
                          (cudaStream_t)stream);
}

size_t fgnn_debug_tc_mlp_workspace_bytes(int32_t G, int32_t c_in, int32_t c_out, int32_t depth, int32_t N) {
  return tc::debug_mlp_workspace_bytes(G, c_in, c_out, depth, N);
}

int fgnn_debug_tc_mlp(int32_t precision, const fgnn_mlp_params* p, const float* x, float* y, int32_t G,
                      int32_t N, const int32_t* n_per_graph, void* workspace, size_t workspace_bytes,
                      void* stream) {
  FGNN_CHECK_ARG(p != nullptr, "null params");
  return tc::debug_mlp(precision, *p, x, y, G, N, n_per_graph, workspace, workspace_bytes, (cudaStream_t)stream);
}

void fgnn_profile_enable(int on) {
  std::lock_guard<std::mutex> lk(prof::g_mu);
  prof::g_enabled = on != 0;
}

void fgnn_profile_reset(void) {
  std::lock_guard<std::mutex> lk(prof::g_mu);
  for (auto& p : prof::g_pool) p.used = 0;
}

int fgnn_profile_read(int32_t kind, double* total_ms, int64_t* launches) {
  FGNN_CHECK_ARG(kind >= 0 && kind < prof::kNumKinds && total_ms && launches, "bad kind %d", kind);
  std::lock_guard<std::mutex> lk(prof::g_mu);
  prof::Pool& p = prof::g_pool[kind];
  double ms = 0.0;
  for (size_t i = 0; i < p.used; ++i) {
    FGNN_CUDA(cudaEventSynchronize(p.ev[i].second));
    float t = 0.f;
    FGNN_CUDA(cudaEventElapsedTime(&t, p.ev[i].first, p.ev[i].second));
    ms += t;
  }
  *total_ms = ms;
  *launches = (int64_t)p.used;
  return FGNN_OK;
}

}  // extern "C"
