// fp32 CUDA-core operators: the parity mode of libfgnn_b200 (FGNN_FP32).
//
// Every kernel here restates one reference module on dense (G,C,N,N) fp32 tensors with an
// optional per-graph vertex count (MaskedTensor prefix masks).  Arithmetic is plain FP32 FMA;
// GraphNorm statistics are accumulated in double.  These kernels are not the roofline path --
// they exist so that (i) every reference module has a CUDA implementation behind the C ABI and
// (ii) the tensor-core path has an on-device fp32 twin to be checked against.
#include "fgnn_f32.cuh"

namespace fgnn {
namespace f32 {

namespace {

constexpr int kPixThreads = 128;  // pixels per CTA in the conv-chain kernels
constexpr int kMaxC = 128;        // widest hidden layer supported
constexpr int kMaxCin = 512;

__device__ __forceinline__ int graph_n(const int32_t* n_per_graph, int g, int N) {
  return n_per_graph ? n_per_graph[g] : N;
}

// ---------------------------------------------------------------------------------------
// weight repack: w (co, ci) row-major  ->  wt (ci, cop) with cop = round_up(co, 8), zero padded
// ---------------------------------------------------------------------------------------
__global__ void transpose_pad_kernel(const float* __restrict__ w, float* __restrict__ wt, int co,
                                     int ci, int cop) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= ci * cop) return;
  int i = idx / cop, o = idx % cop;
  wt[idx] = (o < co) ? w[o * ci + i] : 0.f;
}

// out[i][o] = w[i * ld + o] for o < co, 0 for the padding columns (row-padded copy of co columns of a row-major
// matrix with ld columns)
__global__ void pad_rows_kernel(const float* __restrict__ w, float* __restrict__ out, int rows, int co, int ld, int cop) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * cop) return;
  int i = idx / cop, o = idx % cop;
  out[idx] = (o < co) ? w[i * ld + o] : 0.f;
}

struct ChainArgs {
  int relu_last;                    // apply ReLU after the last layer too (used when layers run one at a time)
  int depth;
  int c_in;
  int c_out;
  int cop;                          // padded c_out (multiple of 8)
  int out_ch, out_off;              // z holds out_ch channels per graph; this chain writes [out_off, out_off + c_out)
  const float* wt[FGNN_MAX_DEPTH];  // (cin_k, cop)
  const float* b[FGNN_MAX_DEPTH];   // (c_out)
};

// ---------------------------------------------------------------------------------------
// conv chain: z = W_d(relu(... relu(W_1 x + b_1) ...)) + b_d, one pixel per thread.
// Hidden vectors live in shared memory as [channel][thread] columns (conflict free).
// layers.py:126-131 (without the GraphNorm, applied by normalize_apply_kernel).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kPixThreads)
conv_chain_fwd_kernel(ChainArgs a, const float* __restrict__ x, float* __restrict__ z, int N,
                      const int32_t* __restrict__ n_per_graph) {
  extern __shared__ float smem[];
  const int g = blockIdx.y;
  const int t = threadIdx.x;
  const long P = (long)N * N;
  const long p = (long)blockIdx.x * kPixThreads + t;
  const int n = graph_n(n_per_graph, g, N);
  const bool inb = p < P;
  const int i = inb ? (int)(p / N) : 0, j = inb ? (int)(p % N) : 0;
  const bool valid = inb && i < n && j < n;
  float* buf0 = smem;                       // [cop][kPixThreads]
  float* buf1 = smem + a.cop * kPixThreads;  // [cop][kPixThreads]
  const float* xg = x + (long)g * a.c_in * P;

  float* in = nullptr;
  float* out = buf0;
  for (int k = 0; k < a.depth; ++k) {
    const int cin = (k == 0) ? a.c_in : a.c_out;
    const float* __restrict__ wt = a.wt[k];
    const float* __restrict__ bk = a.b[k];
    const bool last = (k == a.depth - 1);
    for (int co0 = 0; co0 < a.cop; co0 += 8) {
      float acc[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) acc[u] = (bk != nullptr && co0 + u < a.c_out) ? __ldg(bk + co0 + u) : 0.f;
      for (int ci = 0; ci < cin; ++ci) {
        float v = (k == 0) ? (valid ? __ldg(xg + (long)ci * P + p) : 0.f) : in[ci * kPixThreads + t];
        const float4 w0 = __ldg(reinterpret_cast<const float4*>(wt + (long)ci * a.cop + co0));
        const float4 w1 = __ldg(reinterpret_cast<const float4*>(wt + (long)ci * a.cop + co0 + 4));
        acc[0] = fmaf(w0.x, v, acc[0]);
        acc[1] = fmaf(w0.y, v, acc[1]);
        acc[2] = fmaf(w0.z, v, acc[2]);
        acc[3] = fmaf(w0.w, v, acc[3]);
        acc[4] = fmaf(w1.x, v, acc[4]);
        acc[5] = fmaf(w1.y, v, acc[5]);
        acc[6] = fmaf(w1.z, v, acc[6]);
        acc[7] = fmaf(w1.w, v, acc[7]);
      }
      if (!last) {
#pragma unroll
        for (int u = 0; u < 8; ++u) out[(co0 + u) * kPixThreads + t] = fmaxf(acc[u], 0.f);
      } else if (inb) {
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (co0 + u < a.c_out)
            z[((long)g * a.out_ch + a.out_off + co0 + u) * P + p] = valid ? (a.relu_last ? fmaxf(acc[u], 0.f) : acc[u]) : 0.f;
      }
    }
    in = out;
    out = (out == buf0) ? buf1 : buf0;
  }
}

// ---------------------------------------------------------------------------------------
// per-(g,c) plane statistics in double over the valid n x n corner:
// stats[g,c] = {mean, 1/(2*sqrt(n*(var+eps)))}   (layers.py:71-80, maskedtensor.py:319-335)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
plane_stats_kernel(const float* __restrict__ z, float* __restrict__ stats, int C, int N,
                   const int32_t* __restrict__ n_per_graph, float eps, int constant_n) {
  const int gc = blockIdx.x;
  const int g = gc / C;
  const int n = graph_n(n_per_graph, g, N);
  const float* zp = z + (long)gc * N * N;
  double s = 0.0, ss = 0.0;
  for (long q = threadIdx.x; q < (long)n * n; q += blockDim.x) {
    int i = (int)(q / n), j = (int)(q % n);
    double v = zp[(long)i * N + j];
    s += v;
    ss += v * v;
  }
  __shared__ double sh[2][256];
  sh[0][threadIdx.x] = s;
  sh[1][threadIdx.x] = ss;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      sh[0][threadIdx.x] += sh[0][threadIdx.x + o];
      sh[1][threadIdx.x] += sh[1][threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    double cnt = (double)n * n;
    double mean = sh[0][0] / cnt;
    double var = sh[1][0] / cnt - mean * mean;
    if (var < 0) var = 0;
    stats[2 * gc] = (float)mean;
    stats[2 * gc + 1] = (float)(1.0 / (2.0 * sqrt((double)(constant_n ? N : n) * (var + (double)eps))));
  }
}

// y = gw * (z - mean) * inv + gb on valid positions, 0 elsewhere (in place allowed).  blockIdx.y strides over the
// planes (grid.y is limited to 65535).
__global__ void normalize_apply_kernel(const float* __restrict__ z, float* __restrict__ y,
                                       const float* __restrict__ stats, const float* __restrict__ gw,
                                       const float* __restrict__ gb, int C, int N, long planes,
                                       const int32_t* __restrict__ n_per_graph) {
  const long P = (long)N * N;
  for (long gc = blockIdx.y; gc < planes; gc += gridDim.y) {
    const int g = (int)(gc / C), c = (int)(gc % C);
    const int n = graph_n(n_per_graph, g, N);
    const float mean = stats[2 * gc], inv = stats[2 * gc + 1];
    const float w = gw ? gw[c] : 1.f, b = gb ? gb[c] : 0.f;
    for (long p = (long)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += (long)gridDim.x * blockDim.x) {
      int i = (int)(p / N), j = (int)(p % N);
      float v = 0.f;
      if (i < n && j < n) v = w * ((z[gc * P + p] - mean) * inv) + b;
      y[gc * P + p] = v;
    }
  }
}

// ---------------------------------------------------------------------------------------
// batched matmul out[g,c] = op(a[g,c]) @ op(b[g,c]) over the valid corner (layers.py:161-162)
// 64x64 tile, 256 threads, 4x4 per thread.  blockIdx.z strides over the planes (grid.z is limited to 65535).
// ---------------------------------------------------------------------------------------
template <bool TA, bool TB>
__global__ void __launch_bounds__(256)
matmul_kernel(const float* __restrict__ A, const float* __restrict__ B, float* __restrict__ Cout, int Cch,
              int N, long planes, const int32_t* __restrict__ n_per_graph) {
  __shared__ float As[16][64 + 1];
  __shared__ float Bs[16][64 + 1];
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  const int row0 = blockIdx.y * 64, col0 = blockIdx.x * 64;
  for (long gc = blockIdx.z; gc < planes; gc += gridDim.z) {
    const int g = (int)(gc / Cch);
    const int n = graph_n(n_per_graph, g, N);
    const float* a = A + gc * N * N;
    const float* b = B + gc * N * N;
    float* c = Cout + gc * N * N;
    float acc[4][4] = {};
    if (row0 < n && col0 < n) {
      for (int k0 = 0; k0 < n; k0 += 16) {
        for (int e = threadIdx.x; e < 16 * 64; e += 256) {
          int kk = e / 64, m = e % 64;
          int r = row0 + m, k = k0 + kk;
          float v = 0.f;
          if (r < n && k < n) v = TA ? a[(long)k * N + r] : a[(long)r * N + k];
          As[kk][m] = v;
          int cc = col0 + m;
          float w = 0.f;
          if (cc < n && k < n) w = TB ? b[(long)cc * N + k] : b[(long)k * N + cc];
          Bs[kk][m] = w;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
          float av[4], bv[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) av[u] = As[kk][ty * 4 + u];
#pragma unroll
          for (int u = 0; u < 4; ++u) bv[u] = Bs[kk][tx * 4 + u];
#pragma unroll
          for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int v = 0; v < 4; ++v) acc[u][v] = fmaf(av[u], bv[v], acc[u][v]);
        }
        __syncthreads();
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        int r = row0 + ty * 4 + u, cc = col0 + tx * 4 + v;
        if (r < N && cc < N) c[(long)r * N + cc] = (r < n && cc < n) ? acc[u][v] : 0.f;
      }
  }
}

// ---------------------------------------------------------------------------------------
// column max pooling: out[g,c,i] = max_{j<n} x[g,c,i,j]; padded rows -> 0
// (layers.py:194-203, maskedtensor.py:213-228).  One warp per row.
// ---------------------------------------------------------------------------------------
__global__ void colmax_fwd_kernel(const float* __restrict__ x, float* __restrict__ out,
                                  int32_t* __restrict__ argmax, int C, int N, long rows,
                                  const int32_t* __restrict__ n_per_graph) {
  const long row = (long)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  if (row >= rows) return;
  const int lane = threadIdx.x % 32;
  const int i = (int)(row % N);
  const int g = (int)(row / ((long)N * C));
  const int n = graph_n(n_per_graph, g, N);
  float best = -INFINITY;
  int bi = 0;
  if (i < n) {
    const float* xr = x + row * N;
    for (int j = lane; j < n; j += 32) {
      float v = xr[j];
      if (v > best) { best = v; bi = j; }
    }
    for (int o = 16; o > 0; o >>= 1) {
      float ov = __shfl_xor_sync(0xffffffffu, best, o);
      int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
    }
  } else {
    best = 0.f;
  }
  if (lane == 0) {
    out[row] = best;
    if (argmax) argmax[row] = bi;
  }
}

__global__ void colmax_bwd_kernel(const float* __restrict__ dout, const int32_t* __restrict__ argmax,
                                  float* __restrict__ dx, int C, int N, long rows,
                                  const int32_t* __restrict__ n_per_graph) {
  const long row = (long)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  if (row >= rows) return;
  const int lane = threadIdx.x % 32;
  const int i = (int)(row % N);
  const int g = (int)(row / ((long)N * C));
  const int n = graph_n(n_per_graph, g, N);
  const int bi = argmax[row];
  const float go = (i < n) ? dout[row] : 0.f;
  float* dr = dx + row * N;
  for (int j = lane; j < N; j += 32) dr[j] = (i < n && j == bi) ? go : 0.f;
}

// ---------------------------------------------------------------------------------------
// siamese scores[g,i,j] = sum_c e1[g,c,i] * e2[g,c,j]   (trainers.py:67)
// graph 1 (rows i, e1 (G,C,N1)) has n1[g] vertices, graph 2 (columns j, e2 (G,C,N2)) n2[g]; scores (G,N1,N2)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
scores_fwd_kernel(const float* __restrict__ e1, const float* __restrict__ e2, float* __restrict__ s,
                  int C, int N1, int N2, const int32_t* __restrict__ n1p, const int32_t* __restrict__ n2p) {
  const int g = blockIdx.z;
  const int n1 = graph_n(n1p, g, N1), n2 = graph_n(n2p, g, N2);
  const int i = blockIdx.y * 16 + threadIdx.x / 16;
  const int j = blockIdx.x * 16 + threadIdx.x % 16;
  __shared__ float a[16][17], b[16][17];
  float acc = 0.f;
  for (int c0 = 0; c0 < C; c0 += 16) {
    int cc = c0 + threadIdx.x / 16;
    int ii = blockIdx.y * 16 + threadIdx.x % 16;
    int jj = blockIdx.x * 16 + threadIdx.x % 16;
    a[threadIdx.x / 16][threadIdx.x % 16] = (cc < C && ii < n1) ? e1[((long)g * C + cc) * N1 + ii] : 0.f;
    b[threadIdx.x / 16][threadIdx.x % 16] = (cc < C && jj < n2) ? e2[((long)g * C + cc) * N2 + jj] : 0.f;
    __syncthreads();
#pragma unroll
    for (int c = 0; c < 16; ++c) acc = fmaf(a[c][threadIdx.x / 16], b[c][threadIdx.x % 16], acc);
    __syncthreads();
  }
  if (i < N1 && j < N2) s[((long)g * N1 + i) * N2 + j] = (i < n1 && j < n2) ? acc : 0.f;
}

// de1[g,c,i] = sum_j ds[g,i,j] e2[g,c,j];  de2[g,c,j] = sum_i ds[g,i,j] e1[g,c,i]
__global__ void __launch_bounds__(128)
scores_bwd_kernel(const float* __restrict__ e1, const float* __restrict__ e2, const float* __restrict__ ds,
                  float* __restrict__ de1, float* __restrict__ de2, int C, int N1, int N2,
                  const int32_t* __restrict__ n1p, const int32_t* __restrict__ n2p) {
  const int g = blockIdx.z, c = blockIdx.y;
  const int n1 = graph_n(n1p, g, N1), n2 = graph_n(n2p, g, N2);
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;  // i for de1, j for de2
  if (idx >= N1 && idx >= N2) return;
  const float* dsg = ds + (long)g * N1 * N2;
  const float* e1r = e1 + ((long)g * C + c) * N1;
  const float* e2r = e2 + ((long)g * C + c) * N2;
  float a1 = 0.f, a2 = 0.f;
  if (idx < n1)
    for (int q = 0; q < n2; ++q) a1 = fmaf(dsg[(long)idx * N2 + q], e2r[q], a1);
  if (idx < n2)
    for (int q = 0; q < n1; ++q) a2 = fmaf(dsg[(long)q * N2 + idx], e1r[q], a2);
  if (de1 && idx < N1) de1[((long)g * C + c) * N1 + idx] = a1;
  if (de2 && idx < N2) de2[((long)g * C + c) * N2 + idx] = a2;
}

// ---------------------------------------------------------------------------------------
// row softmax cross-entropy vs the identity matching + row argmax, one CTA per graph.
// losses.py:27-34 / metrics.py:125-134 without the host loop.  Deterministic reduction.
// scores (G,N1,N2); row i's target is column i, so rows i >= n2[g] have none (CE 0, not correct).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
ce_argmax_rows_kernel(const float* __restrict__ s, float* __restrict__ row_ce, int32_t* __restrict__ row_ok,
                      float* __restrict__ row_lse, int32_t* __restrict__ row_argmax, int N1, int N2,
                      const int32_t* __restrict__ n1p, const int32_t* __restrict__ n2p) {
  // one warp per row: row_ce[g,i] = lse_i - s_ii, row_ok[g,i] = (argmax_j s_ij == i); padded rows -> 0
  const int g = blockIdx.y;
  const int n1 = graph_n(n1p, g, N1), n2 = graph_n(n2p, g, N2);
  const int lane = threadIdx.x % 32;
  const int i = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  if (i >= N1) return;
  float ce = 0.f, lse = 0.f;
  int ok = 0, am = -1;
  if (i < n1) {
    const float* r = s + ((long)g * N1 + i) * N2;
    float m = -INFINITY;
    am = 0;
    for (int j = lane; j < n2; j += 32) {
      float v = r[j];
      if (v > m) { m = v; am = j; }
    }
    for (int o = 16; o > 0; o >>= 1) {
      float ov = __shfl_xor_sync(0xffffffffu, m, o);
      int oi = __shfl_xor_sync(0xffffffffu, am, o);
      if (ov > m || (ov == m && oi < am)) { m = ov; am = oi; }
    }
    float se = 0.f;
    for (int j = lane; j < n2; j += 32) se += expf(r[j] - m);
    for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
    lse = m + logf(se);
    if (i < n2) {
      ce = lse - r[i];
      ok = (am == i);
    }
  }
  if (lane == 0) {
    row_ce[(long)g * N1 + i] = ce;
    row_ok[(long)g * N1 + i] = ok;
    if (row_lse) row_lse[(long)g * N1 + i] = lse;
    if (row_argmax) row_argmax[(long)g * N1 + i] = am;
  }
}

// deterministic per-graph reduction of the per-row results (fixed order, one CTA per graph)
__global__ void __launch_bounds__(256)
ce_argmax_reduce_kernel(const float* __restrict__ row_ce, const int32_t* __restrict__ row_ok,
                        float* __restrict__ ce_sum, int32_t* __restrict__ correct, int N) {
  const int g = blockIdx.x;
  float t = 0.f;
  int k = 0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    t += row_ce[(long)g * N + i];
    k += row_ok[(long)g * N + i];
  }
  __shared__ float st[256];
  __shared__ int sk[256];
  st[threadIdx.x] = t;
  sk[threadIdx.x] = k;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      st[threadIdx.x] += st[threadIdx.x + o];
      sk[threadIdx.x] += sk[threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    ce_sum[g] = st[0];
    if (correct) correct[g] = sk[0];
  }
}

// rows without a target (i >= n2) are not in the CE sum: their gradient is zero
__global__ void ce_bwd_kernel(const float* __restrict__ s, const float* __restrict__ row_lse,
                              const float* __restrict__ coef, float* __restrict__ ds, int N1, int N2,
                              const int32_t* __restrict__ n1p, const int32_t* __restrict__ n2p) {
  const int g = blockIdx.z;
  const int n1 = graph_n(n1p, g, N1), n2 = graph_n(n2p, g, N2);
  const int i = blockIdx.y;
  const float cf = coef[g];
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < N2; j += gridDim.x * blockDim.x) {
    float v = 0.f;
    if (i < n1 && i < n2 && j < n2) {
      float sm = expf(s[((long)g * N1 + i) * N2 + j] - row_lse[(long)g * N1 + i]);
      v = cf * (sm - (i == j ? 1.f : 0.f));
    }
    ds[((long)g * N1 + i) * N2 + j] = v;
  }
}

__global__ void concat_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out,
                              int Ca, int Cb, long P, long total) {
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long)gridDim.x * blockDim.x) {
    long p = idx % P;
    long gc = idx / P;
    int c = (int)(gc % (Ca + Cb));
    long g = gc / (Ca + Cb);
    out[idx] = (c < Ca) ? a[(g * Ca + c) * P + p] : b[(g * Cb + (c - Ca)) * P + p];
  }
}

int check_dims(int G, int C, int N) {
  if (G <= 0 || C <= 0 || N <= 0) return fail(FGNN_ERR_INVALID, "non-positive dimension G=%d C=%d N=%d", G, C, N);
  return FGNN_OK;
}

}  // namespace

// ---- pieces shared with fgnn_f32_bwd.cu ---------------------------------------------------------
int run_conv1x1(const float* w, const float* b, int c_in, int c_out, bool transpose_w, bool relu, const float* x,
                float* y, float* wt_scratch, int G, int N, const int32_t* n_per_graph, cudaStream_t st) {
  // y[g,co,p] = sum_ci W'[co,ci] x[g,ci,p] (+ b[co]) (optionally ReLU) on valid pixels, 0 elsewhere.
  // transpose_w: W' = w^T where w is stored (c_in, c_out) row-major, i.e. the backward-data conv.
  // The chain kernel keeps at most kMaxC output channels in shared memory, so a wider c_out (the backward-data conv of
  // an MLP whose input is wider than kMaxC) runs in slices of kMaxC output channels.  Each output channel's sum is
  // formed alone, in ascending ci, so the slicing does not change a single bit.
  // set on every call: the attribute is per device and the call is cheap (a process may drive several GPUs)
  FGNN_CUDA(cudaFuncSetAttribute(conv_chain_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 2 * kMaxC * kPixThreads * (int)sizeof(float)));
  const long P = (long)N * N;
  const dim3 grid((unsigned)((P + kPixThreads - 1) / kPixThreads), G);
  for (int s0 = 0; s0 < c_out; s0 += kMaxC) {
    ChainArgs a;
    a.relu_last = relu ? 1 : 0;
    a.depth = 1;
    a.c_in = c_in;
    a.c_out = std::min(kMaxC, c_out - s0);
    a.cop = (a.c_out + 7) / 8 * 8;
    a.out_ch = c_out;
    a.out_off = s0;
    const int total = c_in * a.cop;
    if (!transpose_w) {
      // rows [s0, s0 + a.c_out) of w (c_out, c_in)
      transpose_pad_kernel<<<ceil_div(total, 256), 256, 0, st>>>(w + (long)s0 * c_in, wt_scratch, a.c_out, c_in, a.cop);
    } else {
      // w is (c_in rows, c_out cols): its columns [s0, s0 + a.c_out) are already "wt" up to the row padding
      pad_rows_kernel<<<ceil_div(total, 256), 256, 0, st>>>(w + s0, wt_scratch, c_in, a.c_out, c_out, a.cop);
    }
    FGNN_LAUNCHED();
    a.wt[0] = wt_scratch;
    a.b[0] = b ? b + s0 : nullptr;
    const size_t smem = (size_t)2 * a.cop * kPixThreads * sizeof(float);
    conv_chain_fwd_kernel<<<grid, kPixThreads, smem, st>>>(a, x, y, N, n_per_graph);
    FGNN_LAUNCHED();
  }
  return FGNN_OK;
}

// ---------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------
size_t mlp_workspace_bytes(int G, int c_in, int c_out, int depth, int N, bool det) {
  Arena ar(nullptr, 0);
  const int cop = (c_out + 7) / 8 * 8;
  for (int k = 0; k < depth; ++k) ar.take<float>((size_t)(k == 0 ? c_in : c_out) * cop);
  // backward scratch: per-(g,c) reductions + (depth + 2) activation tensors for a chunk of graphs
  ar.take<float>((size_t)G * c_out * 2);
  const int cmax = c_out > c_in ? c_out : c_in;
  ar.take<float>((size_t)cmax * ((cmax + 7) / 8 * 8));
  const size_t per_graph = (size_t)(depth + 2) * cmax * N * N * sizeof(float) + 256 * (depth + 2);
  size_t graphs = ((size_t)1 << 30) / per_graph;
  if (graphs < 1) graphs = 1;
  if (graphs > (size_t)G) graphs = G;
  ar.take<char>(graphs * per_graph + 4096);
  if (det) mlp_bwd_records(ar, G, c_out, cmax);
  return align_up(ar.off, 256);
}

static int prepare_chain(const fgnn_mlp_params& p, ChainArgs& a, Arena& ar, cudaStream_t st) {
  FGNN_CHECK_ARG(p.depth >= 1 && p.depth <= FGNN_MAX_DEPTH, "depth %d out of range", p.depth);
  FGNN_CHECK_ARG(p.c_out >= 1 && p.c_out <= kMaxC, "c_out %d unsupported (max %d)", p.c_out, kMaxC);
  FGNN_CHECK_ARG(p.c_in >= 1 && p.c_in <= kMaxCin, "c_in %d unsupported (max %d)", p.c_in, kMaxCin);
  a.relu_last = 0;
  a.depth = p.depth;
  a.c_in = p.c_in;
  a.c_out = p.c_out;
  a.cop = (p.c_out + 7) / 8 * 8;
  a.out_ch = p.c_out;
  a.out_off = 0;
  for (int k = 0; k < p.depth; ++k) {
    FGNN_CHECK_ARG(p.w[k] && p.b[k], "null weight/bias for layer %d", k);
    const int cin = (k == 0) ? p.c_in : p.c_out;
    float* wt = ar.take<float>((size_t)cin * a.cop);
    if (!ar.ok()) return fail(FGNN_ERR_WORKSPACE, "mlp workspace too small");
    int total = cin * a.cop;
    transpose_pad_kernel<<<ceil_div(total, 256), 256, 0, st>>>(p.w[k], wt, p.c_out, cin, a.cop);
    FGNN_LAUNCHED();
    a.wt[k] = wt;
    a.b[k] = p.b[k];
  }
  return FGNN_OK;
}

int graphnorm_fwd(const float* x, float* y, float* stats, const float* gw, const float* gb, float eps,
                  int constant_n, int G, int C, int N, const int32_t* n_per_graph, cudaStream_t st) {
  if (int e = check_dims(G, C, N)) return e;
  FGNN_CHECK_ARG(x && y && stats, "null pointer");
  plane_stats_kernel<<<G * C, 256, 0, st>>>(x, stats, C, N, n_per_graph, eps, constant_n);
  FGNN_LAUNCHED();
  long P = (long)N * N;
  const long planes = (long)G * C;
  dim3 grid((unsigned)min((long)64, (P + 255) / 256), (unsigned)min(planes, 65535L));
  normalize_apply_kernel<<<grid, 256, 0, st>>>(x, y, stats, gw, gb, C, N, planes, n_per_graph);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

int mlp_fwd(const fgnn_mlp_params& p, const float* x, float* y, float* stats, int G, int N,
            const int32_t* n_per_graph, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (int e = check_dims(G, p.c_out, N)) return e;
  FGNN_CHECK_ARG(x && y && stats && ws, "null pointer");
  Arena ar(ws, ws_bytes);
  ChainArgs a;
  if (int e = prepare_chain(p, a, ar, st)) return e;
  const size_t smem = (size_t)2 * a.cop * kPixThreads * sizeof(float);
  // set on every call: the attribute is per device and the call is cheap (a process may drive several GPUs)
  {
    FGNN_CUDA(cudaFuncSetAttribute(conv_chain_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   2 * kMaxC * kPixThreads * (int)sizeof(float)));
  }
  long P = (long)N * N;
  dim3 grid((unsigned)((P + kPixThreads - 1) / kPixThreads), G);
  conv_chain_fwd_kernel<<<grid, kPixThreads, smem, st>>>(a, x, y, N, n_per_graph);
  FGNN_LAUNCHED();
  return graphnorm_fwd(y, y, stats, p.gn_w, p.gn_b, p.eps, p.constant_n, G, p.c_out, N, n_per_graph, st);
}

int matmul_fwd(const float* a, const float* b, float* out, int G, int C, int N,
               const int32_t* n_per_graph, cudaStream_t st, bool ta, bool tb) {
  if (int e = check_dims(G, C, N)) return e;
  FGNN_CHECK_ARG(a && b && out, "null pointer");
  const long planes = (long)G * C;
  dim3 grid(ceil_div(N, 64), ceil_div(N, 64), (unsigned)min(planes, 65535L));
  if (!ta && !tb) matmul_kernel<false, false><<<grid, 256, 0, st>>>(a, b, out, C, N, planes, n_per_graph);
  else if (ta && !tb) matmul_kernel<true, false><<<grid, 256, 0, st>>>(a, b, out, C, N, planes, n_per_graph);
  else if (!ta && tb) matmul_kernel<false, true><<<grid, 256, 0, st>>>(a, b, out, C, N, planes, n_per_graph);
  else matmul_kernel<true, true><<<grid, 256, 0, st>>>(a, b, out, C, N, planes, n_per_graph);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

int colmax_fwd(const float* x, float* out, int32_t* argmax, int G, int C, int N,
               const int32_t* n_per_graph, cudaStream_t st) {
  if (int e = check_dims(G, C, N)) return e;
  FGNN_CHECK_ARG(x && out, "null pointer");
  long rows = (long)G * C * N;
  colmax_fwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(x, out, argmax, C, N, rows, n_per_graph);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

int colmax_bwd(const float* dout, const int32_t* argmax, float* dx, int G, int C, int N,
               const int32_t* n_per_graph, cudaStream_t st) {
  if (int e = check_dims(G, C, N)) return e;
  FGNN_CHECK_ARG(dout && argmax && dx, "null pointer");
  long rows = (long)G * C * N;
  colmax_bwd_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(dout, argmax, dx, C, N, rows, n_per_graph);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

int scores_fwd(const float* e1, const float* e2, float* scores, int G, int C, int N1, int N2,
               const int32_t* n1, const int32_t* n2, cudaStream_t st) {
  if (int e = check_dims(G, C, N1)) return e;
  if (int e = check_dims(G, C, N2)) return e;
  FGNN_CHECK_ARG(e1 && e2 && scores, "null pointer");
  FGNN_CHECK_ARG(G <= 65535, "G=%d exceeds grid.z limit", G);
  dim3 grid(ceil_div(N2, 16), ceil_div(N1, 16), G);
  scores_fwd_kernel<<<grid, 256, 0, st>>>(e1, e2, scores, C, N1, N2, n1, n2);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

int scores_bwd(const float* e1, const float* e2, const float* ds, float* de1, float* de2, int G, int C,
               int N1, int N2, const int32_t* n1, const int32_t* n2, cudaStream_t st) {
  if (int e = check_dims(G, C, N1)) return e;
  if (int e = check_dims(G, C, N2)) return e;
  FGNN_CHECK_ARG(e1 && e2 && ds, "null pointer");
  FGNN_CHECK_ARG(G <= 65535 && C <= 65535, "G/C exceed grid limits");
  dim3 grid(ceil_div(std::max(N1, N2), 128), C, G);
  scores_bwd_kernel<<<grid, 128, 0, st>>>(e1, e2, ds, de1, de2, C, N1, N2, n1, n2);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

int ce_argmax_fwd(const float* scores, float* ce_sum, int32_t* correct, float* row_lse, int32_t* row_argmax, int G,
                  int N1, int N2, const int32_t* n1, const int32_t* n2, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (int e = check_dims(G, 1, N1)) return e;
  if (int e = check_dims(G, 1, N2)) return e;
  FGNN_CHECK_ARG(scores && ce_sum && ws, "null pointer");
  FGNN_CHECK_ARG(G <= 65535, "G=%d exceeds grid.y limit", G);
  Arena ar(ws, ws_bytes);
  float* row_ce = ar.take<float>((size_t)G * N1);
  int32_t* row_ok = ar.take<int32_t>((size_t)G * N1);
  if (!ar.ok()) return fail(FGNN_ERR_WORKSPACE, "ce workspace too small");
  ce_argmax_rows_kernel<<<dim3(ceil_div(N1, 8), G), 256, 0, st>>>(scores, row_ce, row_ok, row_lse, row_argmax, N1, N2, n1, n2);
  FGNN_LAUNCHED();
  ce_argmax_reduce_kernel<<<G, 256, 0, st>>>(row_ce, row_ok, ce_sum, correct, N1);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

int ce_bwd(const float* scores, const float* row_lse, const float* coef, float* ds, int G, int N1, int N2,
           const int32_t* n1, const int32_t* n2, cudaStream_t st) {
  if (int e = check_dims(G, 1, N1)) return e;
  if (int e = check_dims(G, 1, N2)) return e;
  FGNN_CHECK_ARG(scores && row_lse && coef && ds, "null pointer");
  FGNN_CHECK_ARG(G <= 65535 && N1 <= 65535, "G/N exceed grid limits");
  dim3 grid(ceil_div(N2, 256), N1, G);
  ce_bwd_kernel<<<grid, 256, 0, st>>>(scores, row_lse, coef, ds, N1, N2, n1, n2);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

// adjacency (uint8) -> (W, diag(deg)) features, one warp per row  (loaders/data_generator.py:118-125)
__global__ void __launch_bounds__(256)
features_from_adjacency_kernel(const uint8_t* __restrict__ adj, float* __restrict__ out, int N, long rows,
                               const int32_t* __restrict__ n_per_graph) {
  const long row = (long)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x % 32;
  if (row >= rows) return;
  const int g = (int)(row / N), i = (int)(row % N);
  const int n = n_per_graph ? n_per_graph[g] : N;
  const uint8_t* a = adj + ((long)g * N + i) * N;
  float* w = out + (((long)g * 2) * N + i) * N;
  float* d = out + (((long)g * 2 + 1) * N + i) * N;
  int deg = 0;
  for (int j = lane; j < N; j += 32) {
    const int v = (i < n && j < n) ? (a[j] != 0) : 0;
    deg += v;
    w[j] = (float)v;
    d[j] = 0.f;
  }
  for (int o = 16; o > 0; o >>= 1) deg += __shfl_xor_sync(0xffffffffu, deg, o);
  __syncwarp();
  if (lane == 0 && i < n) d[i] = (float)deg;
}

int features_from_adjacency(const uint8_t* adj, float* out, int G, int N, const int32_t* n_per_graph, cudaStream_t st) {
  const long rows = (long)G * N;
  if (rows == 0) return FGNN_OK;
  features_from_adjacency_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(adj, out, N, rows, n_per_graph);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

int concat_channels(const float* a, const float* b, float* out, int G, int Ca, int Cb, int N,
                    cudaStream_t st) {
  long P = (long)N * N;
  long total = (long)G * (Ca + Cb) * P;
  unsigned blocks = (unsigned)min((total + 255) / 256, (long)148 * 16);
  concat_kernel<<<blocks, 256, 0, st>>>(a, b, out, Ca, Cb, P, total);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

}  // namespace f32
}  // namespace fgnn
