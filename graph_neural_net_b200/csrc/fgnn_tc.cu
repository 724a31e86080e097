// Tensor-core path of libfgnn_b200 (FGNN_BF16 / FGNN_FP16): TMA-fed tcgen05 kernels with TMEM
// accumulators for the two GEMM families of a 2-FGNN block, plus the small CUDA-core kernels
// that glue them (weight folding, statistics finalisation, pooling).
//
// HBM layout (DESIGN.md "Data layout").  Every activation is a set of 16-bit planes holding the
// PRE-GraphNorm output of the MLP that produced it.  GraphNorm is never applied to a stored tensor:
// its per-(graph, channel) scale a and shift s
//     a = w / (2 sqrt(n (var + eps))),   s = beta - a * mean                (layers.py:68-80)
// are folded into the consumer: into the first 1x1-conv weights of the next MLP (W diag(a), b + W s),
// into the epilogue of the N x N matmul
//     (a1 Y1 + s1 J)(a2 Y2 + s2 J) = a1 a2 Y1 Y2 + a1 s2 r1 1^T + s1 a2 1 c2^T + s1 s2 n J,
// and into the final max-pool (max(a y + s) = a max(y) + s or a min(y) + s by the sign of a).
// The row sums r1 = Y1 1 and column sums c2 = 1^T Y2 come out of the matmul itself: the operand
// layouts carry a row / column of ones per MMA tile,
//   every plane has physical columns pj = j + j / (BN-1) with pitch NPC = BN * NT; physical columns
//   pj % BN == BN-1 are "holes" (ones in Y2, zero elsewhere), so a 128-pixel tile of the conv kernel is 128
//   consecutive physical columns in every layout and is written with one TMA store per 64-pixel half;
//   layout C (block inputs/outputs, mult): rows i < N;
//   layout A (Y1, the matmul's A operand): physical row i + i / 127, PRA = 128 * MT rows, rows == 127 mod 128
//            hold ones (zero at hole columns);
//   layout B (Y2, the matmul's B operand): physical row k + k / (BN-1) -- the matmul's K index is the PHYSICAL
//            column of Y1 / row of Y2; hole rows are zero, hole columns hold ones,
// so D[127, :] of every 128 x BN accumulator tile is c2 and D[:, BN-1] is r1, at no extra MMA cost.
#include "fgnn_tc.cuh"
#include "fgnn_ptx.cuh"

#include <algorithm>
#include <climits>
#include <type_traits>
#include <cstdlib>
#include <cstring>

namespace fgnn {
namespace tc {

using namespace ptx;

namespace {

// Largest padded graph size of the 16-bit inference path (embedder, fused head).  At N = 4096 a plane holds
// 4096 x 4352 = 17.8 M pixels and one graph 139 264 conv-chain tiles: per-graph pixel and tile indices fit in int,
// and make_plan checks the per-launch tile count (see there).  Training keeps a lower limit (kMaxTrainN) except
// on its checkpoint plan.
constexpr int kMaxN = 4096;
constexpr int kTileM = 128;  // pixels per MLP tile / physical rows per matmul tile
constexpr int kTM1 = 127;    // logical rows per matmul tile

// The three plane layouts (see the top of this file).  Their row counts, plane strides and logical -> physical row maps
// are Geo's rows(), stride() and phys_row(); nothing else works them out.
enum Layout { kLayoutC, kLayoutA, kLayoutB };

struct Geo {
  int N, BN, TN1, NT, NPC, MT, PRA, PRB, BNLOG;
  long PSC, PSA, PSB;
  __host__ __device__ int rows(Layout l) const { return l == kLayoutA ? PRA : (l == kLayoutB ? PRB : N); }
  __host__ __device__ long stride(Layout l) const { return l == kLayoutA ? PSA : (l == kLayoutB ? PSB : PSC); }
  __host__ __device__ int phys_row(int i, Layout l) const { return l == kLayoutA ? i + i / kTM1 : (l == kLayoutB ? i + i / TN1 : i); }
};

inline int round_up(int v, int a) { return (v + a - 1) / a * a; }

Geo make_geo(int N) {
  Geo g;
  g.N = N;
  g.BN = (N <= 63) ? 64 : (N <= 127 ? 128 : 256);
  g.TN1 = g.BN - 1;
  g.BNLOG = (g.BN == 64) ? 6 : (g.BN == 128 ? 7 : 8);
  g.NT = (N + g.TN1 - 1) / g.TN1;
  g.NPC = g.BN * g.NT;
  g.MT = (N + kTM1 - 1) / kTM1;
  g.PRA = 128 * g.MT;
  g.PSC = (long)N * g.NPC;
  g.PRB = (N - 1) + (N - 1) / g.TN1 + 1;   // exactly the physical rows that are written (or zeroed holes): reads beyond are OOB = 0
  g.PSA = (long)g.PRA * g.NPC;
  g.PSB = (long)g.PRB * g.NPC;
  return g;
}

__device__ __forceinline__ int graph_n(const int32_t* n_per_graph, int g, int N) {
  return n_per_graph ? n_per_graph[g] : N;
}
// order-preserving float <-> unsigned code (0 is below every float, so a zeroed buffer is "no value yet")
__device__ __forceinline__ unsigned int enc_ordered(float f) {
  const unsigned int u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float dec_ordered(unsigned int e) {
  return __uint_as_float((e & 0x80000000u) ? (e & 0x7fffffffu) : ~e);
}

// one past the last physical K index (column of Y1 / row of Y2) a graph with n vertices uses
__device__ __forceinline__ int phys_k_end(int n, int TN1) { return (n - 1) + (n - 1) / TN1 + 1; }
// logical rows of a plane that the conv kernels must cover so that K-loops of the matmul may over-read zeros
__device__ __forceinline__ int rows_cover(const int32_t* n_per_graph, int g, const Geo& geo) {
  if (!n_per_graph) return geo.N;
  int r = (phys_k_end(n_per_graph[g], geo.TN1) + 63) / 64 * 64;
  return r < geo.N ? r : geo.N;
}
// (32-bit tile arithmetic: a plane has at most kMaxN x NPC(kMaxN) = 4096 x 4352 physical pixels; the tile total of a
// launch is bounded by make_plan)
__device__ __forceinline__ int mlp_tiles(const int32_t* n_per_graph, int g, const Geo& geo) {
  return (rows_cover(n_per_graph, g, geo) * geo.NPC + kTileM - 1) / kTileM;
}

// =============================================================================================
// small CUDA-core kernels
// =============================================================================================

// fp32 (G,C,N,N) -> 16-bit planes in layout A or B (the operands of debug_matmul).  Padding, holes and the inserted
// rows are written as zero.
template <typename T>
__global__ void to_planes_kernel(const float* __restrict__ x, T* __restrict__ out, int C, Geo geo, Layout l,
                                 const int32_t* __restrict__ n_per_graph) {
  const int gc = blockIdx.y;
  const int g = gc / C;
  const int n = graph_n(n_per_graph, g, geo.N);
  const long PS = geo.stride(l);
  const int period = l == kLayoutA ? kTileM : geo.BN;   // physical rows per inserted row
  for (long p = (long)blockIdx.x * blockDim.x + threadIdx.x; p < PS; p += (long)gridDim.x * blockDim.x) {
    const int pi = (int)(p / geo.NPC), pj = (int)(p % geo.NPC);
    const bool hole = (pj % geo.BN) == geo.BN - 1 || (pi % period) == period - 1;
    const int i = pi - pi / period, j = pj - pj / geo.BN;
    float v = (!hole && i < n && j < n) ? x[((long)gc * geo.N + i) * geo.N + j] : 0.f;
    out[(long)gc * PS + p] = Elem<T>::from_float(v);
  }
}

// fp32 (G,C,N,N) -> 16-bit layout-C planes, row-wise: no per-element division (BN is a power of two), two pixels per 32-bit store
template <typename T>
__global__ void __launch_bounds__(256)
to_planes_c_kernel(const float* __restrict__ x, T* __restrict__ out, int C, Geo geo, const int32_t* __restrict__ n_per_graph) {
  const int gc = blockIdx.y;
  const int n = graph_n(n_per_graph, gc / C, geo.N);
  for (int i = blockIdx.x; i < geo.N; i += gridDim.x) {
    const float* src = x + ((long)gc * geo.N + i) * geo.N;
    uint32_t* dst = reinterpret_cast<uint32_t*>(out + (long)gc * geo.PSC + (long)i * geo.NPC);
    for (int pj = 2 * threadIdx.x; pj < geo.NPC; pj += 2 * blockDim.x) {
      float v[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int q = pj + e;
        const bool hole = (q & (geo.BN - 1)) == geo.BN - 1;
        const int j = q - (q >> geo.BNLOG);
        v[e] = (!hole && i < n && j < n) ? src[j] : 0.f;
      }
      dst[pj >> 1] = Elem<T>::pack(v[0], v[1]);
    }
  }
}

// uint8 adjacency (G,N,N) -> the two layout-C input planes of block 1: channel 0 = W, channel 1 = diag(W.sum(1))
// (loaders/data_generator.py:118-125 without materialising the fp32 (G,2,N,N) tensor).  One warp per plane row;
// values are 0/1 and integer degrees <= N - 1 < 4096.  The degree is counted exactly and rounded to 16 bits once, to
// nearest even, as the fp32 features are on the features-fed path: fp16 is exact up to 2048 and rounds larger degrees
// to even numbers, bf16 is exact up to 256; both paths produce the same planes.
template <typename T>
__global__ void __launch_bounds__(256)
adjacency_to_planes_kernel(const uint8_t* __restrict__ adj, T* __restrict__ out, Geo geo, long rows,
                           const int32_t* __restrict__ n_per_graph) {
  const long row = (long)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x % 32;
  if (row >= rows) return;
  const int g = (int)(row / geo.N), i = (int)(row % geo.N);
  const int n = graph_n(n_per_graph, g, geo.N);
  const uint8_t* a = adj + ((long)g * geo.N + i) * geo.N;
  T* w = out + ((long)g * 2) * geo.PSC + (long)i * geo.NPC;
  T* d = w + geo.PSC;
  int deg = 0;
  for (int pj = lane; pj < geo.NPC; pj += 32) {
    const bool hole = (pj & (geo.BN - 1)) == geo.BN - 1;
    const int j = pj - (pj >> geo.BNLOG);
    const int v = (!hole && i < n && j < n) ? (a[j] != 0) : 0;
    deg += v;
    w[pj] = Elem<T>::from_float((float)v);
    d[pj] = Elem<T>::from_float(0.f);
  }
  for (int o = 16; o > 0; o >>= 1) deg += __shfl_xor_sync(0xffffffffu, deg, o);
  __syncwarp();
  if (lane == 0 && i < n) d[i + i / geo.TN1] = Elem<T>::from_float((float)deg);
}

// zero the inserted rows, which the conv kernel never stores: rows 127 mod 128 of layout A (ones rows; the backward GEMM
// Y1^T dM runs its K index over them), rows BN-1 mod BN of layout B (hole rows, 0 in K sums).  idx < 33 x 4352 at N = 4096.
template <typename T>
__global__ void zero_inserted_rows_kernel(T* __restrict__ y, Geo geo, Layout l) {
  T* plane = y + (long)blockIdx.y * geo.stride(l);
  const int period = l == kLayoutA ? kTileM : geo.BN;
  const int nrows = geo.rows(l) / period;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < nrows * geo.NPC; idx += gridDim.x * blockDim.x) {
    const int h = idx / geo.NPC, col = idx % geo.NPC;
    plane[(long)(h * period + period - 1) * geo.NPC + col] = Elem<T>::from_float(0.f);
  }
}

// layout C planes -> fp32 (G,C,N,N), optionally y = a*v + s on valid positions (debug / tests)
template <typename T>
__global__ void from_planes_kernel(const T* __restrict__ in, float* __restrict__ out, const float* __restrict__ coef,
                                   int C, Geo geo, const int32_t* __restrict__ n_per_graph) {
  const int gc = blockIdx.y;
  const int g = gc / C;
  const int n = graph_n(n_per_graph, g, geo.N);
  const float a = coef ? coef[2 * gc] : 1.f, s = coef ? coef[2 * gc + 1] : 0.f;
  const long P = (long)geo.N * geo.N;
  for (long p = (long)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += (long)gridDim.x * blockDim.x) {
    int i = (int)(p / geo.N), j = (int)(p % geo.N);
    float v = 0.f;
    if (i < n && j < n) v = a * Elem<T>::to_float(in[(long)gc * geo.PSC + (long)i * geo.NPC + j + j / geo.TN1]) + s;
    out[(long)gc * P + p] = v;
  }
}

// fp32 hidden-layer weights (rows, cols) -> 16-bit [co][Kh] zero padded (rows <= co, Kh multiple of 64), for up to all
// hidden-layer matrices of one block in ONE launch (blockIdx.y = matrix)
struct ConvertBatch {
  const float* src[3 * (FGNN_MAX_DEPTH - 1)];
  long dst_off[3 * (FGNN_MAX_DEPTH - 1)];   // element offset of the matrix in `out`
  int rows, cols;                            // real shape of every source matrix
};
template <typename T>
__global__ void convert_weights_batch_kernel(ConvertBatch cb, T* __restrict__ out, int co, int Kh) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= co * Kh) return;
  const int o = idx / Kh, k = idx % Kh;
  out[cb.dst_off[blockIdx.y] + idx] = Elem<T>::from_float(o < cb.rows && k < cb.cols ? cb.src[blockIdx.y][o * cb.cols + k] : 0.f);
}

// up to 2 (FGNN_MAX_DEPTH - 2) fp32 vectors of `real` entries -> [blockIdx.y][C] zero padded (hidden-layer biases)
struct PadBatch {
  const float* src[2 * (FGNN_MAX_DEPTH - 2)];
};
__global__ void pad_vectors_kernel(PadBatch pb, float* __restrict__ out, int C, int real) {
  const int c = threadIdx.x;
  if (c < C) out[blockIdx.y * C + c] = c < real ? pb.src[blockIdx.y][c] : 0.f;
}

// Per-graph folded first-layer weights for up to two MLPs that share their input (mlp1/mlp2).
//   Wf[g][m][co][koff_s + ch] = W_m[co][col_s + ch] * a_s[g][ch]
//   bf[g][m][co]              = b_m[co] + sum_s sum_ch W_m[co][col_s + ch] * s_s[g][ch]
// W_m and b_m have their real shapes; the source planes and the outputs are stored with c_s >= cr_s and c_out >= co_real
// channels, and the padded rows and columns fold to zero (see make_plan).  Real column col_s + ch is stored column
// (s ? c_0 : 0) + ch, so the bias sums visit the real terms in the order a zero-padded copy of W_m would.
struct FoldArgs {
  const float* w[2];     // per MLP: (co_real, cr0 + cr1)
  const float* b[2];     // per MLP: (co_real)
  const float* coef[2];  // per source: [G][c_s][2] or null (identity)
  int c[2], cr[2], koff[2], nsrc, nmlp;
  int c_out, co_real, K1g;
};
template <typename T>
__global__ void __launch_bounds__(256)
fold_weights_kernel(FoldArgs a, T* __restrict__ wf, float* __restrict__ bf, T* __restrict__ bt) {
  const int g = blockIdx.x, m = blockIdx.y;
  const int cin = a.c[0] + (a.nsrc > 1 ? a.c[1] : 0);
  const int cin_real = a.cr[0] + (a.nsrc > 1 ? a.cr[1] : 0);
  __shared__ float s_a[512], s_s[512];          // per stored input column: scale and shift of its source channel
  __shared__ int s_col[512];                    // per stored input column: its column of W_m, or -1 (padding)
  for (int col = threadIdx.x; col < cin; col += blockDim.x) {
    const int s = (col < a.c[0]) ? 0 : 1;
    const int ch = col - (s ? a.c[0] : 0);
    s_a[col] = a.coef[s] ? a.coef[s][((long)g * a.c[s] + ch) * 2] : 1.f;
    s_s[col] = a.coef[s] ? a.coef[s][((long)g * a.c[s] + ch) * 2 + 1] : 0.f;
    s_col[col] = ch < a.cr[s] ? (s ? a.cr[0] : 0) + ch : -1;
  }
  __syncthreads();
  T* wg = wf + ((long)g * a.nmlp + m) * a.c_out * a.K1g;
  const float* w = a.w[m];
  // output channels are split over gridDim.z: the kernel is latency-bound, 19 us with G x nmlp CTAs
  const int co_per = (a.c_out + gridDim.z - 1) / gridDim.z;
  const int co_begin = blockIdx.z * co_per, co_end = min(a.c_out, co_begin + co_per);
  for (int idx = co_begin * a.K1g + threadIdx.x; idx < co_end * a.K1g; idx += blockDim.x) {
    const int co = idx / a.K1g, k = idx % a.K1g;
    float v = 0.f;
    int col = -1;
    if (k < a.koff[1] || a.nsrc == 1) { if (k < a.c[0]) col = k; }
    else if (k - a.koff[1] < a.c[1]) col = a.c[0] + (k - a.koff[1]);
    if (col >= 0 && co < a.co_real && s_col[col] >= 0) v = w[co * cin_real + s_col[col]] * s_a[col];
    wg[idx] = Elem<T>::from_float(v);
  }
  // folded bias: one warp per output channel
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  for (int co = co_begin + warp; co < co_end; co += blockDim.x / 32) {
    float acc = 0.f;
    if (co < a.co_real)
      for (int col = lane; col < cin; col += 32)
        acc = fmaf(s_col[col] >= 0 ? w[co * cin_real + s_col[col]] : 0.f, s_s[col], acc);
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
      const float bias = co < a.co_real ? a.b[m][co] + acc : 0.f;
      bf[((long)g * a.nmlp + m) * a.c_out + co] = bias;
      if (bt) {
        // the same bias as one K = 16 step of the first-layer MMA (conv-chain kernel): row n = m c_out + co of a
        // K-major, un-swizzled B tile [n / 8][2 core matrices][8 rows][8 k]; k = 0 / 1 hold the 16-bit (hi, lo) split
        const int nrow = m * a.c_out + co;
        T* row = bt + (long)g * a.nmlp * a.c_out * 16 + (long)(nrow >> 3) * 128 + (nrow & 7) * 8;
        const T hi = Elem<T>::from_float(bias);
        const T lo = Elem<T>::from_float(bias - Elem<T>::to_float(hi));
        row[0] = hi;
        row[1] = lo;
        for (int k = 2; k < 8; ++k) row[k] = Elem<T>::from_float(0.f);
        for (int k = 0; k < 8; ++k) row[64 + k] = Elem<T>::from_float(0.f);
      }
    }
  }
}

// emb[g][c][i] = max_j (a y[i][j] + s) from the row-wise max / min codes the conv chain left in rowenc (rows >= n -> 0);
// emb is (G, co_real, N): the padded channels c >= co_real are not written
__global__ void pool_finalize_kernel(const unsigned int* __restrict__ rowenc, const float* __restrict__ coef,
                                     float* __restrict__ emb, int C, int co_real, int N, long total,
                                     const int32_t* __restrict__ n_per_graph) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int i = (int)(idx % N);
  const long gc = idx / N;
  const int g = (int)(gc / C), c = (int)(gc % C);
  if (c >= co_real) return;
  const int n = graph_n(n_per_graph, g, N);
  float out = 0.f;
  if (i < n) {
    const float a = coef[2 * gc], sft = coef[2 * gc + 1];
    const float mx = dec_ordered(rowenc[2 * idx]), mn = -dec_ordered(rowenc[2 * idx + 1]);
    out = fmaf(a, a >= 0.f ? mx : mn, sft);
  }
  emb[((long)g * co_real + c) * N + i] = out;
}

// (sum, sum of squares) accumulated by the conv-chain epilogue -> GraphNorm scale / shift.
//   acc[g][m][c][2] (double)  ->  coef_m[g][c] = {a, s}
// gw / gb have co_real[m] entries (null gw: weight 1, bias 0); the padded channels get a zero affine, so a = s = 0.
struct CoefArgs {
  const double* acc;
  float* coef[2];
  const float* gw[2];
  const float* gb[2];
  float eps[2];
  int constant_n[2];
  int co_real[2];
  int nmlp, C, N;
  const int32_t* n_per_graph;
  float* gnstat[2];   // training: [G][C][4] = {mean, 1 / (var + eps), 1 / (2 sqrt(n (var + eps))), 0} kept for backward (or null)
};
__global__ void finalize_coef_kernel(CoefArgs a, int total) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  int c = idx % a.C;
  int m = (idx / a.C) % a.nmlp;
  int g = idx / (a.C * a.nmlp);
  const int n = graph_n(a.n_per_graph, g, a.N);
  const double cnt = (double)n * n;
  const double S = a.acc[2 * (long)idx], SS = a.acc[2 * (long)idx + 1];
  const double mean = S / cnt;
  double var = SS / cnt - mean * mean;
  if (var < 0) var = 0;
  const bool real = c < a.co_real[m];
  const float gw = real ? (a.gw[m] ? a.gw[m][c] : 1.f) : 0.f, gb = real && a.gb[m] ? a.gb[m][c] : 0.f;
  const double sc = (double)gw / (2.0 * sqrt((double)(a.constant_n[m] ? a.N : n) * (var + (double)a.eps[m])));
  a.coef[m][((long)g * a.C + c) * 2] = (float)sc;
  a.coef[m][((long)g * a.C + c) * 2 + 1] = (float)((double)gb - sc * mean);
  if (a.gnstat[m]) {
    float* gs = a.gnstat[m] + ((long)g * a.C + c) * 4;
    gs[0] = (float)mean;
    gs[1] = (float)(1.0 / (var + (double)a.eps[m]));
    gs[2] = (float)(1.0 / (2.0 * sqrt((double)(a.constant_n[m] ? a.N : n) * (var + (double)a.eps[m]))));
    gs[3] = 0.f;
  }
}


// =============================================================================================
// K_A: fused conv chains on tensor cores: kSlots virtual tiles in flight, ONE epilogue group per TMEM slot.
//   tile  = 128 consecutive physical pixels (layout C) of one graph, all channels; NMLP (1 or 2) MLPs
//           consume the same staged input tile ("virtual tiles" v = tile * NMLP + m, slot = v % kSlots)
//   layer1: D[128 px, COUT] = X[px, K1] * W1f[g][m]^T   A = TMA-staged smem (MN-major), B = smem (K-major);
//           with NMLP = 2 the two MLPs' folded weights sit back to back in shared memory and their accumulators in
//           adjacent TMEM columns, so ONE N = 2 COUT MMA chain reads the staged tile once for both
//   layer>=2: D = relu(D) (16-bit, written back to TMEM) * W^T            A = TMEM, B = smem; the bias of every conv that
//           feeds a ReLU is already in the accumulator: one extra K = 16 MMA step, ones tile x (hi, lo) bias tile
//   output: raw last-layer accumulators as 16-bit planes (the last bias cancels in GraphNorm): staged in shared
//           memory with stmatrix.trans (16x256b accumulator fragments, four rounds of 16 registers), stored by TMA;
//           per-(graph, channel) sum and sum of squares are taken from the fp32 accumulators in the same pass (register
//           partials per thread in the fragment layout, folded across lanes and added with double atomics on a graph
//           change; Sum = OrderedSum stores them to records instead, see stat_records_reduce_kernel).  POOL = true (last block): the tile is not stored; the group reads its staged tile back
//           (thread = channel) for the statistics and the row-wise max / min of the fused column-max pooling.
// Warp roles: warps 0-15 = four epilogue groups (group = warp / 4 = TMEM slot, lane quadrant = warp % 4), warp 16 = TMA
// producer, warp 17 = first-layer MMA issuer (the only consumer of the input ring: it sees every phase of every
// barrier it waits on).  The hidden layers' MMAs are issued by the group itself: after its pass the four warps meet
// on a named barrier and one elected thread issues the next layer -- no hand-off to another warp sits on a slot's
// chain accumulator -> tcgen05.ld -> bias/ReLU/pack -> tcgen05.st -> MMA, and the four chains are independent.
// TMEM: accumulator of slot s in columns [s COUT, +COUT), its packed hidden activations and the ones columns of the
// hidden layers' bias step in [kSlots COUT + s (COUT/2 + 8), + COUT/2 + 8).
// =============================================================================================
template <typename T>
struct MlpArgs {
  int G;
  Geo geo;
  int k_src[2], nsrc, K1, K1g;
  int depth, Kh;
  const float* bias1;                        // [G][NMLP][COUT] folded layer-1 bias (fp32: RELU_OUT launches)
  const T* bias1_tile;                       // [G][NMLP COUT / 8][2][8][8] the same as a K = 16 MMA step (depth > 1 launches)
  const float* bias[2][FGNN_MAX_DEPTH];      // per MLP, layer l >= 1 biases
  T* out[2];                                 // per MLP output planes (direct stores of the ones row only)
  Layout out_mode[2];                        // output plane layout
  int ones[2];                               // kLayoutA: write the ones rows; kLayoutB: holes hold ones
  double* stat_acc;                          // [G][NMLP][COUT][2]; OrderedSum: the records of stat_records_reduce_kernel
  // Fused column-max pooling (last block): when rowenc[m] is set, MLP m's tile is NOT stored; the statistics pass
  // folds the row-wise max and min of its valid pixels into rowenc[m][g][c][i][2] (order-preserving unsigned codes
  // of max(y) and max(-y), buffer zeroed by the caller) and pool_finalize_kernel applies the GraphNorm affine.
  unsigned int* rowenc[2];
  const int32_t* n_per_graph;
};

constexpr int kSlots = 4;                    // TMEM slots = epilogue groups

// Deterministic conv-chain statistics (Sum = OrderedSum).  A CTA owns a contiguous range of the launch's flat
// (graph, tile) list, so each of its (TMEM slot, lane quadrant or pixel part) partial sums is flushed at most once per
// graph.  CTA b flushes graph g into record g + b: the CTAs that touch a graph form a contiguous run, and both ends of
// the run never decrease from one graph to the next, so (g, b) -> g + b is one-to-one on the pairs that occur and a
// launch of G graphs on `grid` CTAs fills at most G + grid records of [kSlots][4][COUT][2] doubles (zeroed beforehand:
// slots that saw no tile of the graph write nothing).
constexpr int kStatSubs = 4;   // lane quadrants (register statistics) or pixel parts (POOL, 128 / COUT <= 4) per slot
__host__ __device__ inline long stat_record_doubles(int COUT) { return (long)kSlots * kStatSubs * COUT * 2; }
__device__ __forceinline__ long stat_record(int g, int slot, int sub, int ch, int COUT) {
  return (long)(g + (int)blockIdx.x) * stat_record_doubles(COUT) + (((long)slot * kStatSubs + sub) * COUT + ch) * 2;
}
// CTAs of a tc_mlp_kernel launch: one per SM, at most one per tile (upper bound on the tiles of a ragged launch)
int mlp_grid(int G, const Geo& geo);

// acc[g][m][c][2] = the records of graph g summed in double over its CTAs, the slots of MLP m (slot % NMLP == m) and
// their sub-partials.  One block per (g, m, c): thread t adds records t, t + 256, ... of the graph's run in ascending
// order, then a fixed tree adds the 256 thread sums -- the same order on every run, spread over enough SMs that a
// launch of one large graph (148 CTAs x 16 records per channel) is not one SM's serial loop.
constexpr int kStatReduceThreads = 256;
__global__ void __launch_bounds__(kStatReduceThreads)
stat_records_reduce_kernel(const double* __restrict__ rec, double* __restrict__ acc, int G, int nmlp, int C, int grid,
                           Geo geo, const int32_t* __restrict__ n_per_graph) {
  __shared__ unsigned long long s_base, s_total;
  __shared__ int s_b0, s_b1;
  __shared__ double s_red[2][kStatReduceThreads];
  const int c = blockIdx.x % C, m = (blockIdx.x / C) % nmlp, g = blockIdx.x / (C * nmlp);
  if (threadIdx.x == 0) { s_base = 0; s_total = 0; s_b0 = INT_MAX; s_b1 = -1; }
  __syncthreads();
  unsigned long long base = 0, total = 0;        // tiles of graphs < g, of all graphs (integer sums: any order)
  for (int h = threadIdx.x; h < G; h += blockDim.x) {
    const unsigned long long t = mlp_tiles(n_per_graph, h, geo);
    total += t;
    if (h < g) base += t;
  }
  atomicAdd(&s_base, base);
  atomicAdd(&s_total, total);
  __syncthreads();
  // the run of CTAs whose tile range meets the graph's (the kernel's partition of the tiles); CTAs without tiles inside
  // the run flushed nothing and their records are zero
  const long t0 = (long)s_base, t1 = t0 + mlp_tiles(n_per_graph, g, geo), tot = (long)s_total;
  for (int b = threadIdx.x; b < grid; b += blockDim.x) {
    const long tb = tot * b / grid, te = tot * (b + 1) / grid;
    if (te > tb && tb < t1 && te > t0) { atomicMin(&s_b0, b); atomicMax(&s_b1, b); }
  }
  __syncthreads();
  const int spm = kSlots / nmlp, per_cta = spm * kStatSubs;
  const int nrec = s_b1 >= s_b0 ? (s_b1 - s_b0 + 1) * per_cta : 0;
  double v0 = 0.0, v1 = 0.0;
  for (int k = threadIdx.x; k < nrec; k += blockDim.x) {
    const int b = s_b0 + k / per_cta, slot = m + nmlp * ((k % per_cta) / kStatSubs), sub = k % kStatSubs;
    const double* r = rec + (long)(g + b) * stat_record_doubles(C) + (((long)slot * kStatSubs + sub) * C + c) * 2;
    v0 += r[0];
    v1 += r[1];
  }
  s_red[0][threadIdx.x] = v0;
  s_red[1][threadIdx.x] = v1;
  __syncthreads();
  for (int o = kStatReduceThreads / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      s_red[0][threadIdx.x] += s_red[0][threadIdx.x + o];
      s_red[1][threadIdx.x] += s_red[1][threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    double* a = acc + (((long)g * nmlp + m) * C + c) * 2;
    a[0] = s_red[0][0];
    a[1] = s_red[1][0];
  }
}

constexpr int kWProd = 4 * kSlots, kWL1 = kWProd + 1;
// 18 warps; registers are allocated in units of four warps, so the kernel gets 96 registers per thread (as 20 warps would).
// (setmaxnreg hand-over from the control warps to the epilogue groups was tried: ptxas 12.9 then allocates the WHOLE
// kernel at the smallest setmaxnreg value -- every role spilled.)
constexpr int kMlpThreads = (kWL1 + 1) * 32;

constexpr int kMaxInStages = 4;
__host__ __device__ inline int mlp_in_stages(int K1) { return K1 >= 128 ? 3 : 4; }   // 32 KB stages at K1 = 128

// fp32 biases staged in shared memory (RELU_OUT launches): one folded first-layer bias vector per TMEM slot
__host__ __device__ inline size_t mlp_bias_floats(int COUT, int NMLP, int depth) {
  return (size_t)kSlots * COUT;
}

// Biases through the tensor core (depth > 1): every conv whose output feeds a ReLU gets one extra K = 16 MMA step whose
// A operand is a constant tile of ones (k = 0, 1) and whose B operand holds the bias as a 16-bit (hi, lo) pair --
// the hidden pass is then a bare relu + pack.  Shared memory: the ones tile (4 KB), two buffers of the per-graph folded
// first-layer bias tile, one tile per hidden layer that has a ReLU behind it.
__host__ __device__ inline size_t mlp_bias_mma_bytes(int COUT, int NMLP, int depth) {
  return depth > 1 ? (size_t)4096 + (size_t)2 * NMLP * COUT * 32 + (size_t)NMLP * (depth - 2) * COUT * 32 : 0;
}

template <int COUT, int NMLP>
struct MlpSmem {
  static size_t bytes(int K1, int K1g, int depth, int Kh) {
    return 1024 + (size_t)mlp_in_stages(K1) * K1 * 256 + (size_t)2 * NMLP * K1g * COUT * 2 +
           (size_t)NMLP * (depth - 1) * Kh * COUT * 2 + (size_t)kSlots * COUT * 256 + mlp_bias_mma_bytes(COUT, NMLP, depth) +
           mlp_bias_floats(COUT, NMLP, depth) * 4 + 512;
  }
};

template <typename T, int COUT, int NMLP, bool POOL, bool RELU_OUT, typename Sum>
__global__ void __launch_bounds__(kMlpThreads, 1)
tc_mlp_kernel(const __grid_constant__ CUtensorMap map_x0, const __grid_constant__ CUtensorMap map_x1,
              const __grid_constant__ CUtensorMap map_w1, const __grid_constant__ CUtensorMap map_wh,
              const __grid_constant__ CUtensorMap map_o0, const __grid_constant__ CUtensorMap map_o1,
              const MlpArgs<T> args) {
  static_assert(kSlots % NMLP == 0, "a slot serves one MLP");
  constexpr uint32_t kAccCols = kSlots * COUT, kHidW = COUT / 2 + 8;   // packed activations + the ones columns of the bias step
  constexpr uint32_t kTmemCols = (kAccCols + kSlots * kHidW <= 256) ? 256 : 512;
  extern __shared__ uint8_t smem_raw[];
  // round the base up to 1024 bytes with POINTER arithmetic: an integer round trip makes the compiler treat everything
  // behind it as generic memory (LD.E / ST.E instead of LDS / STS)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int K1 = args.K1, K1g = args.K1g, depth = args.depth, Kh = args.Kh;
  const Geo geo = args.geo;
  const uint32_t stage_bytes = (uint32_t)K1 * 256u;
  const int kInStages = mlp_in_stages(K1);
  const uint32_t w1_mlp_bytes = (uint32_t)K1g * COUT * 2u;     // one MLP's folded first-layer weights
  const uint32_t w1_buf_bytes = w1_mlp_bytes * NMLP;           // one graph's
  const uint32_t wh_mat_bytes = (uint32_t)Kh * COUT * 2u;
  uint8_t* s_in = smem;
  uint8_t* s_w1 = s_in + (size_t)kInStages * stage_bytes;      // [2 buffers][NMLP][atoms][COUT][128B]
  uint8_t* s_wh = s_w1 + (size_t)2 * w1_buf_bytes;             // [NMLP][depth-1][atoms][COUT][128B]
  uint8_t* s_out = s_wh + (size_t)NMLP * (depth - 1) * wh_mat_bytes;   // [kSlots groups][2 halves][COUT][128 B] swizzled
  // Biases live in shared memory: with > 200 KB of it carved out the L1 holds next to nothing, and 16 global
  // loads per epilogue pass (uniform address, L2 latency) were costing more than the rest of the pass together.
  const bool bias_mma = depth > 1;                             // biases of the ReLU-ed layers ride on an extra MMA step
  const uint32_t b1x_bytes = (uint32_t)NMLP * COUT * 32u;      // one graph's folded first-layer bias tile
  uint8_t* s_ones = s_out + (size_t)kSlots * COUT * 256;       // [2 halves][16 k rows][128 B]: rows 0, 1 = ones (1024-byte aligned)
  uint8_t* s_b1x = s_ones + (bias_mma ? 4096 : 0);             // [2 buffers][NMLP COUT / 8][2][128 B] un-swizzled K-major
  uint8_t* s_bhx = s_b1x + (bias_mma ? 2 * b1x_bytes : 0);     // [NMLP][depth-2][COUT / 8][2][128 B]
  // fp32 biases in shared memory serve the RELU_OUT launches (depth 1, training forward) only
  float* s_bias1 = reinterpret_cast<float*>(s_out + (size_t)kSlots * COUT * 256 + mlp_bias_mma_bytes(COUT, NMLP, depth));   // [kSlots][COUT]
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(s_bias1) + mlp_bias_floats(COUT, NMLP, depth) * 4);
  uint64_t* in_full = bars;                      // [kInStages]
  uint64_t* in_empty = in_full + kMaxInStages;   // [kInStages]
  uint64_t* w1_full = in_empty + kMaxInStages;   // [2]
  uint64_t* w1_empty = w1_full + 2;           // [2]
  uint64_t* wh_full = w1_empty + 2;           // [1]
  uint64_t* mma_done = wh_full + 1;           // [kSlots] the slot's accumulator holds the next layer's result
  uint64_t* acc_free = mma_done + kSlots;     // [kSlots] the final pass has drained the slot's accumulator
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_free + kSlots);

  const int warp = uniform_warp_idx(), lane = threadIdx.x % 32;

  // ---- tile range of this CTA: contiguous chunk of the flat (graph, tile) list ----------------
  int total = 0;
  for (int g = 0; g < args.G; ++g) total += mlp_tiles(args.n_per_graph, g, geo);
  const int t_begin = (int)((long)total * blockIdx.x / gridDim.x);
  const int t_end = (int)((long)total * (blockIdx.x + 1) / gridDim.x);
  const int V = (t_end - t_begin) * NMLP;  // virtual tiles of this CTA

  if (threadIdx.x == 0) {
    for (int s = 0; s < kInStages; ++s) { mbar_init(&in_full[s], 1); mbar_init(&in_empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&w1_full[s], 1); mbar_init(&w1_empty[s], 1); }
    mbar_init(wh_full, 1);
    for (int s = 0; s < kSlots; ++s) { mbar_init(&mma_done[s], 1); mbar_init(&acc_free[s], 4); }
    fence_barrier_init();
  }
  if (bias_mma) {
    for (int i = threadIdx.x; i < 1024; i += blockDim.x)      // ones tile: k rows 0 and 1 of both 64-pixel halves
      reinterpret_cast<uint32_t*>(s_ones)[i] = (((i * 4) & 2047) < 256) ? Elem<T>::pack(1.f, 1.f) : 0u;
    for (int i = threadIdx.x; i < NMLP * (depth - 2) * COUT; i += blockDim.x) {
      const int c = i % COUT, ml = i / COUT;                  // ml = m (depth-2) + (layer - 1)
      const float b = args.bias[ml / (depth - 2)][1 + ml % (depth - 2)][c];
      const uint32_t hi = Elem<T>::bits(b);
      const uint16_t hi16 = (uint16_t)hi;
      const float hif = Elem<T>::to_float(*reinterpret_cast<const T*>(&hi16));
      const uint32_t lo = Elem<T>::bits(b - hif);
      uint4* row = reinterpret_cast<uint4*>(s_bhx + (size_t)ml * COUT * 32 + (size_t)(c >> 3) * 256 + (c & 7) * 16);
      row[0] = make_uint4(hi | (lo << 16), 0u, 0u, 0u);        // k = 0, 1 of core matrix 0
      row[8] = make_uint4(0u, 0u, 0u, 0u);                     // core matrix 1 (k = 8 .. 15), 128 bytes further
    }
    fence_proxy_async_smem();                                  // read by tcgen05.mma (async proxy)
  }
  if (warp == kWProd) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // graph walker shared by all roles: flat tile t -> (graph g, first pixel p0); t must not decrease
  struct Walker {
    int g = 0, n = 0;
    int base = 0, tiles = 0;
  };
  auto walker_init = [&](Walker& w) {
    w.g = 0;
    w.base = 0;
    w.n = graph_n(args.n_per_graph, 0, geo.N);
    w.tiles = mlp_tiles(args.n_per_graph, 0, geo);
  };
  auto walker_seek = [&](Walker& w, int t) {
    while (t >= w.base + w.tiles) {
      w.base += w.tiles;
      ++w.g;
      w.n = graph_n(args.n_per_graph, w.g, geo.N);
      w.tiles = mlp_tiles(args.n_per_graph, w.g, geo);
    }
  };

  if (warp == kWProd) {
    if (V > 0) {
      // ================= TMA producer (whole warp, elected lane issues) =================
      if (lane == 0) {
        prefetch_tensormap(&map_x0);
        prefetch_tensormap(&map_w1);
      }
      if (depth > 1) {
        const int atoms = Kh / 64;
        mbar_arrive_expect_tx_e(wh_full, (uint32_t)(NMLP * (depth - 1)) * wh_mat_bytes);
        for (int m = 0; m < NMLP; ++m)
          for (int l = 0; l < depth - 1; ++l)
            for (int at = 0; at < atoms; ++at)
              tma_load_3d_e(s_wh + ((size_t)(m * (depth - 1) + l) * atoms + at) * COUT * 128, &map_wh, wh_full, at * 64,
                          0, m * (depth - 1) + l);
      }
      Walker w;
      walker_init(w);
      int cur_g = -1, nchg = 0;
      uint32_t ph_w1e = 0, ph_ine = 0;   // phase bits (bit i = parity to wait for on barrier i): registers, not arrays
      for (int t = t_begin; t < t_end; ++t) {
        walker_seek(w, t);
        if (w.g != cur_g) {
          const int b = nchg & 1;
          if (nchg >= 2) { mbar_wait(&w1_empty[b], (ph_w1e >> b) & 1u); ph_w1e ^= 1u << b; }
          mbar_arrive_expect_tx_e(&w1_full[b], w1_buf_bytes + (bias_mma ? b1x_bytes : 0u));
          if (bias_mma)
            bulk_load_1d_e(s_b1x + (size_t)b * b1x_bytes, args.bias1_tile + (size_t)w.g * NMLP * COUT * 16, b1x_bytes, &w1_full[b]);
          for (int m = 0; m < NMLP; ++m)
            for (int at = 0; at < K1g / 64; ++at)
              tma_load_3d_e(s_w1 + (size_t)b * w1_buf_bytes + (size_t)m * w1_mlp_bytes + (size_t)at * COUT * 128,
                          &map_w1, &w1_full[b], at * 64, 0, w.g * NMLP + m);
          cur_g = w.g;
          ++nchg;
        }
        const int seq = t - t_begin;
        const int st = seq % kInStages;
        if (seq >= kInStages) { mbar_wait(&in_empty[st], (ph_ine >> st) & 1u); ph_ine ^= 1u << st; }
        const int p0 = (int)((t - w.base) * kTileM);
        uint8_t* dst = s_in + (size_t)st * stage_bytes;
        mbar_arrive_expect_tx_e(&in_full[st], stage_bytes);
        for (int u = 0; u < 2; ++u) {
          tma_load_3d_e(dst + (size_t)u * K1 * 128, &map_x0, &in_full[st], p0 + u * 64, 0, w.g);
          if (args.nsrc > 1)
            tma_load_3d_e(dst + (size_t)u * K1 * 128 + (size_t)args.k_src[0] * 128, &map_x1, &in_full[st], p0 + u * 64,
                        0, w.g);
        }
      }
    }
  } else if (warp == kWL1) {
    // ================= first-layer MMA issuer (whole warp, elected lane issues) =================
    // Consumes the input ring and the per-graph weight buffers in order; slot s of tile `seq` is (seq NMLP + m) % kSlots,
    // so the slots come round robin.  With NMLP = 2 one chain of N = 2 COUT MMAs fills both MLPs' accumulators.
    if (V > 0) {
      constexpr bool kMerge = (NMLP == 2);          // the two folded weight matrices are contiguous only with ONE K atom
      const bool merge = kMerge && K1g == 64;
      const uint32_t idesc1 = make_idesc(Elem<T>::kFmt, /*A MN-major*/ 1, /*B K-major*/ 0, kTileM, COUT);
      const uint32_t idesc1w = make_idesc(Elem<T>::kFmt, 1, 0, kTileM, 2 * COUT);
      const uint64_t a_d0 = smem_desc_sw128(smem_u32(s_in), (uint32_t)K1 * 128u, 1024u);   // MN-major activations
      const uint64_t b_d0 = smem_desc_sw128(smem_u32(s_w1), 16u, 1024u);                   // K-major weights
      const uint32_t a_desc_lo0 = (uint32_t)a_d0, a_desc_hi = (uint32_t)(a_d0 >> 32);
      const uint32_t w1_desc_lo0 = (uint32_t)b_d0, b_desc_hi = (uint32_t)(b_d0 >> 32);
      const uint64_t one_d = smem_desc_sw128(smem_u32(s_ones), 2048u, 1024u);              // ones tile, same format as a stage with K1 = 16
      const uint64_t b1x_d0 = smem_desc_nosw(smem_u32(s_b1x), 128u, 256u);
      const uint32_t one_lo = (uint32_t)one_d, one_hi = (uint32_t)(one_d >> 32);
      const uint32_t b1x_lo0 = (uint32_t)b1x_d0, b1x_hi = (uint32_t)(b1x_d0 >> 32);
      Walker wi;
      walker_init(wi);
      walker_seek(wi, t_begin);
      const int g_first = wi.g;
      int issue_gidx = 0;                      // graphs (relative to g_first) whose weight buffer has been released
      uint32_t ph_free = 0;                    // phase bits of acc_free[s]
      const int ntiles = t_end - t_begin;
      for (int seq = 0; seq < ntiles; ++seq) {
        const int st = (int)(seq % kInStages);
        walker_seek(wi, t_begin + seq);
        const int gidx = wi.g - g_first;
        for (; issue_gidx < gidx; ++issue_gidx) mma_commit_e(&w1_empty[issue_gidx & 1]);   // every MMA that read it was issued
        const int wbuf = gidx & 1;
        mbar_wait(&w1_full[wbuf], (uint32_t)(gidx >> 1) & 1u);
        mbar_wait(&in_full[st], (uint32_t)(seq / kInStages) & 1u);
        const int s0 = (int)((seq * NMLP) % kSlots);
#pragma unroll
        for (int m = 0; m < NMLP; ++m) {
          if (seq * NMLP + m >= kSlots) { mbar_wait(&acc_free[s0 + m], (ph_free >> (s0 + m)) & 1u); ph_free ^= 1u << (s0 + m); }
        }
        tc_fence_after();
        const uint32_t a_lo0 = a_desc_lo0 + (uint32_t)st * (stage_bytes >> 4);
        const uint32_t b_lo0 = w1_desc_lo0 + (((uint32_t)wbuf * w1_buf_bytes) >> 4);
        if (elect_one_sync()) {
          const int ksteps = K1 / 16;
          if (merge) {
            const uint32_t d_tmem = tmem_base + (uint32_t)(s0 * COUT);
            uint32_t a_lo = a_lo0, b_lo = b_lo0;
#pragma unroll 1
            for (int k = 0; k < ksteps; ++k) {
              mma_ss2(d_tmem, a_lo, a_desc_hi, b_lo, b_desc_hi, idesc1w, k > 0 ? 1u : 0u);
              a_lo += 2048u >> 4;                                       // next 16 K-rows of the MN-major tile
              b_lo += 32u >> 4;                                         // next 32 B of the single K atom
            }
            if (bias_mma) mma_ss2(d_tmem, one_lo, one_hi, b1x_lo0 + (((uint32_t)wbuf * b1x_bytes) >> 4), b1x_hi, idesc1w, 1u);
          } else {
#pragma unroll 1
            for (int m = 0; m < NMLP; ++m) {
              const uint32_t d_tmem = tmem_base + (uint32_t)((s0 + m) * COUT);
              uint32_t a_lo = a_lo0, b_lo = b_lo0 + (((uint32_t)m * w1_mlp_bytes) >> 4);
#pragma unroll 1
              for (int k = 0; k < ksteps; ++k) {
                mma_ss2(d_tmem, a_lo, a_desc_hi, b_lo, b_desc_hi, idesc1, k > 0 ? 1u : 0u);
                a_lo += 2048u >> 4;
                b_lo += ((k & 3) == 3) ? ((COUT * 128u - 96u) >> 4) : (32u >> 4);  // next K atom / next 32 B
              }
              if (bias_mma)
                mma_ss2(d_tmem, one_lo, one_hi, b1x_lo0 + (((uint32_t)wbuf * b1x_bytes + (uint32_t)m * COUT * 32u) >> 4), b1x_hi, idesc1, 1u);
            }
          }
          mma_commit(&in_empty[st]);
#pragma unroll
          for (int m = 0; m < NMLP; ++m) mma_commit(&mma_done[s0 + m]);
        }
        __syncwarp();
      }
      Walker wl = wi;                          // the producer may still wait for the release of later graphs
      walker_seek(wl, t_end - 1);
      for (; issue_gidx < wl.g - g_first + 1; ++issue_gidx) mma_commit_e(&w1_empty[issue_gidx & 1]);
    }
  } else {
    // ================= epilogue groups (warps 4s .. 4s+3 own TMEM slot s) =================
    const int s = warp >> 2;                 // group = slot
    const int quad = warp & 3;               // TMEM lane quadrant this warp may access
    const int et = threadIdx.x - s * 128;    // thread index inside the group = pixel of the tile
    const int m = s % NMLP;                  // the MLP this slot serves
    const int bar_id = 1 + s;
    const uint32_t acc_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(s * COUT);
    const uint32_t hid_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + kAccCols + (uint32_t)s * kHidW;
    uint8_t* tile = s_out + (size_t)s * (COUT * 256);      // [half][COUT rows][128 B], 16-byte chunks XOR-swizzled by (row & 7)
    const bool storer = !POOL && lane == 0 && (quad & 1) == 0;   // lane 0 of warps 0 / 2 of the group: its pixel starts a 64-pixel half
    const uint32_t idesc2 = make_idesc(Elem<T>::kFmt, 0, 0, kTileM, COUT);
    const uint32_t wh_desc_lo0 = (uint32_t)smem_desc_sw128(smem_u32(s_wh), 16u, 1024u);
    const uint32_t wh_desc_hi = (uint32_t)(smem_desc_sw128(smem_u32(s_wh), 16u, 1024u) >> 32);
    const uint64_t bhx_d0 = smem_desc_nosw(smem_u32(s_bhx), 128u, 256u);
    if (bias_mma) {
      // the ones columns of this slot's TMEM A operand (k = COUT, COUT + 1 of the hidden layers' bias step): written once
      uint32_t ones8[8] = {Elem<T>::pack(1.f, 1.f), 0u, 0u, 0u, 0u, 0u, 0u, 0u};
      tmem_st8(hid_addr + (uint32_t)(COUT / 2), ones8);
      tmem_wait_st();                          // ordered before the first hidden MMA by the pass's fence + named barrier
    }
    uint32_t ph_mma = 0;                     // parity of mma_done[s]
    bool wh_ready = false;
    Walker w;
    walker_init(w);
    int bias_g = -1;                         // graph whose folded first-layer bias sits in s_bias1[s]

    // ---- statistics state: thread -> (channel c, part): `part` selects a run of kPxPerPart consecutive pixels ----
    constexpr int kParts = 128 / COUT;             // 2 for COUT = 64, 4 for COUT = 32
    constexpr int kPxPerPart = 128 / kParts;       // 64 / 32 pixels = 8 / 4 16-byte chunks of one 64-pixel half
    const int c = et % COUT, part = et / COUT;
    const int half = (part * kPxPerPart) / 64, chunk0 = ((part * kPxPerPart) % 64) / 8;
    float acc_s = 0.f, acc_q = 0.f;
    int acc_g = -1;
    // register statistics (all but the pooled launches): sums of this thread's 16 (COUT = 64) channels over its pixels
    constexpr bool kRegStats = !POOL;
    float st_S[COUT / 4], st_Q[COUT / 4];
#pragma unroll
    for (int i = 0; i < COUT / 4; ++i) { st_S[i] = 0.f; st_Q[i] = 0.f; }
    auto flush_reg = [&]() {
      // the eight lanes with equal lane % 4 hold the same channels: fold them, then lanes 0-3 publish (warp-uniform call)
      if (acc_g < 0) return;
#pragma unroll
      for (int i = 0; i < COUT / 4; ++i) {
        float sv = st_S[i], qv = st_Q[i];
#pragma unroll
        for (int o = 4; o < 32; o <<= 1) {
          sv += __shfl_xor_sync(0xffffffffu, sv, o);
          qv += __shfl_xor_sync(0xffffffffu, qv, o);
        }
        if (lane < 4) {
          const int ch = 8 * (i >> 1) + 2 * lane + (i & 1);
          if constexpr (Sum::kOrdered) {
            double* dst = args.stat_acc + stat_record(acc_g, s, quad, ch, COUT);
            dst[0] = (double)sv;
            dst[1] = (double)qv;
          } else {
            double* dst = args.stat_acc + (((long)acc_g * NMLP + m) * COUT + ch) * 2;
            atomicAdd(dst, (double)sv);
            atomicAdd(dst + 1, (double)qv);
          }
        }
        st_S[i] = 0.f;
        st_Q[i] = 0.f;
      }
    };
    auto flush = [&]() {
      if (acc_g < 0) return;
      if constexpr (Sum::kOrdered) {
        double* dst = args.stat_acc + stat_record(acc_g, s, part, c, COUT);
        dst[0] = (double)acc_s;
        dst[1] = (double)acc_q;
      } else {
        double* dst = args.stat_acc + (((long)acc_g * NMLP + m) * COUT + c) * 2;
        atomicAdd(dst, (double)acc_s);
        atomicAdd(dst + 1, (double)acc_q);
      }
      acc_s = 0.f;
      acc_q = 0.f;
    };
    // fused pooling: running max / min of this thread's channel over the row it is currently in -> one pair of
    // atomics per (row, run of tiles this group sees in it)
    float pool_mx = -INFINITY, pool_mn = INFINITY;
    int pool_row = -1, pool_g = -1;
    auto pool_flush = [&]() {
      if (pool_row >= 0 && pool_mx >= pool_mn) {
        unsigned int* dst = args.rowenc[m] + ((((long)pool_g * COUT + c) * geo.N + pool_row) << 1);
        atomicMax(dst, enc_ordered(pool_mx));
        atomicMax(dst + 1, enc_ordered(-pool_mn));
      }
      pool_mx = -INFINITY;
      pool_mn = INFINITY;
    };

    int cur_g = -1, tp_i = 0, tp_j = 0;      // pixel (row, physical column) of the current tile's first pixel
    for (int v = s; v < V; v += kSlots) {
      const int seq = v / NMLP;
      walker_seek(w, t_begin + seq);
      const int g = w.g, n = w.n;
      // tile position without a division per tile: this group's tiles are kSlots / NMLP apart inside a graph
      const int p0 = (t_begin + seq - w.base) * kTileM;
      if (g != cur_g) {
        tp_i = p0 / geo.NPC;
        tp_j = p0 - tp_i * geo.NPC;
        cur_g = g;
      } else {
        tp_j += (kSlots / NMLP) * kTileM;
        while (tp_j >= geo.NPC) { tp_j -= geo.NPC; ++tp_i; }
      }
      if (RELU_OUT && g != bias_g) {
        // first tile of a new graph in this slot.  Every warp of the group has passed a named barrier since it last
        // read s_bias1 (the barrier that ends the pass), so the vector may be overwritten.
        if (et < COUT) s_bias1[s * COUT + et] = __ldg(args.bias1 + ((long)g * NMLP + m) * COUT + et);
        named_bar_sync(bar_id, 128);
        bias_g = g;
      }
#pragma unroll 1
      for (int l = 0; l < depth - 1; ++l) {
        // ---------------- hidden pass: accumulator -> relu(acc + b) as the next layer's 16-bit A operand in TMEM ----------------
        mbar_wait(&mma_done[s], ph_mma);
        ph_mma ^= 1u;
        tc_fence_after();
        {
          // the bias is already in the accumulator (extra MMA step), so the pass is relu + round + pack; 32 columns per
          // round (the epilogue warps also carry the statistics accumulators: registers)
#pragma unroll
          for (int c0 = 0; c0 < COUT; c0 += 16) {
            uint32_t r[16];
            tmem_ld16(acc_addr + (uint32_t)c0, r);
            tmem_wait_ld();
            uint32_t h[8];
#pragma unroll
            for (int u = 0; u < 8; ++u)
              h[u] = Elem<T>::pack_relu(__uint_as_float(r[2 * u]), __uint_as_float(r[2 * u + 1]));
            tmem_st8(hid_addr + (uint32_t)(c0 / 2), h);
          }
        }
        tmem_wait_st();
        tc_fence_before();
        // the staging buffer must be free before the final pass: the store of this group's previous tile has read it
        if (l == depth - 2 && storer) bulk_wait_group_read0();
        named_bar_sync(bar_id, 128);           // all four quadrants of the operand are written (and fenced)
        if (quad == 0) {
          // this group issues its own next layer: A = packed activations in TMEM, B = the layer's weights in smem
          if (!wh_ready) { mbar_wait(wh_full, 0); wh_ready = true; }
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)(s * COUT);
          const uint32_t a_tmem = tmem_base + kAccCols + (uint32_t)s * kHidW;
          const uint32_t wl_lo = wh_desc_lo0 + (uint32_t)(m * (depth - 1) + l) * (wh_mat_bytes >> 4);
          if (elect_one_sync()) {
#pragma unroll
            for (int k = 0; k < COUT / 16; ++k)
              mma_ts2(d_tmem, a_tmem + (uint32_t)k * 8u,
                      wl_lo + (((uint32_t)(k / 4) * (COUT * 128u) + (uint32_t)(k % 4) * 32u) >> 4), wh_desc_hi, idesc2,
                      k > 0 ? 1u : 0u);
            if (l + 1 <= depth - 2)              // this layer's output feeds a ReLU: its bias rides on one more K = 16 step
              mma_ts2(d_tmem, a_tmem + (uint32_t)(COUT / 2),
                      (uint32_t)bhx_d0 + (((uint32_t)(m * (depth - 2) + l) * COUT * 32u) >> 4), (uint32_t)(bhx_d0 >> 32), idesc2, 1u);
            mma_commit(&mma_done[s]);
          }
          __syncwarp();
        }
      }
      // ---------------- final pass: raw accumulator -> staged 16-bit tile -> TMA store + statistics ----------------
      if (depth == 1) {                        // (with hidden layers the last hidden pass's barrier covers this)
        if (storer) bulk_wait_group_read0();
        named_bar_sync(bar_id, 128);           // staging buffer free: its store and every thread's statistics pass are done
      }
      mbar_wait(&mma_done[s], ph_mma);
      ph_mma ^= 1u;
      tc_fence_after();
      // pixel coordinates: at most two row wraps from the tile's first pixel
      int pi = tp_i;
      int pj = tp_j + et;
      if (pj >= geo.NPC) { pj -= geo.NPC; ++pi; }
      if (pj >= geo.NPC) { pj -= geo.NPC; ++pi; }
      const bool in_plane = pi < geo.N;
      const bool hole = (pj & (geo.BN - 1)) == geo.BN - 1;
      const int j = pj - (pj >> geo.BNLOG);
      const bool valid = in_plane && !hole && pi < n && j < n;
      const Layout mode = args.out_mode[m];
      // holes of Y2 (layout B) hold ones on valid rows: they are the matmul's ones column
      const float marker = (hole && mode == kLayoutB && args.ones[m] && pi < n) ? 1.f : 0.f;
      {
        // Transposing store: the 16x256b TMEM load hands every thread channel PAIRS of four pixels (the mma
        // C-fragment layout), one packed convert per pair, and stmatrix.trans writes 8 channels x 8 pixels as
        // eight 16-byte row pieces.  Two rounds of 16 TMEM lanes each (registers): round hr covers the warp's pixels
        // 16 hr + lane / 4 (registers 4u, 4u+1) and 16 hr + 8 + lane / 4 (registers 4u+2, 4u+3), channels
        // 8u + 2 (lane % 4), +1.  The GraphNorm statistics are taken from the fp32 accumulators in the same pass:
        // every thread keeps the sum and the sum of squares of its 16 channels over its pixels in registers.
        const uint32_t vmask = __ballot_sync(0xffffffffu, valid);
        const uint32_t mmask = __ballot_sync(0xffffffffu, marker != 0.f);
        const int q4 = lane >> 2;
        const uint32_t one2 = Elem<T>::pack(1.f, 1.f);
        if constexpr (kRegStats) {
          if (g != acc_g) { flush_reg(); acc_g = g; }
        }
        // this thread supplies the address of row (lane % 8) of matrix (lane / 8) % 2: channel 8u + lane % 8,
        // pixels quad * 32 + 16 hr + 8 ((lane / 8) % 2) .. + 7 = 16-byte chunk (quad & 1) * 4 + 2 hr + (lane / 8) % 2
        const uint32_t st_base = smem_u32(tile) + (uint32_t)(quad >> 1) * (COUT * 128) + (uint32_t)(lane & 7) * 128;
        auto round = [&](auto all_valid_tag, int hr, int cq) {
          // 16 TMEM lanes x 32 columns per round: 16 registers in flight next to the 2 x COUT / 4 statistics accumulators
          constexpr bool kAllValid = decltype(all_valid_tag)::value;
          uint32_t r[16];
          tmem_ld_16x256b_x4(acc_addr + ((uint32_t)(16 * hr) << 16) + (uint32_t)(32 * cq), r);
          const uint32_t st_addr = st_base + (uint32_t)(((((quad & 1) << 2) + 2 * hr + ((lane >> 3) & 1)) ^ (lane & 7)) << 4) +
                                   (uint32_t)cq * 4096u;
          const bool va = (vmask >> (16 * hr + q4)) & 1u, vb = (vmask >> (16 * hr + 8 + q4)) & 1u;
          const uint32_t fa = ((mmask >> (16 * hr + q4)) & 1u) ? one2 : 0u, fb = ((mmask >> (16 * hr + 8 + q4)) & 1u) ? one2 : 0u;
          tmem_wait_ld();
          if (hr == 1 && cq == COUT / 32 - 1) {
            tc_fence_before();                 // accumulator drained: the slot may take its next tile
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_free[s]);
          }
          if constexpr (RELU_OUT) {
            // training forward, every conv layer is its own depth-1 launch: out = relu(acc + bias), bias of this
            // thread's channel pair 32 cq + 8u + 2 * (lane % 4), +1 from the slot's folded first-layer bias
            const float* bsl = s_bias1 + s * COUT + 32 * cq + 2 * (lane & 3);     // RELU_OUT launches have depth == 1
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float2 bb = *reinterpret_cast<const float2*>(bsl + 8 * u);
              r[4 * u] = __float_as_uint(__uint_as_float(r[4 * u]) + bb.x);
              r[4 * u + 1] = __float_as_uint(__uint_as_float(r[4 * u + 1]) + bb.y);
              r[4 * u + 2] = __float_as_uint(__uint_as_float(r[4 * u + 2]) + bb.x);
              r[4 * u + 3] = __float_as_uint(__uint_as_float(r[4 * u + 3]) + bb.y);
            }
          }
          if constexpr (kRegStats) {
            if constexpr (!kAllValid) {
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                if (!va) { r[4 * u] = 0u; r[4 * u + 1] = 0u; }
                if (!vb) { r[4 * u + 2] = 0u; r[4 * u + 3] = 0u; }
              }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int a = 8 * cq + 2 * u;
              sum_sq2(st_S[a], st_S[a + 1], st_Q[a], st_Q[a + 1], __uint_as_float(r[4 * u]), __uint_as_float(r[4 * u + 1]));
              sum_sq2(st_S[a], st_S[a + 1], st_Q[a], st_Q[a + 1], __uint_as_float(r[4 * u + 2]), __uint_as_float(r[4 * u + 3]));
            }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            uint32_t w0, w1;
            if constexpr (RELU_OUT) {
              w0 = Elem<T>::pack_relu(__uint_as_float(r[4 * u]), __uint_as_float(r[4 * u + 1]));
              w1 = Elem<T>::pack_relu(__uint_as_float(r[4 * u + 2]), __uint_as_float(r[4 * u + 3]));
            } else {
              w0 = Elem<T>::pack(__uint_as_float(r[4 * u]), __uint_as_float(r[4 * u + 1]));
              w1 = Elem<T>::pack(__uint_as_float(r[4 * u + 2]), __uint_as_float(r[4 * u + 3]));
            }
            if constexpr (!kAllValid) {
              w0 = va ? w0 : fa;
              w1 = vb ? w1 : fb;
            }
            stmatrix_x2_trans(st_addr + (uint32_t)u * 1024u, w0, w1);
          }
        };
        if (vmask == 0xffffffffu) {
#pragma unroll
          for (int hr = 0; hr < 2; ++hr)
#pragma unroll
            for (int cq = 0; cq < COUT / 32; ++cq) round(std::true_type{}, hr, cq);
        } else {
#pragma unroll
          for (int hr = 0; hr < 2; ++hr)
#pragma unroll
            for (int cq = 0; cq < COUT / 32; ++cq) round(std::false_type{}, hr, cq);
        }
      }
      fence_proxy_async_smem();            // generic-proxy smem writes -> visible to the TMA (async proxy)
      named_bar_sync(bar_id, 128);         // the tile is staged
      if (storer) {
        // store it: one 64-pixel half per TMA (a half never straddles a row because NPC % 64 == 0)
        const CUtensorMap* mo = (m == 0) ? &map_o0 : &map_o1;
        const int prow = geo.phys_row(pi, mode);
        if (pi < geo.N) tma_store_3d(mo, tile + (size_t)(quad >> 1) * (COUT * 128), pj, prow, g * COUT);
        bulk_commit_group();
      }
      // ones rows of Y1 (layout A): the last logical row of every 127-row matmul tile writes the row below it
      if (mode == kLayoutA && args.ones[m] && in_plane && pi < n) {
        const int mt = pi / kTM1;
        if (pi - mt * kTM1 == kTM1 - 1 || pi == n - 1) {
          const long ps = geo.stride(kLayoutA);
          T* o1 = args.out[m] + (long)g * COUT * ps + (long)(mt * 128 + 127) * geo.NPC + pj;
          const T ov = Elem<T>::from_float((!hole && j < n) ? 1.f : 0.f);
          for (int cc = 0; cc < COUT; ++cc) o1[(long)cc * ps] = ov;
        }
      }
      // ---------------- statistics of the staged tile: sum / sum of squares per channel (+ row max / min) ----------------
      if constexpr (!kRegStats) {
      if (g != acc_g) { flush(); acc_g = g; }
      {
        const uint8_t* row = tile + (size_t)half * (COUT * 128) + (size_t)c * 128;
        const uint32_t row_s = smem_u32(row);          // explicit shared-space loads
        float sv = 0.f, qv = 0.f;
        // fused pooling: position of this thread's run, and whether all of it lies inside the graph
        const int pstart = p0 + part * kPxPerPart;
        const int pool_pi = pstart / geo.NPC, pool_pj0 = pstart - pool_pi * geo.NPC;
        const bool pool_in = POOL && pool_pi < n && pool_pi < geo.N;
        const int pool_pj_end = phys_k_end(n, geo.TN1);
        const bool pool_full = pool_in && pool_pj0 + kPxPerPart <= pool_pj_end;      // warp-uniform (part is per warp)
        if (POOL && (pool_pi != pool_row || g != pool_g)) {
          pool_flush();
          pool_row = pool_in ? pool_pi : -1;
          pool_g = g;
        }
        if (!pool_full) {
          float sa = 0.f, sb = 0.f, qa = 0.f, qb = 0.f;    // even / odd pixels, packed fp32x2 arithmetic
#pragma unroll
          for (int k = 0; k < kPxPerPart / 8; ++k) {
            const uint4 wv = lds128u(row_s + (uint32_t)(((chunk0 + k) ^ (c & 7)) << 4));
            const uint32_t ww[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float2 f = Elem<T>::unpack2(ww[u]);
              sum_sq2(sa, sb, qa, qb, f.x, f.y);
            }
          }
          sv = sa + sb;
          qv = qa + qb;
        } else {
          // same pass with the row max / min folded in.  A hole column can only be the LAST pixel of a run (runs start
          // at multiples of kPxPerPart, BN is a multiple of 64): one guarded element, no per-pixel tests.
          const bool last_hole = ((pool_pj0 + kPxPerPart - 1) & (geo.BN - 1)) == geo.BN - 1;
          float sa = 0.f, sb = 0.f, qa = 0.f, qb = 0.f, mx = pool_mx, mn = pool_mn;
#pragma unroll
          for (int k = 0; k < kPxPerPart / 8; ++k) {
            const uint4 wv = lds128u(row_s + (uint32_t)(((chunk0 + k) ^ (c & 7)) << 4));
            const uint32_t ww[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float2 f = Elem<T>::unpack2(ww[u]);
              sum_sq2(sa, sb, qa, qb, f.x, f.y);
              mx = fmaxf(mx, f.x);
              mn = fminf(mn, f.x);
              if (k < kPxPerPart / 8 - 1 || u < 3 || !last_hole) { mx = fmaxf(mx, f.y); mn = fminf(mn, f.y); }
            }
          }
          sv = sa + sb;
          qv = qa + qb;
          pool_mx = mx;
          pool_mn = mn;
        }
        // hole pixels hold a marker (0 or 1), not data: take them out again
        for (int hp = (geo.BN - 1 - (p0 & (geo.BN - 1))) & (geo.BN - 1); hp < 128; hp += geo.BN) {
          if (hp >= part * kPxPerPart && hp < (part + 1) * kPxPerPart) {
            const uint8_t* hrow = tile + (size_t)(hp >> 6) * (COUT * 128) + (size_t)c * 128;
            const uint16_t raw = *reinterpret_cast<const uint16_t*>(hrow + ((((hp & 63) >> 3) ^ (c & 7)) << 4) + (hp & 7) * 2);
            const float x = Elem<T>::to_float(*reinterpret_cast<const T*>(&raw));
            sv -= x;
            qv -= x * x;
          }
        }
        acc_s += sv;
        acc_q += qv;
        if (pool_in && !pool_full) {
          // run that crosses the end of the graph's columns: per-pixel tests
          float mx = pool_mx, mn = pool_mn;
#pragma unroll 1
          for (int k = 0; k < kPxPerPart / 8; ++k) {
            const uint4 wv = lds128u(row_s + (uint32_t)(((chunk0 + k) ^ (c & 7)) << 4));
            const uint32_t ww[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float2 f = Elem<T>::unpack2(ww[u]);
              const int pjx = pool_pj0 + 8 * k + 2 * u;
              if (pjx < pool_pj_end && (pjx & (geo.BN - 1)) != geo.BN - 1) { mx = fmaxf(mx, f.x); mn = fminf(mn, f.x); }
              if (pjx + 1 < pool_pj_end && ((pjx + 1) & (geo.BN - 1)) != geo.BN - 1) { mx = fmaxf(mx, f.y); mn = fminf(mn, f.y); }
            }
          }
          pool_mx = mx;
          pool_mn = mn;
        }
      }
      }
    }
    if (POOL && pool_row >= 0) pool_flush();
    if (storer) bulk_wait_group0();   // every store has landed before the CTA exits
    if constexpr (kRegStats) flush_reg(); else flush();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == kWProd) {
    __syncwarp();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// =============================================================================================
// K_B: batched per-(graph, channel) N x N matmul with the GraphNorm rank-1 corrections in the
// epilogue.  out = a1 a2 (Y1 Y2) + a1 s2 r1 1^T + s1 a2 1 c2^T + s1 s2 n, r1 / c2 read from the
// accumulator tile itself (ones column of Y2 / ones row of Y1).
//   A = Y1 plane (layout A), K-major;  B = Y2 plane (layout C), MN-major;  out = layout C
//   tile 128 x BN (127 x BN-1 logical), K step 64, kStages-deep TMA ring, two TMEM accumulator stages.
// Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer, warps 2-5 = epilogue.
// =============================================================================================
template <typename T>
struct MatmulArgs {
  int G, C;
  Geo geo;
  T* out;                 // layout C
  const float* coef_a;    // [G*C][2] (a1, s1) or null
  const float* coef_b;    // [G*C][2] (a2, s2) or null
  const int32_t* n_per_graph;
};

template <int BN>
struct MatmulCfg {
  static constexpr int kStageBytes = 128 * 128 + BN * 128;  // A: 128 rows x 64 k, B: 64 k x BN
  static constexpr int kStages = (BN == 256) ? 4 : 6;
  static constexpr int kStoreBytes = 4 * 2 * 32 * 128;      // per epilogue warp: 2 buffers of 32 rows x 64 columns
  static constexpr size_t kSmemBytes =
      (size_t)kStages * kStageBytes + kStoreBytes + 2 * BN * sizeof(float) + (2 * kStages + 4) * 8 + 16;   // + barriers, TMEM slot
};

// Work items of the matmul: (plane, row tile, column tile), dealt to the CTAs round robin.
struct TileWalker {
  int g = 0;
  long base = 0;
  int mt = 0, nt = 0;
  long tiles_g = 0;
  __device__ void set(const int32_t* npg, int N, int C, int TN1) {
    int n = graph_n(npg, g, N);
    mt = (n + kTM1 - 1) / kTM1;
    nt = (n + TN1 - 1) / TN1;
    tiles_g = (long)mt * nt * C;
  }
  __device__ void init(const int32_t* npg, int N, int C, int TN1) {
    g = 0;
    base = 0;
    set(npg, N, C, TN1);
  }
  // -> plane q, row tile m, col tile nn for flat tile t (t must not decrease between calls)
  __device__ void locate(long t, const int32_t* npg, int N, int C, int TN1, int& q, int& m, int& nn, int& n) {
    while (t >= base + tiles_g) {
      base += tiles_g;
      ++g;
      set(npg, N, C, TN1);
    }
    long local = t - base;
    int per_plane = mt * nt;
    int c = (int)(local / per_plane);
    int rem = (int)(local % per_plane);
    q = g * C + c;
    m = rem / nt;
    nn = rem % nt;
    n = graph_n(npg, g, N);
  }
};

template <typename T, int BN>
__global__ void __launch_bounds__(192, 1)
tc_matmul_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                 const __grid_constant__ CUtensorMap map_o32, const __grid_constant__ CUtensorMap map_o31,
                 const MatmulArgs<T> args) {
  using Cfg = MatmulCfg<BN>;
  constexpr int kStages = Cfg::kStages;
  constexpr uint32_t kTmemCols = (2 * BN <= 128) ? 128 : (2 * BN <= 256 ? 256 : 512);
  // No static shared memory in this kernel, so the dynamic window starts 1024-byte aligned (checked: the swizzled TMA /
  // UMMA tiles need it, and at BN = 256 there is no room left for alignment slack).
  extern __shared__ uint8_t smem_mm[];
  uint8_t* smem = smem_mm;
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  uint8_t* s_store = smem + (size_t)kStages * Cfg::kStageBytes;                        // [4 warps][2][32 rows][128 B]
  float* s_cc = reinterpret_cast<float*>(s_store + Cfg::kStoreBytes);                  // [2][BN]
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_cc + 2 * BN);
  uint64_t* full = bars;
  uint64_t* empty = bars + kStages;
  uint64_t* tmem_full = bars + 2 * kStages;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;       // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  const int warp = uniform_warp_idx(), lane = threadIdx.x % 32;
  const Geo geo = args.geo;

  long total = 0;                              // work items: (plane, row tile, column tile)
  for (int g = 0; g < args.G; ++g) {
    int n = graph_n(args.n_per_graph, g, geo.N);
    total += (long)((n + kTM1 - 1) / kTM1) * ((n + geo.TN1 - 1) / geo.TN1) * args.C;
  }
  const long item0 = blockIdx.x, item_step = gridDim.x;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], 4); }
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    {
      // ================= TMA producer (whole warp, elected lane issues) =================
      if (lane == 0) {
        prefetch_tensormap(&map_a);
        prefetch_tensormap(&map_b);
      }
      TileWalker tw;
      tw.init(args.n_per_graph, geo.N, args.C, geo.TN1);
      int stage = 0;
      uint32_t phase = 0;
      for (long t = item0; t < total; t += item_step) {
        int q, m, nn, n;
        tw.locate(t, args.n_per_graph, geo.N, args.C, geo.TN1, q, m, nn, n);
        const int kts = (phys_k_end(n, geo.TN1) + 63) / 64;     // K runs over PHYSICAL columns of Y1 / rows of Y2
        for (int kt = 0; kt < kts; ++kt) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sa = smem + (size_t)stage * Cfg::kStageBytes;
          uint8_t* sb = sa + 128 * 128;
          mbar_arrive_expect_tx_e(&full[stage], (uint32_t)Cfg::kStageBytes);
          tma_load_3d_e(sa, &map_a, &full[stage], kt * 64, m * 128, q);     // rows beyond the plane are zero-filled
          for (int u = 0; u < BN / 64; ++u)
            tma_load_3d_e(sb + (size_t)u * 8192, &map_b, &full[stage], nn * BN + u * 64, kt * 64, q);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    {
      // ================= MMA issuer (whole warp, elected lane issues) =================
      const uint32_t idesc = make_idesc(Elem<T>::kFmt, /*A K-major*/ 0, /*B MN-major*/ 1, 128, BN);
      const uint64_t a_d0 = smem_desc_sw128(smem_u32(smem), 16u, 1024u);                 // K-major A tile
      const uint64_t b_d0 = smem_desc_sw128(smem_u32(smem) + 128 * 128, 8192u, 1024u);   // MN-major B tile
      const uint32_t a_desc_lo0 = (uint32_t)a_d0, a_desc_hi = (uint32_t)(a_d0 >> 32);
      const uint32_t b_desc_lo0 = (uint32_t)b_d0, b_desc_hi = (uint32_t)(b_d0 >> 32);
      TileWalker tw;
      tw.init(args.n_per_graph, geo.N, args.C, geo.TN1);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      for (long t = item0; t < total; t += item_step) {
        int q, m, nn, n;
        tw.locate(t, args.n_per_graph, geo.N, args.C, geo.TN1, q, m, nn, n);
        const int kts = (phys_k_end(n, geo.TN1) + 63) / 64;
        mbar_wait(&tmem_empty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
        for (int kt = 0; kt < kts; ++kt) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t a_lo = a_desc_lo0 + (uint32_t)stage * (Cfg::kStageBytes >> 4);
          const uint32_t b_lo = b_desc_lo0 + (uint32_t)stage * (Cfg::kStageBytes >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            mma_ss2_e(d_tmem, a_lo + (uint32_t)k * (32u >> 4), a_desc_hi, b_lo + (uint32_t)k * (2048u >> 4), b_desc_hi,
                      idesc, (kt > 0 || k > 0) ? 1u : 0u);
          mma_commit_e(&empty[stage]);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        mma_commit_e(&tmem_full[as]);
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    }
  } else {
    // ================= epilogue (warps 2..5, TMEM lane quadrant = warp % 4) =================
    const int quad = warp % 4;
    TileWalker tw;
    tw.init(args.n_per_graph, geo.N, args.C, geo.TN1);
    int as = 0;
    uint32_t aphase = 0;
    int sbuf = 0;                            // staging buffer of the next 64-column chunk
    for (long t = item0; t < total; t += item_step) {
      int q, m, nn, n;
      tw.locate(t, args.n_per_graph, geo.N, args.C, geo.TN1, q, m, nn, n);
      float a1 = 1.f, s1 = 0.f, a2 = 1.f, s2 = 0.f;
      if (args.coef_a) { a1 = args.coef_a[2 * q]; s1 = args.coef_a[2 * q + 1]; }
      if (args.coef_b) { a2 = args.coef_b[2 * q]; s2 = args.coef_b[2 * q + 1]; }
      const int r = quad * 32 + lane;        // physical row inside the tile; r == 127 is the ones row
      const int i = m * kTM1 + r;            // logical row
      float* cc = s_cc + as * BN;
      mbar_wait(&tmem_full[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * BN);
      // the warp that owns lane 127 publishes s1*a2*c2[j] for the tile's columns
      if (quad == 3) {
        const float k2 = s1 * a2;
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
          uint32_t rr[32];
          tmem_ld32(taddr + (uint32_t)c0, rr);
          tmem_wait_ld();
          if (lane == 31) {
#pragma unroll
            for (int u = 0; u < 32; ++u) cc[c0 + u] = k2 * __uint_as_float(rr[u]);
          }
        }
      }
      // r1 of this row sits in the tile's last column
      const float r1 = __uint_as_float(tmem_ld1(taddr + (uint32_t)(BN - 1)));
      tmem_wait_ld();
      asm volatile("bar.sync 1, 128;" ::: "memory");
      const float scale = a1 * a2;
      const float rc = fmaf(a1 * s2, r1, s1 * s2 * (float)n);
      const bool row_ok = (r < kTM1) && (i < n);
      const int jlog0 = nn * geo.TN1;        // logical column of tile column 0
      // The tile leaves through shared memory and TMA: every warp stages 64-column chunks of its 32 rows (128-byte
      // rows, 16-byte pieces XOR-swizzled by row) and stores them as one box.  Direct stores -- 16 bytes per thread
      // at a row pitch of NPC * 2 bytes -- were partial-sector writes and cost 40% of this kernel.  The quadrant
      // that ends with the ones row stores a 31-row box (row 127 belongs to the next row tile).
      const CUtensorMap* mo = (quad == 3) ? &map_o31 : &map_o32;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 64) {
        if (jlog0 + c0 >= n) break;          // columns beyond the graph: nothing to write (warp-uniform)
        uint8_t* buf = s_store + (size_t)(quad * 2 + sbuf) * 4096;
        if (lane == 0) bulk_wait_group_read1();   // the store issued two chunks ago has read this buffer
        __syncwarp();
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint32_t rr[32];
          tmem_ld32(taddr + (uint32_t)(c0 + 32 * h), rr);
          tmem_wait_ld();
          uint32_t pk[16];
#pragma unroll
          for (int u = 0; u < 16; ++u) {
            const int ca = c0 + 32 * h + 2 * u, cb = ca + 1;
            float x0 = fmaf(scale, __uint_as_float(rr[2 * u]), rc + cc[ca]);
            float x1 = fmaf(scale, __uint_as_float(rr[2 * u + 1]), rc + cc[cb]);
            if (!row_ok || ca == BN - 1 || jlog0 + ca >= n) x0 = 0.f;   // hole column / beyond the graph: zeros
            if (!row_ok || cb == BN - 1 || jlog0 + cb >= n) x1 = 0.f;
            pk[u] = Elem<T>::pack(x0, x1);
          }
#pragma unroll
          for (int vv = 0; vv < 4; ++vv)
            *reinterpret_cast<uint4*>(buf + lane * 128 + (((h * 4 + vv) ^ (lane & 7)) << 4)) =
                make_uint4(pk[4 * vv], pk[4 * vv + 1], pk[4 * vv + 2], pk[4 * vv + 3]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_3d(mo, buf, nn * BN + c0, m * kTM1 + quad * 32, q);
          bulk_commit_group();
        }
        sbuf ^= 1;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[as]);
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
    if (lane == 0) bulk_wait_group0();       // this warp's stores have landed before the CTA exits
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 0) {
    __syncwarp();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// =============================================================================================
// K_H: fused siamese head (models/trainers.py:67 + toolbox/losses.py:27-33 + toolbox/metrics.py:125-134):
// scores = E1^T E2 on tcgen05 with the row softmax / cross-entropy against the identity matching and the row
// argmax in the epilogue (online max / sum of exponentials over column tiles, flash style).  The (G,N,N) scores are
// written only on request; otherwise nothing but (sum CE, #correct) per (pair, row tile) leaves the SM.
//   A = E1^T tile (128 rows i x K = C), B = E2 tile (K = C x 256 columns j), both MN-major in shared memory, built here
//   from the fp32 embeddings as 16-bit (hi, lo) pairs: D = Ahi Bhi + Alo Bhi + Ahi Blo recovers fp32-level accuracy
//   (the dropped lo x lo term is 2^-22 relative) at 3 x the (tiny, K = C) MMA work.
// One CTA per (pair, 128-row tile); warps 0-3 = epilogue rows (TMEM quadrant = warp), warp 4 = MMA issuer; everybody
// converts operands.  kRowLse (training forward) also stores every row's log-sum-exp for the backward below; it is a
// template parameter, not a run-time flag, so that the inference instance is the kernel it was without it.
// The backward (tc_head_bwd_kernel) needs no (G,N,N) buffer either: it recomputes S tile by tile from the same (hi, lo)
// operands, forms dS = P - I in the epilogue from the saved lse, and accumulates dS E2^T (or dS^T E1^T) on tcgen05 as
// three (hi, lo) MMAs per product; coef[g] = d loss / d ce_sum[g] scales the fp32 accumulator, not the 16-bit operand
// (coef p falls below fp16's normal range at coef = 1 / #rows).  One CTA per (pair, 128-row tile) walks the column
// tiles for d E1, one per (pair, 128-column tile) walks the row tiles for d E2: every output is written once.
// =============================================================================================
// Graph 1 (rows i) has n_per_graph[g] <= N vertices, graph 2 (columns j) n2[g] <= N2; N2 == N, n2 == n_per_graph is the
// square head.  Row i's target is column i: rows i >= n2[g] have none and add nothing to (sum CE, #correct).
struct HeadArgs {
  const float* e1;       // (G,C,N)
  const float* e2;       // (G,C,N2)
  float* scores;         // (G,N,N2) or null
  float* partial;        // [G][MT][2] = (sum CE, #correct) of the row tile
  int G, C, N, MT;
  const int32_t* n_per_graph;
  float* row_lse;        // (G,N), kRowLse only: log sum_j exp(s_ij) of valid rows, 0 elsewhere
  int N2;
  const int32_t* n2;     // null: every graph 2 has N2 vertices
};

template <typename T, bool kRowLse>
__global__ void __launch_bounds__(160, 1) tc_head_kernel(const HeadArgs a) {
  extern __shared__ uint8_t smem_head[];
  uint8_t* smem = smem_head + ((1024u - (smem_u32(smem_head) & 1023u)) & 1023u);
  const int C = a.C, N = a.N;
  const uint32_t a_bytes = (uint32_t)C * 256u, b_bytes = (uint32_t)C * 512u;   // 128 rows / 256 columns x C x 2 bytes
  uint8_t* sAhi = smem;
  uint8_t* sAlo = sAhi + a_bytes;
  uint8_t* sBhi = sAlo + a_bytes;
  uint8_t* sBlo = sBhi + b_bytes;
  uint64_t* bar = reinterpret_cast<uint64_t*>(sBlo + b_bytes);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 1);
  float* red = reinterpret_cast<float*>(tmem_slot + 2);     // [4 warps][2]
  const int warp = uniform_warp_idx(), lane = threadIdx.x % 32;
  const int mt = blockIdx.x, b = blockIdx.y;
  const int N2 = a.N2;
  const int n = graph_n(a.n_per_graph, b, N), n2 = graph_n(a.n2, b, N2);
  const float* e1 = a.e1 + (size_t)b * C * N;
  const float* e2 = a.e2 + (size_t)b * C * N2;
  const int i0 = mt * 128;
  const bool want_scores = a.scores != nullptr;
  if (i0 >= n && !want_scores) {                            // nothing valid in this row tile
    if (threadIdx.x == 0) { a.partial[((size_t)b * a.MT + mt) * 2] = 0.f; a.partial[((size_t)b * a.MT + mt) * 2 + 1] = 0.f; }
    if constexpr (kRowLse)
      if (threadIdx.x < 128 && i0 + (int)threadIdx.x < N) a.row_lse[(size_t)b * N + i0 + threadIdx.x] = 0.f;
    return;
  }
  if (threadIdx.x == 0) { mbar_init(bar, 1); fence_barrier_init(); }
  if (warp == 4) tmem_alloc(tmem_slot, 256);
  // 8 consecutive MN elements of K row c -> one 16-byte chunk of the 128-byte-swizzled MN-major tile, as (hi, lo)
  auto put8 = [&](const float* src_row, int first, int limit, uint8_t* hi_tile, uint8_t* lo_tile, int c, int pos) {
    uint32_t hw[4], lw[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int x0 = first + 2 * u, x1 = x0 + 1;
      const float v0 = x0 < limit ? src_row[x0] : 0.f, v1 = x1 < limit ? src_row[x1] : 0.f;
      const float h0 = Elem<T>::to_float(Elem<T>::from_float(v0)), h1 = Elem<T>::to_float(Elem<T>::from_float(v1));
      hw[u] = Elem<T>::pack(v0, v1);
      lw[u] = Elem<T>::pack(v0 - h0, v1 - h1);
    }
    const uint32_t off = (uint32_t)(pos >> 6) * (uint32_t)(C * 128) + (uint32_t)c * 128u + (uint32_t)((((pos & 63) >> 3) ^ (c & 7)) << 4);
    *reinterpret_cast<uint4*>(hi_tile + off) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
    *reinterpret_cast<uint4*>(lo_tile + off) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
  };
  for (int idx = threadIdx.x; idx < C * 16; idx += blockDim.x) {      // A: rows i0 .. i0+127 of E1^T
    const int c = idx / 16, q = idx % 16;
    put8(e1 + (size_t)c * N, i0 + q * 8, n, sAhi, sAlo, c, q * 8);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int r = warp * 32 + lane;                           // row of the tile (epilogue warps)
  const int i = i0 + r;
  const bool row_ok = warp < 4 && i < n;
  float run_m = -INFINITY, run_l = 0.f, diag = 0.f, best = -INFINITY;
  int best_j = -1;
  uint32_t phase = 0;
  const int ncol = want_scores ? N2 : n2;
  for (int j0 = 0; j0 < ncol; j0 += 256) {
    if (j0 < n2) {
      for (int idx = threadIdx.x; idx < C * 32; idx += blockDim.x) {    // B: columns j0 .. j0+255 of E2
        const int c = idx / 32, q = idx % 32;
        put8(e2 + (size_t)c * N2, j0 + q * 8, n2, sBhi, sBlo, c, q * 8);
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncthreads();
      if (warp == 4) {
        tc_fence_after();
        const uint32_t idesc = make_idesc(Elem<T>::kFmt, 1, 1, 128, 256);
        const uint64_t dah = smem_desc_sw128(smem_u32(sAhi), (uint32_t)C * 128u, 1024u), dal = smem_desc_sw128(smem_u32(sAlo), (uint32_t)C * 128u, 1024u);
        const uint64_t dbh = smem_desc_sw128(smem_u32(sBhi), (uint32_t)C * 128u, 1024u), dbl = smem_desc_sw128(smem_u32(sBlo), (uint32_t)C * 128u, 1024u);
        if (elect_one_sync()) {
          for (int k = 0; k < C / 16; ++k) {
            const uint64_t adv = (uint64_t)((uint32_t)k * 2048u >> 4);
            mma_ss(tmem_base, dah + adv, dbh + adv, idesc, k > 0 ? 1u : 0u);
            mma_ss(tmem_base, dal + adv, dbh + adv, idesc, 1u);
            mma_ss(tmem_base, dah + adv, dbl + adv, idesc, 1u);
          }
          mma_commit(bar);
        }
        __syncwarp();
      }
    }
    if (warp < 4) {
      if (j0 < n2) { mbar_wait(bar, phase); phase ^= 1u; tc_fence_after(); }
      const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16);
      float* srow = want_scores && i < N ? a.scores + ((size_t)b * N + i) * N2 : nullptr;
#pragma unroll 1
      for (int c0 = 0; c0 < 256; c0 += 32) {
        if (j0 + c0 >= ncol) break;
        uint32_t v[32];
        if (j0 < n2) { tmem_ld32(taddr + (uint32_t)c0, v); tmem_wait_ld(); }
        if (row_ok && j0 + c0 < n2) {
          float cmax = -INFINITY;
#pragma unroll
          for (int u = 0; u < 32; ++u) {
            const int j = j0 + c0 + u;
            const float x = __uint_as_float(v[u]);
            if (j < n2) {
              cmax = fmaxf(cmax, x);
              if (x > best) { best = x; best_j = j; }
              if (j == i) diag = x;
            }
          }
          const float m_new = fmaxf(run_m, cmax);
          float acc = 0.f;
#pragma unroll
          for (int u = 0; u < 32; ++u)
            if (j0 + c0 + u < n2) acc += __expf(__uint_as_float(v[u]) - m_new);
          run_l = run_l * __expf(run_m - m_new) + acc;
          run_m = m_new;
        }
        if (srow) {
#pragma unroll
          for (int u = 0; u < 32; ++u) {
            const int j = j0 + c0 + u;
            if (j < N2) srow[j] = (row_ok && j < n2) ? __uint_as_float(v[u]) : 0.f;
          }
        }
      }
      tc_fence_before();
    }
    __syncthreads();                                        // accumulator and B tiles are free again
  }
  if (warp < 4) {
    if constexpr (kRowLse)
      if (i < N) a.row_lse[(size_t)b * N + i] = row_ok ? run_m + logf(run_l) : 0.f;
    const bool has_target = row_ok && i < n2;
    float ce = has_target ? (run_m + logf(run_l) - diag) : 0.f;
    float ok = (has_target && best_j == i) ? 1.f : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      ce += __shfl_xor_sync(0xffffffffu, ce, o);
      ok += __shfl_xor_sync(0xffffffffu, ok, o);
    }
    if (lane == 0) { red[2 * warp] = ce; red[2 * warp + 1] = ok; }
  }
  __syncthreads();
  if (threadIdx.x == 0) {                                   // fixed order: deterministic
    a.partial[((size_t)b * a.MT + mt) * 2] = (red[0] + red[2]) + (red[4] + red[6]);
    a.partial[((size_t)b * a.MT + mt) * 2 + 1] = (red[1] + red[3]) + (red[5] + red[7]);
  }
  if (warp == 4) {
    __syncwarp();
    tmem_dealloc(tmem_base, 256);
  }
}

__global__ void head_finalize_kernel(const float* __restrict__ partial, float* __restrict__ ce_sum, int32_t* __restrict__ correct,
                                     int G, int MT) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= G) return;
  float ce = 0.f, ok = 0.f;
  for (int m = 0; m < MT; ++m) { ce += partial[((size_t)b * MT + m) * 2]; ok += partial[((size_t)b * MT + m) * 2 + 1]; }
  ce_sum[b] = ce;
  correct[b] = (int32_t)(ok + 0.5f);
}

// K_H backward (see above).  kRows: the CTA owns 128 rows i of S (x = E1, y = E2, dx = d E1) and its rows' lse;
// otherwise 128 columns j (x = E2, y = E1, dx = d E2) and the walked tiles are rows of S, whose lse is staged in shared
// memory.  Per walked 128-wide tile t of y:
//   T = X^T Y_t (tcgen05, TMEM cols [0,128); = S or S^T)  ->  P = exp(s - lse_row) - [i == j], zero outside n x n,
//   as 16-bit (hi, lo) K-major tiles  ->  D (TMEM cols [128, 128 + C)) += P Y_t^T.
// The y tile is stored MN-major (K = channel) for the first product; the same bytes are the K-major B operand
// (K = position, N = channel) of the second.  The steps of one tile are serialised (commit / wait): the kernel is
// bound by the exponentials of the epilogue, not by the MMAs.  Rows i >= n2 have no target (forward): their dS row is
// zero, so the kRows CTA owns rows i < min(n1, n2) and the column CTA walks those rows only.
struct HeadBwdArgs {
  const float* x;        // (G,C,Nx): the side whose gradient this launch writes
  const float* y;        // (G,C,Ny): the other side
  const float* row_lse;  // (G,N1), N1 = Nx (kRows) or Ny
  const float* coef;     // [G]
  float* dx;             // (G,C,Nx)
  int C, Nx, Ny;
  const int32_t* nx;     // sizes of x's graphs (null: Nx) ...
  const int32_t* ny;     // ... and of y's (null: Ny)
};

template <typename T, bool kRows>
__global__ void __launch_bounds__(160, 1) tc_head_bwd_kernel(const HeadBwdArgs a) {
  extern __shared__ uint8_t smem_head_bwd[];
  uint8_t* smem = smem_head_bwd + ((1024u - (smem_u32(smem_head_bwd) & 1023u)) & 1023u);
  const int C = a.C, Nx = a.Nx, Ny = a.Ny;
  const uint32_t xy_bytes = (uint32_t)C * 256u;             // 128 positions x C x 2 bytes
  uint8_t* sXhi = smem;
  uint8_t* sXlo = sXhi + xy_bytes;
  uint8_t* sYhi = sXlo + xy_bytes;
  uint8_t* sYlo = sYhi + xy_bytes;
  uint8_t* sPhi = sYlo + xy_bytes;                          // [2 K chunks][128 rows][128 B], 16-byte units XOR (row & 7)
  uint8_t* sPlo = sPhi + 32768;
  uint64_t* bar = reinterpret_cast<uint64_t*>(sPlo + 32768);   // [0] T ready, [1] P Y^T done
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + 2);
  float* s_lse = reinterpret_cast<float*>(tmem_slot + 2);   // [128] lse of the walked rows (!kRows)
  const int warp = uniform_warp_idx(), lane = threadIdx.x % 32;
  const int t0 = blockIdx.x * 128, b = blockIdx.y;
  const int nx = graph_n(a.nx, b, Nx), ny = graph_n(a.ny, b, Ny);
  const int n_own = kRows ? min(nx, ny) : nx;               // owned positions with a nonzero gradient
  const int n_walk = kRows ? ny : min(nx, ny);              // walked positions with a nonzero dS
  const int N1 = kRows ? Nx : Ny;                           // pitch of row_lse
  const float* xg = a.x + (size_t)b * C * Nx;
  const float* yg = a.y + (size_t)b * C * Ny;
  float* dxg = a.dx + (size_t)b * C * Nx;
  if (t0 >= n_own || n_walk == 0) {                         // no valid position: exact zeros
    for (int idx = threadIdx.x; idx < C * 128; idx += blockDim.x) {
      const int c = idx / 128, p = t0 + idx % 128;
      if (p < Nx) dxg[(size_t)c * Nx + p] = 0.f;
    }
    return;
  }
  if (threadIdx.x == 0) { mbar_init(&bar[0], 1); mbar_init(&bar[1], 1); fence_barrier_init(); }
  if (warp == 4) tmem_alloc(tmem_slot, 256);
  auto put8 = [&](const float* src_row, int first, int limit, uint8_t* hi_tile, uint8_t* lo_tile, int c, int pos) {
    uint32_t hw[4], lw[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int x0 = first + 2 * u, x1 = x0 + 1;
      const float v0 = x0 < limit ? src_row[x0] : 0.f, v1 = x1 < limit ? src_row[x1] : 0.f;
      const float h0 = Elem<T>::to_float(Elem<T>::from_float(v0)), h1 = Elem<T>::to_float(Elem<T>::from_float(v1));
      hw[u] = Elem<T>::pack(v0, v1);
      lw[u] = Elem<T>::pack(v0 - h0, v1 - h1);
    }
    const uint32_t off = (uint32_t)(pos >> 6) * (uint32_t)(C * 128) + (uint32_t)c * 128u + (uint32_t)((((pos & 63) >> 3) ^ (c & 7)) << 4);
    *reinterpret_cast<uint4*>(hi_tile + off) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
    *reinterpret_cast<uint4*>(lo_tile + off) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
  };
  for (int idx = threadIdx.x; idx < C * 16; idx += blockDim.x) {
    const int c = idx / 16, q = idx % 16;
    put8(xg + (size_t)c * Nx, t0 + q * 8, n_own, sXhi, sXlo, c, q * 8);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int r = warp * 32 + lane;                           // row of the CTA's tile (epilogue warps)
  const int p_own = t0 + r;                                 // its position: i (kRows) or j
  const bool own_ok = warp < 4 && p_own < n_own;
  const float lse_own = (kRows && own_ok) ? a.row_lse[(size_t)b * N1 + p_own] : 0.f;
  uint32_t phase = 0;
  for (int w0 = 0; w0 < n_walk; w0 += 128) {
    if (w0 > 0) { mbar_wait(&bar[1], phase ^ 1u); tc_fence_after(); }   // previous P Y^T has read sY and sP
    for (int idx = threadIdx.x; idx < C * 16; idx += blockDim.x) {
      const int c = idx / 16, q = idx % 16;
      put8(yg + (size_t)c * Ny, w0 + q * 8, n_walk, sYhi, sYlo, c, q * 8);
    }
    if (!kRows && threadIdx.x < 128) s_lse[threadIdx.x] = w0 + (int)threadIdx.x < n_walk ? a.row_lse[(size_t)b * N1 + w0 + threadIdx.x] : 0.f;
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
      tc_fence_after();
      const uint32_t idesc = make_idesc(Elem<T>::kFmt, 1, 1, 128, 128);
      const uint64_t dxh = smem_desc_sw128(smem_u32(sXhi), (uint32_t)C * 128u, 1024u), dxl = smem_desc_sw128(smem_u32(sXlo), (uint32_t)C * 128u, 1024u);
      const uint64_t dyh = smem_desc_sw128(smem_u32(sYhi), (uint32_t)C * 128u, 1024u), dyl = smem_desc_sw128(smem_u32(sYlo), (uint32_t)C * 128u, 1024u);
      if (elect_one_sync()) {
        for (int k = 0; k < C / 16; ++k) {
          const uint64_t adv = (uint64_t)((uint32_t)k * 2048u >> 4);
          mma_ss(tmem_base, dxh + adv, dyh + adv, idesc, k > 0 ? 1u : 0u);
          mma_ss(tmem_base, dxl + adv, dyh + adv, idesc, 1u);
          mma_ss(tmem_base, dxh + adv, dyl + adv, idesc, 1u);
        }
        mma_commit(&bar[0]);
      }
      __syncwarp();
    }
    if (warp < 4) {
      mbar_wait(&bar[0], phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
      for (int c0 = 0; c0 < 128; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(taddr + (uint32_t)c0, v);
        tmem_wait_ld();
        float pv[32];
#pragma unroll
        for (int u = 0; u < 32; ++u) {
          const int q = w0 + c0 + u;                        // the walked position: j (kRows) or i
          const float lse = kRows ? lse_own : s_lse[c0 + u];
          pv[u] = (own_ok && q < n_walk) ? __expf(__uint_as_float(v[u]) - lse) - (q == p_own ? 1.f : 0.f) : 0.f;
        }
#pragma unroll
        for (int s8 = 0; s8 < 4; ++s8) {
          uint32_t hw[4], lw[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float v0 = pv[s8 * 8 + 2 * e], v1 = pv[s8 * 8 + 2 * e + 1];
            const float h0 = Elem<T>::to_float(Elem<T>::from_float(v0)), h1 = Elem<T>::to_float(Elem<T>::from_float(v1));
            hw[e] = Elem<T>::pack(v0, v1);
            lw[e] = Elem<T>::pack(v0 - h0, v1 - h1);
          }
          const int k = c0 + s8 * 8;                        // K position of the 8 values
          const uint32_t off = (uint32_t)(k >> 6) * 16384u + (uint32_t)r * 128u + (uint32_t)((((k & 63) >> 3) ^ (r & 7)) << 4);
          *reinterpret_cast<uint4*>(sPhi + off) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
          *reinterpret_cast<uint4*>(sPlo + off) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
        }
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
      tc_fence_after();
      const uint32_t idesc = make_idesc(Elem<T>::kFmt, 0, 0, 128, C);
      const uint64_t dph = smem_desc_sw128(smem_u32(sPhi), 16u, 1024u), dpl = smem_desc_sw128(smem_u32(sPlo), 16u, 1024u);
      const uint64_t dyh = smem_desc_sw128(smem_u32(sYhi), 16u, 1024u), dyl = smem_desc_sw128(smem_u32(sYlo), 16u, 1024u);
      if (elect_one_sync()) {
        for (int k = 0; k < 8; ++k) {                       // K = 128 walked positions, 16 per MMA
          const uint64_t pa = (uint64_t)(((uint32_t)(k >> 2) * 16384u + (uint32_t)(k & 3) * 32u) >> 4);
          const uint64_t ya = (uint64_t)(((uint32_t)(k >> 2) * (uint32_t)(C * 128) + (uint32_t)(k & 3) * 32u) >> 4);
          mma_ss(tmem_base + 128u, dph + pa, dyh + ya, idesc, (w0 > 0 || k > 0) ? 1u : 0u);
          mma_ss(tmem_base + 128u, dpl + pa, dyh + ya, idesc, 1u);
          mma_ss(tmem_base + 128u, dph + pa, dyl + ya, idesc, 1u);
        }
        mma_commit(&bar[1]);
      }
      __syncwarp();
    }
    phase ^= 1u;
  }
  if (warp < 4) {
    mbar_wait(&bar[1], phase ^ 1u);
    tc_fence_after();
    const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + 128u;
    const float cf = a.coef[b];
#pragma unroll 1
    for (int c0 = 0; c0 < C; c0 += 16) {
      uint32_t v[16];
      tmem_ld16(taddr + (uint32_t)c0, v);
      tmem_wait_ld();
      if (p_own < Nx) {
#pragma unroll
        for (int u = 0; u < 16; ++u) dxg[(size_t)(c0 + u) * Nx + p_own] = own_ok ? cf * __uint_as_float(v[u]) : 0.f;
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 4) {
    __syncwarp();
    tmem_dealloc(tmem_base, 256);
  }
}

// =============================================================================================
// host side
// =============================================================================================
using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                              const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                              CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeFn get_encode() {
  static EncodeFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeFn>(p);
  }
  return fn;
}

// 3-D tensor map over 16-bit data: dims (d0 contiguous, d1, d2), strides in elements, 128B swizzle.
int make_map3(CUtensorMap* m, int fmt_is_bf16, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
              uint64_t stride1_elems, uint64_t stride2_elems, uint32_t b0, uint32_t b1, uint32_t b2 = 1) {
  EncodeFn enc = get_encode();
  if (!enc) return fail(FGNN_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1_elems * 2, stride2_elems * 2};
  cuuint32_t box[3] = {b0, b1, b2};
  cuuint32_t estr[3] = {1, 1, 1};
  if ((reinterpret_cast<uintptr_t>(base) & 15) || (strides[0] & 15) || (strides[1] & 15))
    return fail(FGNN_ERR_INVALID, "tensor map alignment: base %p strides %llu %llu", base,
                (unsigned long long)strides[0], (unsigned long long)strides[1]);
  CUresult r = enc(m, fmt_is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(FGNN_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) dims %llu,%llu,%llu box %u,%u", (int)r,
                (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2, b0, b1);
  return FGNN_OK;
}

// [planes][rows][NPC] view of planes in layout l, boxes of 64 columns x box_rows rows x box_planes planes
template <typename T>
int plane_map(CUtensorMap* m, const T* base, Layout l, const Geo& geo, uint64_t planes, uint32_t box_rows, uint32_t box_planes = 1) {
  return make_map3(m, Elem<T>::kFmt, base, geo.NPC, geo.rows(l), planes, geo.NPC, (uint64_t)geo.stride(l), 64, box_rows, box_planes);
}

// flat [G][channels][PSC] view of layout-C planes: each plane is one row of PSC pixels; boxes of 64 pixels x box_channels
// channels of one graph (channels beyond `channels` are zero-filled)
template <typename T>
int pixel_map(CUtensorMap* m, const T* base, int channels, int G, const Geo& geo, uint32_t box_channels) {
  return make_map3(m, Elem<T>::kFmt, base, geo.PSC, channels, G, geo.PSC, (uint64_t)channels * geo.PSC, 64, box_channels);
}

// f(std::integral_constant<int, BN>{}) for the geometry's BN: the 128 x BN tile kernels are instantiated per BN
template <typename F>
int with_bn(const Geo& geo, F&& f) {
  if (geo.BN == 64) return f(std::integral_constant<int, 64>{});
  if (geo.BN == 128) return f(std::integral_constant<int, 128>{});
  return f(std::integral_constant<int, 256>{});
}

int num_sms() {   // of the CURRENT device (a process may drive several GPUs): not cached across devices
  static int cache[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && cache[dev]) return cache[dev];
  int n = 0;
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  if (n <= 0) n = 148;
  if (dev >= 0 && dev < 64) cache[dev] = n;
  return n;
}

int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v ? atoi(v) : dflt;
}

// ---- launchers -------------------------------------------------------------------------------
template <typename T>
int launch_matmul(const T* y1, const T* y2, T* out, const float* coef_a, const float* coef_b, int G, int C,
                  const Geo& geo, const int32_t* npg, cudaStream_t st) {
  CUtensorMap ma, mb;
  const uint64_t planes = (uint64_t)G * C;
  // K = physical column of Y1 (layout A) = physical row of Y2 (layout B); reads past either extent are zero filled
  if (int e = plane_map(&ma, y1, kLayoutA, geo, planes, 128)) return e;
  if (int e = plane_map(&mb, y2, kLayoutB, geo, planes, 64)) return e;
  // output (layout C) as 64-column x 32-row (31 for the quadrant that ends with the ones row) store boxes
  CUtensorMap mo32, mo31;
  if (int e = plane_map(&mo32, out, kLayoutC, geo, planes, 32)) return e;
  if (int e = plane_map(&mo31, out, kLayoutC, geo, planes, 31)) return e;
  MatmulArgs<T> a{G, C, geo, out, coef_a, coef_b, npg};
  const int grid = num_sms();
  return with_bn(geo, [&](auto bn) -> int {
    constexpr int BN = decltype(bn)::value;
    const size_t smem = MatmulCfg<BN>::kSmemBytes;
    prof::begin(prof::kMatmul, st);
    // per device and cheap: set on every call
    FGNN_CUDA(cudaFuncSetAttribute(tc_matmul_kernel<T, BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    tc_matmul_kernel<T, BN><<<grid, 192, smem, st>>>(ma, mb, mo32, mo31, a);
    prof::end(prof::kMatmul, st);
    FGNN_LAUNCHED();
    return FGNN_OK;
  });
}

// a conv's source: planes of c stored channels, the first c_real real, through the GraphNorm fold coef (null: identity)
template <typename T>
struct Src {
  const T* x;
  int c, c_real;
  const float* coef;   // [G][c][2] = {a, s}
};

// what a launch reads of one MLP: real shapes, first-layer weight w0 (co_real, the sources' c_real summed), b[l] of layer l
struct MlpLayers {
  const float* w0;
  const float* b[FGNN_MAX_DEPTH];
  int depth, co_real;
  const fgnn_mlp_params* gn;   // GraphNorm whose coefficients the launch finalises, or null (hidden layers, backward convs)
};

// mp's layers as one fused conv chain
MlpLayers chain(const fgnn_mlp_params& mp) {
  MlpLayers d{mp.w[0], {}, mp.depth, mp.c_out, &mp};
  for (int l = 0; l < mp.depth; ++l) d.b[l] = mp.b[l];
  return d;
}

// fold + conv chain(s) + statistics finalisation for 1 or 2 MLPs sharing their sources; see make_plan for the widths.
template <typename T>
struct MlpGroup {
  int nmlp, nsrc;
  MlpLayers mlp[2];
  Src<T> src[2];
  T* wf;             // [G][nmlp][C][K1g] folded first-layer weights
  float* bf;         // [G][nmlp][C] folded first-layer bias
  T* bt;             // [G][nmlp][C][16] folded first-layer bias as an MMA step (may be null for depth-1 launches)
  const T* wh;       // [nmlp][depth-1][C][Kh]
  float* bias_pad;   // room for [nmlp][depth-2][C] floats: the hidden biases zero-padded to C when c_out < C
  T* out[2];
  Layout out_mode[2];
  int ones[2];
  float* coef[2];
  double* stat_acc;  // [G][nmlp][C][2], zeroed by the launch
  double* stat_rec;  // deterministic mode: room for (G + mlp_grid) conv-chain statistics records (null: atomics)
  unsigned int* rowenc[2];   // fused max pooling of this MLP's output instead of storing it (see MlpArgs), or null
  // training path (depth-1 launches, see fgnn_tc_train.cuh)
  int relu_out;              // out = relu(conv + bias) instead of the raw accumulator
  float* gnstat[2];          // statistics kept for backward (or null)
};

int mlp_grid(int G, const Geo& geo) {
  const long total_tiles = (long)G * ((geo.PSC + kTileM - 1) / kTileM);
  return (int)std::max<long>(1, std::min<long>((long)num_sms(), total_tiles));
}

// doubles of the conv-chain statistics records a launch of G graphs at width C may fill (deterministic mode)
size_t stat_rec_doubles(int G, int C, const Geo& geo) { return (size_t)(G + mlp_grid(G, geo)) * stat_record_doubles(C); }

template <typename T, int COUT, int NMLP>
int launch_mlp_t(const MlpGroup<T>& M, int G, const Geo& geo, const int32_t* npg, cudaStream_t st) {
  MlpArgs<T> a{};
  a.G = G;
  a.geo = geo;
  a.nsrc = M.nsrc;
  for (int s = 0; s < M.nsrc; ++s) a.k_src[s] = round_up(M.src[s].c, 16);
  a.K1 = a.k_src[0] + a.k_src[1];
  a.K1g = round_up(a.K1, 64);
  a.depth = M.mlp[0].depth;
  a.Kh = COUT < 64 ? 64 : COUT;
  a.bias1 = M.bf;
  a.bias1_tile = M.bt;
  FGNN_CHECK_ARG(a.depth == 1 || M.bt != nullptr, "conv chains with hidden layers need the folded bias tile");
  for (int m = 0; m < NMLP; ++m) {
    FGNN_CHECK_ARG(M.mlp[m].depth == a.depth, "MLPs fused in one launch must have the same depth");
    for (int l = 0; l < a.depth; ++l) a.bias[m][l] = M.mlp[m].b[l];
    a.out[m] = M.out[m];
    a.out_mode[m] = M.out_mode[m];
    a.ones[m] = M.ones[m];
    a.rowenc[m] = M.rowenc[m];
  }
  a.stat_acc = M.stat_acc;
  a.n_per_graph = npg;
  FGNN_CHECK_ARG(a.K1 <= 256, "first-layer K=%d too wide for the tensor-core MLP kernel", a.K1);
  CUtensorMap mx[2], mw1, mwh, mo[2];
  for (int m = 0; m < NMLP; ++m)   // one 64-pixel row piece of all COUT channels per store
    if (int e = plane_map(&mo[m], M.out[m], M.out_mode[m], geo, (uint64_t)G * COUT, 1, COUT)) return e;
  if (NMLP == 1) mo[1] = mo[0];
  for (int s = 0; s < M.nsrc; ++s)
    if (int e = pixel_map(&mx[s], M.src[s].x, M.src[s].c, G, geo, a.k_src[s])) return e;
  if (M.nsrc == 1) mx[1] = mx[0];
  constexpr int is_bf16 = Elem<T>::kFmt;
  if (int e = make_map3(&mw1, is_bf16, M.wf, a.K1g, COUT, (uint64_t)G * NMLP, a.K1g, (uint64_t)COUT * a.K1g, 64, COUT)) return e;
  if (a.depth > 1) {
    if (int e = make_map3(&mwh, is_bf16, M.wh, a.Kh, COUT, (uint64_t)NMLP * (a.depth - 1), a.Kh, (uint64_t)COUT * a.Kh, 64, COUT)) return e;
  } else {
    mwh = mw1;
  }
  const size_t smem = MlpSmem<COUT, NMLP>::bytes(a.K1, a.K1g, a.depth, a.Kh);
  FGNN_CHECK_ARG(smem <= 227 * 1024, "MLP kernel needs %zu bytes of shared memory", smem);
  const bool pool = a.rowenc[0] != nullptr;
  FGNN_CHECK_ARG(!pool || NMLP == 1, "fused pooling is only built for single-MLP launches");
  FGNN_CHECK_ARG(!M.relu_out || (a.depth == 1 && !pool), "relu_out is a depth-1, non-pooled launch");
  const int grid = mlp_grid(G, geo);
  auto launch = [&](auto sum) -> int {
    using S = decltype(sum);
    auto kernel = M.relu_out ? tc_mlp_kernel<T, COUT, NMLP, false, true, S> : tc_mlp_kernel<T, COUT, NMLP, false, false, S>;
    if constexpr (NMLP == 1) {
      if (pool) kernel = tc_mlp_kernel<T, COUT, NMLP, true, false, S>;
    }
    // the opt-in is per device and cheap: set on every call
    FGNN_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    prof::begin(prof::kMlp, st);
    kernel<<<grid, kMlpThreads, smem, st>>>(mx[0], mx[1], mw1, mwh, mo[0], mo[1], a);
    prof::end(prof::kMlp, st);
    FGNN_LAUNCHED();
    return FGNN_OK;
  };
  if (!M.stat_rec) {
    FGNN_CUDA(cudaMemsetAsync(M.stat_acc, 0, (size_t)G * NMLP * COUT * 2 * sizeof(double), st));
    return launch(AtomicSum{});
  }
  // records of the launch (their statistics are only read when the coefficients are finalised)
  a.stat_acc = M.stat_rec;
  if (M.mlp[0].gn) FGNN_CUDA(cudaMemsetAsync(M.stat_rec, 0, (size_t)(G + grid) * stat_record_doubles(COUT) * sizeof(double), st));
  return launch(OrderedSum{});
}

template <typename T>
int launch_mlp(const MlpGroup<T>& M, int C, int G, const Geo& geo, const int32_t* npg, cudaStream_t st) {
  if (C == 32 && M.nmlp == 1) return launch_mlp_t<T, 32, 1>(M, G, geo, npg, st);
  if (C == 32 && M.nmlp == 2) return launch_mlp_t<T, 32, 2>(M, G, geo, npg, st);
  if (C == 64 && M.nmlp == 1) return launch_mlp_t<T, 64, 1>(M, G, geo, npg, st);
  if (C == 64 && M.nmlp == 2) return launch_mlp_t<T, 64, 2>(M, G, geo, npg, st);
  return fail(FGNN_ERR_UNSUPPORTED, "tensor-core path supports out_features 32 or 64 (got %d); use FGNN_FP32", C);
}

template <typename T>
int run_mlp_group(MlpGroup<T> M, int C, int G, const Geo& geo, const int32_t* npg, cudaStream_t st) {
  const int co_real = M.mlp[0].co_real;
  FoldArgs fa{};
  fa.nmlp = M.nmlp;
  fa.nsrc = M.nsrc;
  for (int m = 0; m < M.nmlp; ++m) { fa.w[m] = M.mlp[m].w0; fa.b[m] = M.mlp[m].b[0]; }
  for (int s = 0; s < M.nsrc; ++s) { fa.c[s] = M.src[s].c; fa.cr[s] = M.src[s].c_real; fa.coef[s] = M.src[s].coef; }
  fa.koff[0] = 0;
  fa.koff[1] = round_up(fa.c[0], 16);
  fa.c_out = C;
  fa.co_real = co_real;
  fa.K1g = round_up(fa.koff[1] + round_up(fa.c[1], 16), 64);
  FGNN_CHECK_ARG(fa.c[0] + fa.c[1] <= 512, "too many input channels for the fold kernel");
  fold_weights_kernel<T><<<dim3(G, M.nmlp, 8), 256, 0, st>>>(fa, M.wf, M.bf, M.bt);
  FGNN_LAUNCHED();
  // the conv-chain kernel reads C entries of every hidden bias that feeds a ReLU: point it at zero-padded copies
  const int depth = M.mlp[0].depth;
  if (co_real < C && depth > 2) {
    FGNN_CHECK_ARG(M.bias_pad != nullptr, "zero-padded hidden layers need room for their biases");
    PadBatch pb{};
    for (int m = 0; m < M.nmlp; ++m)
      for (int l = 1; l < depth - 1; ++l) {
        const int v = m * (depth - 2) + l - 1;
        pb.src[v] = M.mlp[m].b[l];
        M.mlp[m].b[l] = M.bias_pad + (size_t)v * C;
      }
    pad_vectors_kernel<<<dim3(1, M.nmlp * (depth - 2)), 64, 0, st>>>(pb, M.bias_pad, C, co_real);
    FGNN_LAUNCHED();
  }
  if (int e = launch_mlp<T>(M, C, G, geo, npg, st)) return e;
  if (!M.mlp[0].gn) return FGNN_OK;
  if (M.stat_rec) {
    prof::begin(prof::kStats, st);
    stat_records_reduce_kernel<<<G * M.nmlp * C, kStatReduceThreads, 0, st>>>(M.stat_rec, M.stat_acc, G, M.nmlp, C,
                                                                               mlp_grid(G, geo), geo, npg);
    prof::end(prof::kStats, st);
    FGNN_LAUNCHED();
  }
  CoefArgs ca{};
  ca.acc = M.stat_acc;
  ca.nmlp = M.nmlp;
  ca.C = C;
  ca.N = geo.N;
  ca.n_per_graph = npg;
  for (int m = 0; m < M.nmlp; ++m) {
    ca.coef[m] = M.coef[m];
    ca.gw[m] = M.mlp[m].gn->gn_w;
    ca.gb[m] = M.mlp[m].gn->gn_b;
    ca.eps[m] = M.mlp[m].gn->eps;
    ca.constant_n[m] = M.mlp[m].gn->constant_n;
    ca.co_real[m] = M.mlp[m].co_real;
    ca.gnstat[m] = M.gnstat[m];
  }
  const int total = G * M.nmlp * C;
  prof::begin(prof::kStats, st);
  finalize_coef_kernel<<<ceil_div(total, 256), 256, 0, st>>>(ca, total);
  prof::end(prof::kStats, st);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

// ---- workspace plan -----------------------------------------------------------------------------
struct Plan {
  int chunk, C, cin0, depth_max;
  Geo geo;
  int K1g12_max, K1g3_max;
};

// Widths.  The kernels run one width C in {32, 64} through every block: 32 when the widest MLP output is at most 32, else
// 64.  Each block has one real output width co <= C (its three MLPs'), and its output planes hold C channels, of which
// the first co are real; the input planes hold cin0 channels.  Parameters keep their real shapes, and every kernel that
// reads one maps real indices to stored ones; mlp3's first layer reads cat[mult, block input], real columns [0, co) at
// stored [0, C) and real [co, co + cin) at stored [C, C + cin).  Padded rows, columns, biases and GraphNorm affines are
// zero, so the padded channels are exactly zero everywhere (a = s = 0) and the embeddings are (G, co_last, N).
int make_plan(const fgnn_embed_params& p, int G, int N, Plan& pl) {
  if (N > kMaxN) return fail(FGNN_ERR_UNSUPPORTED, "tensor-core path supports N <= %d (got %d)", kMaxN, N);
  pl.geo = make_geo(N);
  pl.cin0 = p.block[0].mlp1.c_in;
  pl.depth_max = 1;
  pl.K1g12_max = 64;
  pl.K1g3_max = 64;
  int cmax = 0;
  for (int b = 0; b < p.num_blocks; ++b) {
    const fgnn_block_params& bp = p.block[b];
    const int co = bp.mlp1.c_out;
    if (co < 1 || bp.mlp2.c_out != co || bp.mlp3.c_out != co)
      return fail(FGNN_ERR_INVALID, "block %d: mlp1, mlp2 and mlp3 must have the same c_out >= 1", b);
    if (co > 64)
      return fail(FGNN_ERR_UNSUPPORTED, "tensor-core path supports in/out_features up to 64 (got %d); use FGNN_FP32", co);
    cmax = std::max(cmax, co);
  }
  pl.C = cmax <= 32 ? 32 : 64;
  int cur = pl.cin0, cur_store = pl.cin0;
  for (int b = 0; b < p.num_blocks; ++b) {
    const fgnn_block_params& bp = p.block[b];
    const int co = bp.mlp1.c_out;
    if (bp.mlp1.c_in != cur || bp.mlp2.c_in != cur || bp.mlp3.c_in != cur + co)
      return fail(FGNN_ERR_INVALID, "block %d: channel counts do not chain", b);
    if (bp.mlp1.depth != bp.mlp2.depth)
      return fail(FGNN_ERR_UNSUPPORTED, "block %d: mlp1 and mlp2 must have the same depth", b);
    pl.depth_max = std::max(pl.depth_max, std::max(bp.mlp1.depth, std::max(bp.mlp2.depth, bp.mlp3.depth)));
    pl.K1g12_max = std::max(pl.K1g12_max, round_up(round_up(cur_store, 16), 64));
    pl.K1g3_max = std::max(pl.K1g3_max, round_up(pl.C + round_up(cur_store, 16), 64));
    cur = co;
    cur_store = pl.C;
  }
  if (pl.cin0 > 64) return fail(FGNN_ERR_UNSUPPORTED, "original_features_num %d > 64 unsupported", pl.cin0);
  const int chunk_env = env_int("FGNN_TC_CHUNK", 0);
  // per_graph: 16-bit planes of one graph (input, two block outputs, mult, Y1, Y2): 11.6 GB at N = 4096, C = 64
  long per_graph = ((long)(3 * pl.C + pl.cin0) * pl.geo.PSC + (long)pl.C * (pl.geo.PSA + pl.geo.PSB)) * 2;
  // activation planes of one pass: at most FGNN_TC_WS_GB (default 16) GB of the caller's workspace; the batch is cut
  // into EQUAL passes (64 graphs at the headline shape need 9.8 GB: one pass)
  long budget = (long)std::max(1, env_int("FGNN_TC_WS_GB", 16)) << 30;
  long chunk = chunk_env > 0 ? chunk_env : std::max<long>(1, budget / std::max<long>(per_graph, 1));
  chunk = std::min<long>(chunk, 65535 / std::max(pl.C, pl.cin0));   // grid.y limits of the helper kernels
  chunk = std::min<long>(G, chunk);
  const long passes = (G + chunk - 1) / chunk;
  pl.chunk = (int)((G + passes - 1) / passes);
  // The conv-chain kernel numbers the (graph, 128-pixel tile) work of a launch, times two fused MLPs, in int, and the
  // pixel offset of a tile inside its graph too.  Refuse a plan whose counts could overflow rather than widen them.
  const long tiles_per_graph = (pl.geo.PSC + kTileM - 1) / kTileM;
  if (pl.geo.PSC > INT_MAX || (long)pl.chunk * 2 * tiles_per_graph > INT_MAX)
    return fail(FGNN_ERR_UNSUPPORTED, "tensor-core path: %d graphs of N=%d per pass exceed the kernels' 32-bit tile counts",
                pl.chunk, N);
  return FGNN_OK;
}

struct Buffers {
  void *xin, *xa, *xb, *y1, *y2, *mult;        // 16-bit planes
  float *coef1, *coef2, *coef3a, *coef3b;      // [chunk][C][2]
  void *wf12, *wf3;                            // folded first-layer weights
  float *bf12, *bf3;                           // folded first-layer biases
  void *bt12, *bt3;                            // the same as 16-bit MMA-step tiles
  double* stat_acc;                            // [chunk][2][C][2]
  void* wh;                                    // [blocks][3][depth-1][C][Kh]
  unsigned int* rowenc;                        // [chunk][C][N][2] row max / min codes of the last block's output
  double* stat_rec;                            // deterministic mode: conv-chain statistics records (else null)
};

size_t carve(const Plan& pl, int num_blocks, bool det, Arena& ar, Buffers& B) {
  const size_t actC = (size_t)pl.chunk * pl.C * pl.geo.stride(kLayoutC);
  B.xin = ar.take<uint16_t>((size_t)pl.chunk * pl.cin0 * pl.geo.stride(kLayoutC), 1024);
  B.xa = ar.take<uint16_t>(actC, 1024);
  B.xb = ar.take<uint16_t>(actC, 1024);
  B.y1 = ar.take<uint16_t>((size_t)pl.chunk * pl.C * pl.geo.stride(kLayoutA), 1024);
  B.y2 = ar.take<uint16_t>((size_t)pl.chunk * pl.C * pl.geo.stride(kLayoutB), 1024);
  B.mult = ar.take<uint16_t>(actC, 1024);
  const size_t nc = (size_t)pl.chunk * pl.C;
  B.coef1 = ar.take<float>(nc * 2);
  B.coef2 = ar.take<float>(nc * 2);
  B.coef3a = ar.take<float>(nc * 2);
  B.coef3b = ar.take<float>(nc * 2);
  B.wf12 = ar.take<uint16_t>(2 * nc * pl.K1g12_max, 1024);
  B.wf3 = ar.take<uint16_t>(nc * pl.K1g3_max, 1024);
  B.bf12 = ar.take<float>(2 * nc);
  B.bf3 = ar.take<float>(nc);
  B.bt12 = ar.take<uint16_t>(2 * nc * 16, 1024);
  B.bt3 = ar.take<uint16_t>(nc * 16, 1024);
  B.stat_acc = ar.take<double>(4 * nc);
  const int Kh = pl.C < 64 ? 64 : pl.C;
  B.wh = ar.take<uint16_t>((size_t)num_blocks * 3 * std::max(pl.depth_max - 1, 1) * pl.C * Kh, 1024);
  B.rowenc = ar.take<unsigned int>(nc * pl.geo.N * 2, 1024);
  B.stat_rec = det ? ar.take<double>(stat_rec_doubles(pl.chunk, pl.C, pl.geo)) : nullptr;
  return align_up(ar.off, 1024);
}

template <typename T>
int embed_fwd_t(const fgnn_embed_params& p, bool det, const float* x, const uint8_t* adj, float* emb, int G, int N,
                const int32_t* npg, void* ws, size_t ws_bytes, cudaStream_t st) {
  Plan pl;
  if (int e = make_plan(p, G, N, pl)) return e;
  Arena ar(ws, ws_bytes);
  Buffers B;
  size_t need = carve(pl, p.num_blocks, det, ar, B);
  if (need > ws_bytes) return fail(FGNN_ERR_WORKSPACE, "embed workspace too small: %zu < %zu", ws_bytes, need);
  const int C = pl.C;
  const Geo& geo = pl.geo;
  const int Kh = C < 64 ? 64 : C;
  const int dm1 = std::max(pl.depth_max - 1, 1);
  // hidden-layer weights -> 16-bit, once per call.  Layout [block][3 * dm1 matrices][C][Kh]: mlp1's and
  // mlp2's matrices are packed back to back (one tensor map serves the fused launch), mlp3's start at 2*dm1.
  for (int b = 0; b < p.num_blocks; ++b) {
    const fgnn_mlp_params* mlps[3] = {&p.block[b].mlp1, &p.block[b].mlp2, &p.block[b].mlp3};
    ConvertBatch cb{};
    cb.rows = cb.cols = p.block[b].mlp1.c_out;
    int nmat = 0;
    for (int j = 0; j < 3; ++j)
      for (int l = 1; l < mlps[j]->depth; ++l) {
        const int dj = mlps[j]->depth - 1;
        cb.src[nmat] = mlps[j]->w[l];
        cb.dst_off[nmat] = (long)(((size_t)b * 3 * dm1 + (size_t)(j < 2 ? j * dj : 2 * dm1) + (l - 1)) * C * Kh);
        ++nmat;
      }
    if (nmat > 0) {
      convert_weights_batch_kernel<T><<<dim3(ceil_div(C * Kh, 256), nmat), 256, 0, st>>>(cb, reinterpret_cast<T*>(B.wh), C, Kh);
      FGNN_LAUNCHED();
    }
  }
  for (int g0 = 0; g0 < G; g0 += pl.chunk) {
    const int gc = std::min(pl.chunk, G - g0);
    const int32_t* n_c = npg ? npg + g0 : nullptr;
    if (adj) {
      const long rows = (long)gc * N;
      adjacency_to_planes_kernel<T><<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(adj + (size_t)g0 * N * N,
                                                                                reinterpret_cast<T*>(B.xin), geo, rows, n_c);
      FGNN_LAUNCHED();
    } else {
      dim3 grid((unsigned)std::min(N, 256), gc * pl.cin0);
      to_planes_c_kernel<T><<<grid, 256, 0, st>>>(x + (size_t)g0 * pl.cin0 * N * N, reinterpret_cast<T*>(B.xin), pl.cin0, geo, n_c);
      FGNN_LAUNCHED();
    }
    {
      dim3 grid(4, gc * C);
      zero_inserted_rows_kernel<T><<<grid, 256, 0, st>>>(reinterpret_cast<T*>(B.y2), geo, kLayoutB);
      FGNN_LAUNCHED();
    }
    Src<T> cur{reinterpret_cast<const T*>(B.xin), pl.cin0, pl.cin0, nullptr};
    T* nxt = reinterpret_cast<T*>(B.xa);
    float* nxt_coef = B.coef3a;
    T* y1 = reinterpret_cast<T*>(B.y1);
    T* y2 = reinterpret_cast<T*>(B.y2);
    T* mult = reinterpret_cast<T*>(B.mult);
    for (int b = 0; b < p.num_blocks; ++b) {
      const fgnn_block_params& bp = p.block[b];
      const int co = bp.mlp1.c_out;
      const T* whb = reinterpret_cast<const T*>(B.wh) + (size_t)b * 3 * dm1 * C * Kh;
      // zero-padded hidden biases live in the other group's folded-weight buffer, which is free while a group runs
      // (wf3 holds at least C * 64 and wf12 2 C * 64 16-bit values: room for 2 (FGNN_MAX_DEPTH - 2) C floats)
      {
        MlpGroup<T> M{};
        M.nmlp = 2;
        M.mlp[0] = chain(bp.mlp1); M.mlp[1] = chain(bp.mlp2);
        M.src[0] = cur; M.nsrc = 1;
        M.wf = reinterpret_cast<T*>(B.wf12); M.bf = B.bf12; M.bt = reinterpret_cast<T*>(B.bt12);
        M.wh = whb;
        M.bias_pad = static_cast<float*>(B.wf3);
        M.out[0] = y1; M.out_mode[0] = kLayoutA; M.ones[0] = 1; M.coef[0] = B.coef1;
        M.out[1] = y2; M.out_mode[1] = kLayoutB; M.ones[1] = 1; M.coef[1] = B.coef2;
        M.stat_acc = B.stat_acc;
        M.stat_rec = B.stat_rec;
        if (int e = run_mlp_group<T>(M, C, gc, geo, n_c, st)) return e;
      }
      if (int e = launch_matmul<T>(y1, y2, mult, B.coef1, B.coef2, gc, C, geo, n_c, st)) return e;
      {
        MlpGroup<T> M{};
        M.nmlp = 1;
        M.mlp[0] = chain(bp.mlp3);
        M.src[0] = Src<T>{mult, C, co, nullptr}; M.src[1] = cur; M.nsrc = 2;
        M.wf = reinterpret_cast<T*>(B.wf3); M.bf = B.bf3; M.bt = reinterpret_cast<T*>(B.bt3);
        M.wh = whb + (size_t)2 * dm1 * C * Kh;
        M.bias_pad = static_cast<float*>(B.wf12);
        M.out[0] = nxt; M.out_mode[0] = kLayoutC; M.ones[0] = 0; M.coef[0] = nxt_coef;
        M.stat_acc = B.stat_acc;
        M.stat_rec = B.stat_rec;
        if (b == p.num_blocks - 1) {
          // the last block's output is only ever max-pooled: keep its row max / min and never write the planes
          M.rowenc[0] = B.rowenc;
          FGNN_CUDA(cudaMemsetAsync(B.rowenc, 0, (size_t)gc * C * N * 2 * sizeof(unsigned int), st));
        }
        if (int e = run_mlp_group<T>(M, C, gc, geo, n_c, st)) return e;
      }
      cur = Src<T>{nxt, C, co, nxt_coef};
      nxt = (nxt == reinterpret_cast<T*>(B.xa)) ? reinterpret_cast<T*>(B.xb) : reinterpret_cast<T*>(B.xa);
      nxt_coef = (nxt_coef == B.coef3a) ? B.coef3b : B.coef3a;
    }
    const long rows = (long)gc * C * N;
    pool_finalize_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(B.rowenc, cur.coef, emb + (size_t)g0 * cur.c_real * N, C,
                                                                       cur.c_real, N, rows, n_c);
    FGNN_LAUNCHED();
  }
  return FGNN_OK;
}

#include "fgnn_tc_train.cuh"

// Guard of the 16-bit entry points: an sm_100 device, then f(T{}) with T the element type of `precision`; any other
// precision is refused.
template <typename F>
int with_16bit(int precision, const char* what, F&& f) {
  if (!fgnn_device_supports_tcgen05())
    return fail(FGNN_ERR_UNSUPPORTED, "%s needs an sm_100 device (tcgen05); there is no fallback", what);
  if (precision == FGNN_BF16) return f(__nv_bfloat16{});
  if (precision == FGNN_FP16) return f(__half{});
  return fail(FGNN_ERR_INVALID, "%s supports FGNN_BF16 / FGNN_FP16 only (got precision %d)", what, precision);
}

}  // namespace

size_t embed_train_workspace_bytes(const fgnn_embed_params& p, int G, int N, bool det, bool ckpt) {
  TrainPlan tp;
  if (make_train_plan(p, G, N, det, ckpt, tp)) return 0;
  return train_workspace_bytes(tp);
}

int embed_fwd_train(const fgnn_embed_params& p, int precision, bool det, bool ckpt, const float* x, float* emb, int G, int N,
                    const int32_t* n_per_graph, void* ws, size_t ws_bytes, cudaStream_t st) {
  return with_16bit(precision, "fgnn_embed_fwd_train", [&](auto t) -> int {
    if (reinterpret_cast<uintptr_t>(ws) & 1023) return fail(FGNN_ERR_INVALID, "workspace must be 1024-byte aligned");
    return embed_fwd_train_t<decltype(t)>(p, det, ckpt, x, emb, G, N, n_per_graph, ws, ws_bytes, st);
  });
}

int embed_bwd(const fgnn_embed_params& p, const fgnn_embed_grads& g, int precision, bool det, bool ckpt, const float* demb,
              int grad_scale_log2, int G, int N, const int32_t* n_per_graph, void* ws, size_t ws_bytes, cudaStream_t st) {
  return with_16bit(precision, "fgnn_embed_bwd", [&](auto t) -> int {
    if (reinterpret_cast<uintptr_t>(ws) & 1023) return fail(FGNN_ERR_INVALID, "workspace must be 1024-byte aligned");
    if (grad_scale_log2 < -24 || grad_scale_log2 > 15) return fail(FGNN_ERR_INVALID, "grad_scale_log2 %d outside [-24, 15]", grad_scale_log2);
    return embed_bwd_t<decltype(t)>(p, g, det, ckpt, demb, grad_scale_log2, G, N, n_per_graph, ws, ws_bytes, st);
  });
}

size_t embed_workspace_bytes(const fgnn_embed_params& p, int G, int N, bool det) {
  Plan pl;
  if (make_plan(p, G, N, pl)) return 0;
  Arena ar(nullptr, 0);
  Buffers B;
  return carve(pl, p.num_blocks, det, ar, B);
}

int embed_fwd(const fgnn_embed_params& p, int precision, bool det, const float* x, float* emb, int G, int N,
              const int32_t* n_per_graph, void* ws, size_t ws_bytes, cudaStream_t st) {
  return with_16bit(precision, "fgnn_embed_fwd", [&](auto t) -> int {
    if (reinterpret_cast<uintptr_t>(ws) & 1023) return fail(FGNN_ERR_INVALID, "workspace must be 1024-byte aligned");
    return embed_fwd_t<decltype(t)>(p, det, x, nullptr, emb, G, N, n_per_graph, ws, ws_bytes, st);
  });
}

int embed_fwd_adjacency(const fgnn_embed_params& p, int precision, bool det, const uint8_t* adj, float* emb, int G, int N,
                        const int32_t* n_per_graph, void* ws, size_t ws_bytes, cudaStream_t st) {
  return with_16bit(precision, "fgnn_embed_fwd_adjacency_u8", [&](auto t) -> int {
    if (reinterpret_cast<uintptr_t>(ws) & 1023) return fail(FGNN_ERR_INVALID, "workspace must be 1024-byte aligned");
    FGNN_CHECK_ARG(p.num_blocks >= 1 && p.block[0].mlp1.c_in == 2,
                   "the adjacency input builds exactly the reference's 2 features (W, diag(deg))");
    return embed_fwd_t<decltype(t)>(p, det, nullptr, adj, emb, G, N, n_per_graph, ws, ws_bytes, st);
  });
}

size_t head_workspace_bytes(int G, int N) { return align_up((size_t)G * ((N + 127) / 128) * 2 * sizeof(float), 256); }

template <typename T, bool kRowLse>
int head_fwd_t(const float* e1, const float* e2, float* scores, float* ce_sum, int32_t* correct, float* row_lse, int G, int C,
               int N1, int N2, const int32_t* n1, const int32_t* n2, void* ws, cudaStream_t st) {
  HeadArgs a{};
  a.e1 = e1; a.e2 = e2; a.scores = scores;
  a.partial = static_cast<float*>(ws);
  a.G = G; a.C = C; a.N = N1; a.MT = (N1 + 127) / 128;
  a.n_per_graph = n1;
  a.row_lse = row_lse;
  a.N2 = N2; a.n2 = n2;
  const size_t smem = 1024 + (size_t)C * 256 * 2 + (size_t)C * 512 * 2 + 128;
  FGNN_CUDA(cudaFuncSetAttribute(tc_head_kernel<T, kRowLse>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  prof::begin(prof::kGlue, st);
  tc_head_kernel<T, kRowLse><<<dim3(a.MT, G), 160, smem, st>>>(a);
  FGNN_LAUNCHED();
  head_finalize_kernel<<<ceil_div(G, 128), 128, 0, st>>>(a.partial, ce_sum, correct, G, a.MT);
  prof::end(prof::kGlue, st);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

// the shapes every fused-head entry point accepts
int check_head_shape(int G, int C, int N1, int N2) {
  FGNN_CHECK_ARG(G >= 1 && G <= 65535 && N1 >= 1 && N1 <= kMaxN && N2 >= 1 && N2 <= kMaxN,
                 "fused head supports G <= 65535 and N1, N2 <= %d (got G=%d N1=%d N2=%d)", kMaxN, G, N1, N2);
  FGNN_CHECK_ARG(C >= 16 && C <= 128 && C % 16 == 0, "the fused head needs an embedding width that is a multiple of 16, at most 128 (got %d)", C);
  return FGNN_OK;
}

int head_fwd(int precision, const float* e1, const float* e2, float* scores, float* ce_sum, int32_t* correct, int G, int C,
             int N1, int N2, const int32_t* n1, const int32_t* n2, void* ws, size_t ws_bytes, cudaStream_t st) {
  return with_16bit(precision, "fgnn_head_pair_fwd", [&](auto t) -> int {
    FGNN_CHECK_ARG(e1 && e2 && ce_sum && correct && ws, "null pointer");
    if (int e = check_head_shape(G, C, N1, N2)) return e;
    if (ws_bytes < head_workspace_bytes(G, N1)) return fail(FGNN_ERR_WORKSPACE, "head workspace too small");
    return head_fwd_t<decltype(t), false>(e1, e2, scores, ce_sum, correct, nullptr, G, C, N1, N2, n1, n2, ws, st);
  });
}

int head_fwd_train(int precision, const float* e1, const float* e2, float* ce_sum, int32_t* correct, float* row_lse, int G,
                   int C, int N1, int N2, const int32_t* n1, const int32_t* n2, void* ws, size_t ws_bytes, cudaStream_t st) {
  return with_16bit(precision, "fgnn_head_pair_fwd_train", [&](auto t) -> int {
    FGNN_CHECK_ARG(e1 && e2 && ce_sum && correct && row_lse && ws, "null pointer");
    if (int e = check_head_shape(G, C, N1, N2)) return e;
    if (ws_bytes < head_workspace_bytes(G, N1)) return fail(FGNN_ERR_WORKSPACE, "head workspace too small");
    return head_fwd_t<decltype(t), true>(e1, e2, nullptr, ce_sum, correct, row_lse, G, C, N1, N2, n1, n2, ws, st);
  });
}

int head_bwd(int precision, const float* e1, const float* e2, const float* row_lse, const float* coef, float* de1, float* de2,
             int G, int C, int N1, int N2, const int32_t* n1, const int32_t* n2, cudaStream_t st) {
  return with_16bit(precision, "fgnn_head_pair_bwd", [&](auto t) -> int {
    using T = decltype(t);
    FGNN_CHECK_ARG(e1 && e2 && row_lse && coef && de1 && de2, "null pointer");
    if (int e = check_head_shape(G, C, N1, N2)) return e;
    const size_t smem = 1024 + (size_t)C * 256 * 4 + 2 * 32768 + 16 + 8 + 128 * sizeof(float);
    prof::begin(prof::kGlue, st);
    FGNN_CUDA(cudaFuncSetAttribute(tc_head_bwd_kernel<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    tc_head_bwd_kernel<T, true><<<dim3((N1 + 127) / 128, G), 160, smem, st>>>(HeadBwdArgs{e1, e2, row_lse, coef, de1, C, N1, N2, n1, n2});
    FGNN_LAUNCHED();
    FGNN_CUDA(cudaFuncSetAttribute(tc_head_bwd_kernel<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    tc_head_bwd_kernel<T, false><<<dim3((N2 + 127) / 128, G), 160, smem, st>>>(HeadBwdArgs{e2, e1, row_lse, coef, de2, C, N2, N1, n2, n1});
    prof::end(prof::kGlue, st);
    FGNN_LAUNCHED();
    return FGNN_OK;
  });
}

// ---- debug: one tensor-core matmul on fp32 host-layout tensors ---------------------------------
size_t debug_matmul_workspace_bytes(int G, int C, int N) {
  Geo geo = make_geo(N);
  return align_up(((size_t)G * C * (geo.PSC + geo.PSA + geo.PSB)) * 2 + 8192, 1024);
}

template <typename T>
int debug_matmul_t(const float* a, const float* b, float* out, int G, int C, int N, const int32_t* npg, void* ws,
                   size_t ws_bytes, cudaStream_t st) {
  Geo geo = make_geo(N);
  if (ws_bytes < debug_matmul_workspace_bytes(G, C, N)) return fail(FGNN_ERR_WORKSPACE, "debug workspace too small");
  Arena ar(ws, ws_bytes);
  T* y1 = ar.take<T>((size_t)G * C * geo.stride(kLayoutA), 1024);
  T* y2 = ar.take<T>((size_t)G * C * geo.stride(kLayoutB), 1024);
  T* mo = ar.take<T>((size_t)G * C * geo.stride(kLayoutC), 1024);
  auto grid = [&](Layout l) { return dim3((unsigned)std::min<long>(64, (geo.stride(l) + 255) / 256), G * C); };
  to_planes_kernel<T><<<grid(kLayoutA), 256, 0, st>>>(a, y1, C, geo, kLayoutA, npg);
  FGNN_LAUNCHED();
  to_planes_kernel<T><<<grid(kLayoutB), 256, 0, st>>>(b, y2, C, geo, kLayoutB, npg);
  FGNN_LAUNCHED();
  FGNN_CUDA(cudaMemsetAsync(mo, 0, (size_t)G * C * geo.PSC * sizeof(T), st));
  if (int e = launch_matmul<T>(y1, y2, mo, nullptr, nullptr, G, C, geo, npg, st)) return e;
  from_planes_kernel<T><<<grid(kLayoutC), 256, 0, st>>>(mo, out, nullptr, C, geo, npg);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

int debug_matmul(int precision, const float* a, const float* b, float* out, int G, int C, int N,
                 const int32_t* n_per_graph, void* ws, size_t ws_bytes, cudaStream_t st) {
  return with_16bit(precision, "fgnn_debug_tc_matmul", [&](auto t) -> int {
    FGNN_CHECK_ARG(a && b && out && ws, "null pointer");
    FGNN_CHECK_ARG(N <= kMaxN, "tensor-core matmul supports N <= %d (got %d)", kMaxN, N);
    return debug_matmul_t<decltype(t)>(a, b, out, G, C, N, n_per_graph, ws, ws_bytes, st);
  });
}

// ---- debug: one tensor-core MlpBlock_Real (fold -> conv chain + statistics -> normalise) ----------
size_t debug_mlp_workspace_bytes(int G, int c_in, int c_out, int depth, int N) {
  Geo geo = make_geo(N);
  const int K1g = round_up(round_up(c_in, 16), 64);
  const int Kh = c_out < 64 ? 64 : c_out;
  return align_up((size_t)G * (c_in + c_out) * geo.PSC * 2 + (size_t)G * c_out * K1g * 2 +
                      (size_t)std::max(depth - 1, 1) * c_out * Kh * 2 + (size_t)G * c_out * (3 * 4 + 16 + 32) + 16384, 1024);
}

template <typename T>
int debug_mlp_t(const fgnn_mlp_params& mp, const float* x, float* y, int G, int N, const int32_t* npg, void* ws,
                size_t ws_bytes, cudaStream_t st) {
  Geo geo = make_geo(N);
  const int C = mp.c_out;
  const int K1g = round_up(round_up(mp.c_in, 16), 64);
  const int Kh = C < 64 ? 64 : C;
  if (ws_bytes < debug_mlp_workspace_bytes(G, mp.c_in, C, mp.depth, N)) return fail(FGNN_ERR_WORKSPACE, "debug workspace too small");
  FGNN_CHECK_ARG(mp.c_in <= 128, "c_in too large for the debug entry");
  Arena ar(ws, ws_bytes);
  T* xin = ar.take<T>((size_t)G * mp.c_in * geo.stride(kLayoutC), 1024);
  T* out = ar.take<T>((size_t)G * C * geo.stride(kLayoutC), 1024);
  T* wf = ar.take<T>((size_t)G * C * K1g, 1024);
  T* wh = ar.take<T>((size_t)std::max(mp.depth - 1, 1) * C * Kh, 1024);
  float* bf = ar.take<float>((size_t)G * C);
  T* bt = ar.take<T>((size_t)G * C * 16, 1024);
  float* coef = ar.take<float>((size_t)G * C * 2);
  double* acc = ar.take<double>((size_t)G * C * 2);
  to_planes_c_kernel<T><<<dim3((unsigned)std::min(N, 256), G * mp.c_in), 256, 0, st>>>(x, xin, mp.c_in, geo, npg);
  FGNN_LAUNCHED();
  ConvertBatch cb{};
  cb.rows = cb.cols = C;
  for (int l = 1; l < mp.depth; ++l) { cb.src[l - 1] = mp.w[l]; cb.dst_off[l - 1] = (long)(l - 1) * C * Kh; }
  if (mp.depth > 1) {
    convert_weights_batch_kernel<T><<<dim3(ceil_div(C * Kh, 256), mp.depth - 1), 256, 0, st>>>(cb, wh, C, Kh);
    FGNN_LAUNCHED();
  }
  MlpGroup<T> M{};
  M.nmlp = 1;
  M.mlp[0] = chain(mp);
  M.src[0] = Src<T>{xin, mp.c_in, mp.c_in, nullptr}; M.nsrc = 1;
  M.wf = wf; M.bf = bf; M.bt = bt; M.wh = wh;
  M.out[0] = out; M.out_mode[0] = kLayoutC; M.ones[0] = 0; M.coef[0] = coef;
  M.stat_acc = acc;
  if (int e = run_mlp_group<T>(M, C, G, geo, npg, st)) return e;
  dim3 grid((unsigned)std::min<long>(64, (geo.PSC + 255) / 256), G * C);
  from_planes_kernel<T><<<grid, 256, 0, st>>>(out, y, coef, C, geo, npg);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

int debug_mlp(int precision, const fgnn_mlp_params& mp, const float* x, float* y, int G, int N,
              const int32_t* n_per_graph, void* ws, size_t ws_bytes, cudaStream_t st) {
  return with_16bit(precision, "fgnn_debug_tc_mlp", [&](auto t) -> int {
    FGNN_CHECK_ARG(x && y && ws, "null pointer");
    FGNN_CHECK_ARG(N <= kMaxN, "tensor-core MLP supports N <= %d (got %d)", kMaxN, N);
    if (mp.c_out != 32 && mp.c_out != 64) return fail(FGNN_ERR_UNSUPPORTED, "c_out must be 32 or 64");
    return debug_mlp_t<decltype(t)>(mp, x, y, G, N, n_per_graph, ws, ws_bytes, st);
  });
}

}  // namespace tc
}  // namespace fgnn
