// Batched linear assignment on the device: accuracy_linear_assignment of the reference
// (toolbox/metrics.py:92-116) without the per-graph device->host copy and the host Hungarian.
//
// The reference minimises cost = -log_softmax(scores) with scipy.optimize.linear_sum_assignment.  The kernel forms
// the log-softmax weights in fp32 as torch does ((x - rowmax) - log(sum exp(x - rowmax)), on the fly from two
// per-row constants in shared memory) and runs the algorithm scipy implements --
// shortest augmenting paths with dual variables (Jonker-Volgenant as restated by Crouse 2016) -- in double
// precision with scipy's own operation order (r = minVal + cost - u[i] - v[j]) and scipy's own tie rule, so the
// matching is the one scipy returns even when the optimum is not unique (an untrained network on a graph with
// automorphisms produces exact ties).  scipy scans the list `remaining` (initially the columns in DESCENDING order,
// compacted by swap-with-last) and keeps, among the columns of lowest path cost, the LAST unassigned one of the
// list, else the FIRST assigned one; the kernel keeps the same list in shared memory and reduces over list
// POSITIONS with that preference.  One CTA per graph: the scan of every Dijkstra step is spread over the CTA's
// threads and closed by a block-wide arg-min; duals, path and matching arrays live in shared memory: 53 bytes per
// column (smem_bytes), so the solver's column count M = max(N1, N2) is limited by the device's opt-in shared memory per
// block -- M <= 4380 with the 227 KB of an sm_100 device, 217 104 bytes at M = 4096.  Indices into the (G,N1,N2) scores
// are 64-bit; the rest are column / row numbers < M.
// Rectangular problems (graph 1 with n1 rows, graph 2 with n2 columns) are solved as scipy's rectangular_lsap solves
// them: as they are when n1 <= n2, transposed when n1 > n2 (solver rows = graph-2 vertices), with the cost of each entry
// always formed from its ORIGINAL row's log-softmax constants.  Rows left without a column get -1.
#include "fgnn_common.cuh"

#include <cfloat>

namespace fgnn {
namespace lap {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;

struct Best {
  double val;
  int idx;     // POSITION in the list `remaining`
  int free_;   // 1 if the column at that position is unassigned
};

// scipy's scan keeps `it` when spc < lowest || (spc == lowest && the column is unassigned): among the positions of
// lowest cost the winner is the last unassigned one, else the first (assigned) one
__device__ __forceinline__ bool better(const Best& a, const Best& b) {   // is a strictly better than b
  if (a.val != b.val) return a.val < b.val;
  if (a.free_ != b.free_) return a.free_ > b.free_;
  return a.free_ ? a.idx > b.idx : a.idx < b.idx;
}

__global__ void __launch_bounds__(kThreads)
lap_kernel(const float* __restrict__ scores, int32_t* __restrict__ col_of_row, int32_t* __restrict__ correct,
           double* __restrict__ total_cost, int N1, int N2, const int32_t* __restrict__ n1p, const int32_t* __restrict__ n2p) {
  extern __shared__ __align__(16) unsigned char lap_smem[];
  const int g = blockIdx.x;
  const int n1 = n1p ? n1p[g] : N1, n2 = n2p ? n2p[g] : N2;
  const bool tr = n1 > n2;                              // solve the transposed problem
  const int nr = tr ? n2 : n1, nc = tr ? n1 : n2;       // solver rows <= solver columns
  const int N = max(N1, N2);                            // capacity of every shared array
  double* u = reinterpret_cast<double*>(lap_smem);      // row duals
  double* v = u + N;                                    // column duals
  double* spc = v + N;                                  // shortest path cost to each column
  int* path = reinterpret_cast<int*>(spc + N);          // predecessor row of each column
  int* col4row = path + N;
  int* row4col = col4row + N;
  int* vis = row4col + N;                               // rows visited by the current search (SR)
  int* remaining = vis + N;                             // scipy's list of columns not yet scanned by the current search
  unsigned char* sc = reinterpret_cast<unsigned char*>(remaining + N);   // columns scanned by the current search (SC)
  float* rmx = reinterpret_cast<float*>(lap_smem + (((size_t)N * (3 * sizeof(double) + 5 * sizeof(int) + 1) + 15) / 16 * 16));
  float* rlg = rmx + N;                                 // log_softmax(x)[i][j] = (x - rmx[i]) - rlg[i]
  __shared__ Best s_best[kWarps];
  __shared__ Best s_pick;
  const int tid = threadIdx.x, lane = tid % 32, warp = tid / 32;
  const float* S = scores + (long)g * N1 * N2;
  // weight of solver entry (i, j): log_softmax of the original row, fp32 as torch forms it
  auto weight = [&](int i, int j) -> float {
    const int r = tr ? j : i, c = tr ? i : j;
    return (S[(long)r * N2 + c] - rmx[r]) - rlg[r];
  };

  for (int k = tid; k < N; k += kThreads) {
    u[k] = 0.0;
    v[k] = 0.0;
    col4row[k] = -1;
    row4col[k] = -1;
  }
  for (int r = warp; r < n1; r += kWarps) {              // row constants of the log-softmax over the valid columns
    const float* row = S + (long)r * N2;
    float mx = -INFINITY;
    for (int j = lane; j < n2; j += 32) mx = fmaxf(mx, row[j]);
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
    for (int j = lane; j < n2; j += 32) sum += expf(row[j] - mx);
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) { rmx[r] = mx; rlg[r] = logf(sum); }
  }
  __syncthreads();

  for (int cur = 0; cur < nr; ++cur) {
    for (int j = tid; j < nc; j += kThreads) {
      spc[j] = INFINITY;
      sc[j] = 0;
      remaining[j] = nc - j - 1;
    }
    __syncthreads();
    double min_val = 0.0;
    int i = cur, sink = -1, nvis = 0, num_remaining = nc;
    while (sink < 0) {
      if (tid == 0) vis[nvis] = i;
      ++nvis;
      const double ui = u[i];
      Best b{INFINITY, 0x7fffffff, 0};
      for (int it = tid; it < num_remaining; it += kThreads) {
        const int j = remaining[it];
        const double r = min_val + (-(double)weight(i, j)) - ui - v[j];   // cost = -weight, scipy's operation order
        double cur_cost = spc[j];
        if (r < cur_cost) {
          spc[j] = r;
          path[j] = i;
          cur_cost = r;
        }
        Best c{cur_cost, it, row4col[j] < 0 ? 1 : 0};
        if (b.idx == 0x7fffffff || better(c, b)) b = c;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        Best c;
        c.val = __shfl_xor_sync(0xffffffffu, b.val, o);
        c.idx = __shfl_xor_sync(0xffffffffu, b.idx, o);
        c.free_ = __shfl_xor_sync(0xffffffffu, b.free_, o);
        if (c.idx != 0x7fffffff && (b.idx == 0x7fffffff || better(c, b))) b = c;
      }
      if (lane == 0) s_best[warp] = b;
      __syncthreads();
      if (tid == 0) {
        Best p = s_best[0];
        for (int w = 1; w < kWarps; ++w)
          if (s_best[w].idx != 0x7fffffff && (p.idx == 0x7fffffff || better(s_best[w], p))) p = s_best[w];
        const int j = remaining[p.idx];
        remaining[p.idx] = remaining[num_remaining - 1];   // scipy: remaining[index] = remaining[--num_remaining]
        p.idx = j;                                         // publish the COLUMN
        s_pick = p;
        sc[j] = 1;
      }
      __syncthreads();
      const Best p = s_pick;
      --num_remaining;
      min_val = p.val;
      if (p.free_) sink = p.idx;
      else i = row4col[p.idx];
    }
    // dual update (Crouse 2016, step 4) and augmentation along the path
    for (int k = tid; k < nvis; k += kThreads) {
      const int r = vis[k];
      if (r == cur) u[r] += min_val;
      else u[r] += min_val - spc[col4row[r]];
    }
    for (int j = tid; j < nc; j += kThreads)
      if (sc[j]) v[j] -= min_val - spc[j];
    __syncthreads();
    if (tid == 0) {
      int j = sink;
      while (true) {
        const int r = path[j];
        row4col[j] = r;
        const int prev = col4row[r];
        col4row[r] = j;
        j = prev;
        if (r == cur) break;
      }
    }
    __syncthreads();
  }

  // outputs: matching, #fixed points (the identity is the ground truth, metrics.py:103), optimal cost
  int hits = 0;
  double cost = 0.0;
  for (int r = tid; r < N1; r += kThreads) {            // r: an original row; transposed, its column is row4col[r]
    const int c = r < n1 ? (tr ? row4col[r] : col4row[r]) : -1;
    if (col_of_row) col_of_row[(long)g * N1 + r] = c;
    if (c >= 0) {
      hits += (c == r);
      cost -= (double)((S[(long)r * N2 + c] - rmx[r]) - rlg[r]);
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    hits += __shfl_xor_sync(0xffffffffu, hits, o);
    cost += __shfl_xor_sync(0xffffffffu, cost, o);
  }
  __shared__ int s_hits[kWarps];
  __shared__ double s_cost[kWarps];
  if (lane == 0) { s_hits[warp] = hits; s_cost[warp] = cost; }
  __syncthreads();
  if (tid == 0) {
    int h = 0;
    double c = 0.0;
    for (int w = 0; w < kWarps; ++w) { h += s_hits[w]; c += s_cost[w]; }
    correct[g] = h;
    if (total_cost) total_cost[g] = c;
  }
}

inline size_t smem_bytes(int N) { return align_up((size_t)N * (3 * sizeof(double) + 5 * sizeof(int) + 1), 16) + (size_t)N * 2 * sizeof(float) + 16; }

// largest N whose dynamic shared memory fits next to the kernel's static shared memory in `limit` bytes
int max_n(size_t limit) {
  int lo = 0, hi = 1 << 16;
  while (lo < hi) {
    const int mid = (lo + hi + 1) / 2;
    if (smem_bytes(mid) <= limit) lo = mid; else hi = mid - 1;
  }
  return lo;
}

}  // namespace

int lap_fwd(const float* scores, int32_t* col_of_row, int32_t* correct, double* total_cost, int G, int N1, int N2,
            const int32_t* n1, const int32_t* n2, cudaStream_t st) {
  FGNN_CHECK_ARG(scores && correct, "null pointer");
  FGNN_CHECK_ARG(G >= 1 && N1 >= 1 && N2 >= 1, "bad sizes G=%d N1=%d N2=%d", G, N1, N2);
  const int N = std::max(N1, N2);
  const size_t smem = smem_bytes(N);
  int dev = 0, optin = 0;
  FGNN_CUDA(cudaGetDevice(&dev));
  FGNN_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  cudaFuncAttributes fa;
  FGNN_CUDA(cudaFuncGetAttributes(&fa, lap_kernel));
  const size_t limit = (size_t)optin > fa.sharedSizeBytes ? (size_t)optin - fa.sharedSizeBytes : 0;
  if (smem > limit)
    return fail(FGNN_ERR_UNSUPPORTED, "linear assignment supports N <= %d, N = max(N1, N2), on this device (%d bytes of shared "
                "memory per block; got N1=%d N2=%d)", max_n(limit), optin, N1, N2);
  FGNN_CUDA(cudaFuncSetAttribute(lap_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  lap_kernel<<<G, kThreads, smem, st>>>(scores, col_of_row, correct, total_cost, N1, N2, n1, n2);
  FGNN_LAUNCHED();
  return FGNN_OK;
}

}  // namespace lap
}  // namespace fgnn
