// fp32 backward of MlpBlock_Real (conv chain + GraphNorm), FGNN_FP32 training path.
//
// Nothing but the block input x and the GraphNorm statistics is kept from the forward pass: hidden
// activations are recomputed layer by layer, then the chain is differentiated layer by layer
// (backward-data = 1x1 conv with the transposed weight, backward-weight = a reduction GEMM over
// pixels).  Work is chunked over graphs so the scratch stays bounded.  GraphNorm backward follows
//   dz = w s [ g - mean(g) - (z - mu) mean(g (z - mu)) / (var + eps) ],  s = 1 / (2 sqrt(n (var + eps)))
// (derived from layers.py:68-80; checked against torch autograd in tests/test_gpu_f32.py).
#include "fgnn_f32.cuh"
#include <algorithm>

namespace fgnn {
namespace f32 {

namespace {

__device__ __forceinline__ int graph_n(const int32_t* n_per_graph, int g, int N) {
  return n_per_graph ? n_per_graph[g] : N;
}

// per plane (g,c): a1 = sum dy, a2 = sum dy (z - mu) over valid pixels; dgw += inv * a2, dgb += a1
// (OrderedSum: the two terms go to rec[0][gc] / rec[1][gc] instead, rec = dgw, and the caller sums them over g)
template <typename Sum>
__global__ void __launch_bounds__(256)
gn_bwd_stats_kernel(const float* __restrict__ dy, const float* __restrict__ z, const float* __restrict__ stats,
                    float* __restrict__ sums, float* __restrict__ dgw, float* __restrict__ dgb, int C, int N,
                    const int32_t* __restrict__ n_per_graph) {
  const int gc = blockIdx.x;
  const int g = gc / C, c = gc % C;
  const int n = graph_n(n_per_graph, g, N);
  const float mu = stats[2 * gc], inv = stats[2 * gc + 1];
  const float* dp = dy + (long)gc * N * N;
  const float* zp = z + (long)gc * N * N;
  double a1 = 0.0, a2 = 0.0;
  for (long q = threadIdx.x; q < (long)n * n; q += blockDim.x) {
    int i = (int)(q / n), j = (int)(q % n);
    double d = dp[(long)i * N + j];
    a1 += d;
    a2 += d * ((double)zp[(long)i * N + j] - (double)mu);
  }
  __shared__ double sh[2][256];
  sh[0][threadIdx.x] = a1;
  sh[1][threadIdx.x] = a2;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      sh[0][threadIdx.x] += sh[0][threadIdx.x + o];
      sh[1][threadIdx.x] += sh[1][threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    sums[2 * gc] = (float)sh[0][0];
    sums[2 * gc + 1] = (float)sh[1][0];
    if constexpr (Sum::kOrdered) {
      dgw[gc] = (float)(sh[1][0] * (double)inv);
      dgw[(long)gridDim.x + gc] = (float)sh[0][0];
    } else {
      if (dgw) atomicAdd(dgw + c, (float)(sh[1][0] * (double)inv));
      if (dgb) atomicAdd(dgb + c, (float)sh[0][0]);
    }
  }
}

// dz = gw * inv * (dy - a1/cnt - (z - mu) * (a2/cnt) * 4 n inv^2) on valid pixels, 0 elsewhere (in place on dy ok)
__global__ void gn_bwd_apply_kernel(const float* __restrict__ dy, const float* __restrict__ z,
                                    const float* __restrict__ stats, const float* __restrict__ sums,
                                    const float* __restrict__ gw, float* __restrict__ dz, int C, int N,
                                    const int32_t* __restrict__ n_per_graph, int constant_n) {
  const int gc = blockIdx.y;
  const int g = gc / C, c = gc % C;
  const int n = graph_n(n_per_graph, g, N);
  const long P = (long)N * N;
  const float mu = stats[2 * gc], inv = stats[2 * gc + 1];
  const float cnt = (float)n * (float)n;
  const float m1 = sums[2 * gc] / cnt;
  const float m2 = sums[2 * gc + 1] / cnt * 4.f * (float)(constant_n ? N : n) * inv * inv;   // mean(g (z-mu)) / (var + eps)
  const float w = (gw ? gw[c] : 1.f) * inv;
  for (long p = (long)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += (long)gridDim.x * blockDim.x) {
    int i = (int)(p / N), j = (int)(p % N);
    float v = 0.f;
    if (i < n && j < n) v = w * (dy[(long)gc * P + p] - m1 - (z[(long)gc * P + p] - mu) * m2);
    dz[(long)gc * P + p] = v;
  }
}

// d *= (h > 0)   (ReLU backward with the recomputed post-activation h)
__global__ void relu_mask_kernel(float* __restrict__ d, const float* __restrict__ h, long total) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x)
    if (!(h[i] > 0.f)) d[i] = 0.f;
}

// dW[co][ci] += sum_{g,p} d[g,co,p] in[g,ci,p];  db[co] += sum_{g,p} d[g,co,p]
// grid: (ci tiles of 16, co tiles of 16, pixel splits); block 16x16; K chunk 64 pixels staged in smem.
// OrderedSum: split z stores its partials to dW[z][co][ci] / db[z][co] (records) and the caller sums them over z.
template <typename Sum>
__global__ void __launch_bounds__(256)
wgrad_kernel(const float* __restrict__ d, const float* __restrict__ in, float* __restrict__ dW, float* __restrict__ db,
             int Co, int Ci, long P, int G) {
  __shared__ float sd[16][65], si[16][65];
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  const int co0 = blockIdx.y * 16, ci0 = blockIdx.x * 16;
  const long total = (long)G * P;
  const long chunk = (total + gridDim.z - 1) / gridDim.z;
  const long k_begin = (long)blockIdx.z * chunk;
  const long k_end = min(total, k_begin + chunk);
  float acc = 0.f, bacc = 0.f;
  for (long k0 = k_begin; k0 < k_end; k0 += 64) {
    for (int e = threadIdx.x; e < 16 * 64; e += 256) {
      int r = e / 64, q = e % 64;
      long k = k0 + q;
      float vd = 0.f, vi = 0.f;
      if (k < k_end) {
        long g = k / P, p = k % P;
        if (co0 + r < Co) vd = d[(g * Co + co0 + r) * P + p];
        if (ci0 + r < Ci) vi = in[(g * Ci + ci0 + r) * P + p];
      }
      sd[r][q] = vd;
      si[r][q] = vi;
    }
    __syncthreads();
#pragma unroll 16
    for (int q = 0; q < 64; ++q) {
      acc = fmaf(sd[ty][q], si[tx][q], acc);
      if (tx == 0) bacc += sd[ty][q];
    }
    __syncthreads();
  }
  if constexpr (Sum::kOrdered) {
    if (co0 + ty < Co && ci0 + tx < Ci) dW[((long)blockIdx.z * Co + co0 + ty) * Ci + ci0 + tx] = acc;
    if (db && blockIdx.x == 0 && tx == 0 && co0 + ty < Co) db[(long)blockIdx.z * Co + co0 + ty] = bacc;
  } else {
    if (co0 + ty < Co && ci0 + tx < Ci) atomicAdd(dW + (long)(co0 + ty) * Ci + ci0 + tx, acc);
    if (db && blockIdx.x == 0 && tx == 0 && co0 + ty < Co) atomicAdd(db + co0 + ty, bacc);
  }
}

}  // namespace

int mlp_bwd(const fgnn_mlp_params& p, const fgnn_mlp_grads& gr, const float* x, const float* stats,
            const float* dy, float* dx, int G, int N, const int32_t* n_per_graph, void* ws, size_t ws_bytes,
            cudaStream_t st, bool det) {
  FGNN_CHECK_ARG(x && stats && dy && ws, "null pointer");
  FGNN_CHECK_ARG(p.depth >= 1 && p.depth <= FGNN_MAX_DEPTH, "depth %d out of range", p.depth);
  const int Co = p.c_out, Ci = p.c_in, depth = p.depth;
  const long P = (long)N * N;
  const int cmax = Co > Ci ? Co : Ci;
  // scratch: weight repack + (depth + 2) activation tensors for one chunk of graphs
  Arena ar(ws, ws_bytes);
  float* wt = ar.take<float>((size_t)(Ci > Co ? Ci : Co) * ((cmax + 7) / 8 * 8));
  float* sums = ar.take<float>((size_t)G * Co * 2);
  const MlpBwdRecords rec = det ? mlp_bwd_records(ar, G, Co, cmax) : MlpBwdRecords{};
  const size_t fixed = align_up(ar.off, 256);
  if (fixed >= ws_bytes) return fail(FGNN_ERR_WORKSPACE, "mlp backward workspace too small");
  const size_t per_graph = (size_t)(depth + 2) * cmax * P * sizeof(float) + 256 * (depth + 2);
  long chunk = (long)((ws_bytes - fixed) / per_graph);
  if (chunk < 1) return fail(FGNN_ERR_WORKSPACE, "mlp backward workspace too small for one graph (%zu bytes needed)", fixed + per_graph);
  if (chunk > G) chunk = G;
  float* h[FGNN_MAX_DEPTH];   // h[k]: output of layer k (post-ReLU for k < depth-1, pre-norm z for the last)
  for (int k = 0; k < depth; ++k) h[k] = ar.take<float>((size_t)chunk * cmax * P);
  float* dcur = ar.take<float>((size_t)chunk * cmax * P);
  float* dnxt = ar.take<float>((size_t)chunk * cmax * P);
  if (!ar.ok()) return fail(FGNN_ERR_WORKSPACE, "mlp backward workspace too small");

  for (int g0 = 0; g0 < G; g0 += (int)chunk) {
    const int gc = (int)std::min<long>(chunk, G - g0);
    const int32_t* n_c = n_per_graph ? n_per_graph + g0 : nullptr;
    const float* xc = x + (long)g0 * Ci * P;
    const float* dyc = dy + (long)g0 * Co * P;
    const float* stc = stats + (long)g0 * Co * 2;
    float* smc = sums + (long)g0 * Co * 2;
    // 1. recompute the chain, keeping every layer's output
    for (int k = 0; k < depth; ++k) {
      const float* in = (k == 0) ? xc : h[k - 1];
      if (int e = run_conv1x1(p.w[k], p.b[k], k == 0 ? Ci : Co, Co, false, k < depth - 1, in, h[k], wt, gc, N, n_c, st))
        return e;
    }
    // 2. GraphNorm backward -> dz
    if (det) {
      // records [2][gc * Co], then dgw[c] / dgb[c] += their sum over the chunk's graphs in ascending order
      gn_bwd_stats_kernel<OrderedSum><<<gc * Co, 256, 0, st>>>(dyc, h[depth - 1], stc, smc, rec.gn, nullptr, Co, N, n_c);
      FGNN_LAUNCHED();
      if (gr.gn_w) if (int e = sum_records(rec.gn, gr.gn_w, Co, gc, Co, true, st)) return e;
      if (gr.gn_b) if (int e = sum_records(rec.gn + (long)gc * Co, gr.gn_b, Co, gc, Co, true, st)) return e;
    } else {
      gn_bwd_stats_kernel<AtomicSum><<<gc * Co, 256, 0, st>>>(dyc, h[depth - 1], stc, smc, gr.gn_w, gr.gn_b, Co, N, n_c);
      FGNN_LAUNCHED();
    }
    {
      dim3 grid((unsigned)std::min<long>(64, (P + 255) / 256), gc * Co);
      gn_bwd_apply_kernel<<<grid, 256, 0, st>>>(dyc, h[depth - 1], stc, smc, p.gn_w, dcur, Co, N, n_c, p.constant_n);
      FGNN_LAUNCHED();
    }
    // 3. layers in reverse
    for (int k = depth - 1; k >= 0; --k) {
      const int cin = (k == 0) ? Ci : Co;
      const float* in = (k == 0) ? xc : h[k - 1];
      if (gr.w[k]) {
        const int splits = (int)std::min<long>(kMaxWgradSplits, std::max<long>(1, (long)gc * P / 4096));
        dim3 grid(ceil_div(cin, 16), ceil_div(Co, 16), splits);
        if (det) {
          wgrad_kernel<OrderedSum><<<grid, 256, 0, st>>>(dcur, in, rec.w, gr.b[k] ? rec.b : nullptr, Co, cin, P, gc);
          FGNN_LAUNCHED();
          if (int e = sum_records(rec.w, gr.w[k], (long)Co * cin, splits, Co * cin, true, st)) return e;
          if (gr.b[k]) if (int e = sum_records(rec.b, gr.b[k], Co, splits, Co, true, st)) return e;
        } else {
          wgrad_kernel<AtomicSum><<<grid, 256, 0, st>>>(dcur, in, gr.w[k], gr.b[k], Co, cin, P, gc);
          FGNN_LAUNCHED();
        }
      }
      if (k == 0 && dx == nullptr) break;
      float* dst = (k == 0) ? dx + (long)g0 * Ci * P : dnxt;
      // backward-data: d_in[ci] = sum_co W[co][ci] d[co]  == 1x1 conv with w^T; w (Co, cin) is "(c_in'=Co rows, c_out'=cin cols)"
      if (int e = run_conv1x1(p.w[k], nullptr, Co, cin, true, false, dcur, dst, wt, gc, N, n_c, st)) return e;
      if (k > 0) {
        const long total = (long)gc * Co * P;
        relu_mask_kernel<<<(unsigned)std::min<long>(148 * 8, (total + 255) / 256), 256, 0, st>>>(dnxt, h[k - 1], total);
        FGNN_LAUNCHED();
        std::swap(dcur, dnxt);
      }
    }
  }
  return FGNN_OK;
}

}  // namespace f32
}  // namespace fgnn
