// 16-bit TRAINING path of the tensor-core embedder: forward that keeps what backward needs, and the backward of the
// whole block stack with every contraction on tcgen05 (included by fgnn_tc.cu inside namespace fgnn::tc::<anon>).
//
// The reference trains through autograd of models/layers.py:126-131,161-162 under Lightning's precision=16
// (commander_explore.py:120-123, models/trainers.py:70-76).  Here:
//   forward  every 1x1 conv is its own depth-1 launch of tc_mlp_kernel (hidden layers with the RELU_OUT epilogue), so the
//            hidden activations h_l exist as 16-bit planes; z (pre-GraphNorm), Y1/Y2/mult and the GraphNorm statistics
//            are kept as in inference.  ColumnMaxPooling keeps its arg-max.
//   backward GraphNorm in closed form from two plane reductions (sum dy, sum dy z):
//                dz = a dy + beta z + gamma,  beta = -a m2, gamma = -a m1 + a m2 mu,
//                m1 = mean(dy), m2 = mean(dy (z - mu)) / (var + eps)                      (layers.py:68-80)
//            data gradients of the convs   = depth-1 launches of tc_mlp_kernel with transposed weights,
//            weight gradients of the convs = tc_wgrad_kernel (pixel-reduction GEMM, K = pixels, split over CTAs),
//            matmul gradients              = tc_bmm_bwd_kernel: dY1 = dM Y2^T, dY2 = Y1^T dM with the GraphNorm
//                                            scale / shift of the other operand applied in the epilogue,
//            ReLU masks, the pooling scatter and the small per-(graph, channel) algebra on CUDA cores.
//   16-bit gradients are scaled by a power of two chosen from max |d emb| (fp16 range); parameter gradients are
//   accumulated in fp32 and un-scaled when they are added to the caller's buffers.
//
// First-layer weights see the NORMALISED input y = a u + s through the per-graph fold W diag(a), b + W s, so
//   dW0 = sum_g ( P_g diag(a_g) + (sum_px g0) s_g^T ),  P_g = sum_px g0 u^T  (per-graph pixel GEMM),  db0 = sum g0,
// and the data gradient W0^T g0 is the gradient with respect to y, i.e. the "dy" of the producing MLP.

template <typename T>
__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
  const float2 a = Elem<T>::unpack2(v.x), b = Elem<T>::unpack2(v.y), c = Elem<T>::unpack2(v.z), d = Elem<T>::unpack2(v.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
template <typename T>
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  return make_uint4(Elem<T>::pack(f[0], f[1]), Elem<T>::pack(f[2], f[3]), Elem<T>::pack(f[4], f[5]), Elem<T>::pack(f[6], f[7]));
}
// validity mask (bit e) of the 8 physical columns pj0 .. pj0+7 of a row i < n
__device__ __forceinline__ uint32_t valid8(int pj0, int n, const Geo& geo) {
  uint32_t m = 0;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int pj = pj0 + e;
    const bool hole = (pj & (geo.BN - 1)) == geo.BN - 1;
    const int j = pj - (pj >> geo.BNLOG);
    if (!hole && j < n) m |= 1u << e;
  }
  return m;
}

// bias-gradient partial of CTA (x, gc): added to bsum[gc] (AtomicSum) or stored to bsum[gc][x] (OrderedSum records)
template <typename Sum>
__device__ __forceinline__ void add_bsum(float* bsum, int gc, float t) {
  if constexpr (Sum::kOrdered) bsum[(long)gc * gridDim.x + blockIdx.x] = t;
  else atomicAdd(bsum + gc, t);
}

__device__ __forceinline__ float block_sum(float v, float* s_red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  __syncthreads();
  if (lane == 0) s_red[warp] = v;
  __syncthreads();
  float t = 0.f;
  if (warp == 0) {
    t = lane < (int)(blockDim.x / 32) ? s_red[lane] : 0.f;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  }
  return t;   // valid in warp 0
}

// acc[gc] += (sum dy, sum dy z) over the valid n x n block; dy = dya (+ dyb), layout C; z in layout zmode.
// OrderedSum: CTA (x, gc) stores its pair to acc[gc][x] (records, reduced by the caller).
template <typename T, typename Sum>
__global__ void __launch_bounds__(256)
gn_bwd_stats_kernel(const T* __restrict__ dya, const T* __restrict__ dyb, const T* __restrict__ z, Layout zmode,
                    double* __restrict__ acc, int C, Geo geo, const int32_t* __restrict__ npg) {
  __shared__ float s_red[8];
  const int gc = blockIdx.y, g = gc / C;
  const int n = graph_n(npg, g, geo.N);
  const int ch = geo.NPC / 8;
  const long PSz = geo.stride(zmode);
  const int pj_end = phys_k_end(n, geo.TN1);
  float s1 = 0.f, s2 = 0.f;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < (long)n * ch; idx += (long)gridDim.x * blockDim.x) {
    const int i = (int)(idx / ch), pj0 = (int)(idx % ch) * 8;
    if (pj0 >= pj_end) continue;
    const uint32_t vm = valid8(pj0, n, geo);
    const long oc = (long)gc * geo.PSC + (long)i * geo.NPC + pj0;
    float d[8], zz[8];
    unpack8<T>(*reinterpret_cast<const uint4*>(dya + oc), d);
    if (dyb) {
      float d2[8];
      unpack8<T>(*reinterpret_cast<const uint4*>(dyb + oc), d2);
#pragma unroll
      for (int e = 0; e < 8; ++e) d[e] += d2[e];
    }
    unpack8<T>(*reinterpret_cast<const uint4*>(z + (long)gc * PSz + (long)geo.phys_row(i, zmode) * geo.NPC + pj0), zz);
#pragma unroll
    for (int e = 0; e < 8; ++e)
      if (vm & (1u << e)) { s1 += d[e]; s2 = fmaf(d[e], zz[e], s2); }
  }
  const float t1 = block_sum(s1, s_red);
  const float t2 = block_sum(s2, s_red);
  if (threadIdx.x == 0) {
    if constexpr (Sum::kOrdered) {
      double* r = acc + 2 * ((long)gc * gridDim.x + blockIdx.x);
      r[0] = (double)t1;
      r[1] = (double)t2;
    } else {
      atomicAdd(acc + 2 * (long)gc, (double)t1);
      atomicAdd(acc + 2 * (long)gc + 1, (double)t2);
    }
  }
}

// bc[gc] = {a, beta, gamma, 0}
__global__ void gn_bwd_coef_kernel(const double* __restrict__ acc, const float* __restrict__ coef,
                                   const float* __restrict__ gnstat, float* __restrict__ bc, int C, int N,
                                   const int32_t* __restrict__ npg, int total) {
  const int gc = blockIdx.x * blockDim.x + threadIdx.x;
  if (gc >= total) return;
  const int n = graph_n(npg, gc / C, N);
  const double cnt = (double)n * n;
  const double S1 = acc[2 * (long)gc], S2 = acc[2 * (long)gc + 1];
  const double mu = gnstat[4 * (long)gc], ivar = gnstat[4 * (long)gc + 1];
  const double a = coef[2 * (long)gc];
  const double m1 = S1 / cnt, m2 = (S2 - mu * S1) / cnt * ivar;
  bc[4 * (long)gc] = (float)a;
  bc[4 * (long)gc + 1] = (float)(-a * m2);
  bc[4 * (long)gc + 2] = (float)(-a * m1 + a * m2 * mu);
  bc[4 * (long)gc + 3] = 0.f;
}

// d gn.weight[c] += inv * sum_g s0 (S2 - mu S1),  d gn.bias[c] += inv * sum_g S1     (layers.py:68-69), c < co_real
__global__ void gn_param_grad_kernel(const double* __restrict__ acc, const float* __restrict__ gnstat, float* dgw, float* dgb,
                                     const float* __restrict__ scale, int G, int C, int co_real) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= co_real) return;
  double sw = 0.0, sb = 0.0;
  for (int g = 0; g < G; ++g) {
    const long gc = (long)g * C + c;
    const double S1 = acc[2 * gc], S2 = acc[2 * gc + 1];
    sw += (double)gnstat[4 * gc + 2] * (S2 - (double)gnstat[4 * gc] * S1);
    sb += S1;
  }
  const double inv = 1.0 / (double)scale[0];
  if (dgw) dgw[c] += (float)(sw * inv);
  if (dgb) dgb[c] += (float)(sb * inv);
}

// dz = a dy + beta z + gamma on the valid block, 0 elsewhere (layout C out, covered rows only);
// bsum[gc] += sum of the ROUNDED dz (the last conv's bias gradient: zero up to rounding, as in the reference)
template <typename T, typename Sum>
__global__ void __launch_bounds__(256)
gn_bwd_apply_kernel(const T* __restrict__ dya, const T* __restrict__ dyb, const T* __restrict__ z, Layout zmode,
                    const float* __restrict__ bc, T* __restrict__ out, float* __restrict__ bsum, int C, Geo geo,
                    const int32_t* __restrict__ npg) {
  __shared__ float s_red[8];
  float ssum = 0.f;
  const int gc = blockIdx.y, g = gc / C;
  const int n = graph_n(npg, g, geo.N);
  const int rows = rows_cover(npg, g, geo);
  const int ch = geo.NPC / 8;
  const long PSz = geo.stride(zmode);
  const float a = bc[4 * (long)gc], be = bc[4 * (long)gc + 1], ga = bc[4 * (long)gc + 2];
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < (long)rows * ch; idx += (long)gridDim.x * blockDim.x) {
    const int i = (int)(idx / ch), pj0 = (int)(idx % ch) * 8;
    const long oc = (long)gc * geo.PSC + (long)i * geo.NPC + pj0;
    float r[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const uint32_t vm = i < n ? valid8(pj0, n, geo) : 0u;
    if (vm) {
      float d[8], zz[8];
      unpack8<T>(*reinterpret_cast<const uint4*>(dya + oc), d);
      if (dyb) {
        float d2[8];
        unpack8<T>(*reinterpret_cast<const uint4*>(dyb + oc), d2);
#pragma unroll
        for (int e = 0; e < 8; ++e) d[e] += d2[e];
      }
      unpack8<T>(*reinterpret_cast<const uint4*>(z + (long)gc * PSz + (long)geo.phys_row(i, zmode) * geo.NPC + pj0), zz);
#pragma unroll
      for (int e = 0; e < 8; ++e)
        if (vm & (1u << e)) r[e] = fmaf(a, d[e], fmaf(be, zz[e], ga));
    }
    const uint4 pk = pack8<T>(r);
    *reinterpret_cast<uint4*>(out + oc) = pk;
    if (vm) {
      float rr[8];
      unpack8<T>(pk, rr);
#pragma unroll
      for (int e = 0; e < 8; ++e) ssum += rr[e];
    }
  }
  const float t = block_sum(ssum, s_red);
  if (threadIdx.x == 0) add_bsum<Sum>(bsum, gc, t);
}

// ReLU backward in place: pre <- pre * [h > 0]; bsum[gc] += sum of the result (bias gradient of the layer below)
template <typename T, typename Sum>
__global__ void __launch_bounds__(256)
relu_mask_kernel(T* __restrict__ pre, const T* __restrict__ h, float* __restrict__ bsum, int C, Geo geo,
                 const int32_t* __restrict__ npg) {
  __shared__ float s_red[8];
  const int gc = blockIdx.y, g = gc / C;
  const int rows = rows_cover(npg, g, geo);
  const long tot = (long)rows * (geo.NPC / 8);
  float s = 0.f;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < tot; idx += (long)gridDim.x * blockDim.x) {
    const long oc = (long)gc * geo.PSC + idx * 8;
    float p[8], hh[8];
    unpack8<T>(*reinterpret_cast<const uint4*>(pre + oc), p);
    unpack8<T>(*reinterpret_cast<const uint4*>(h + oc), hh);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      p[e] = hh[e] > 0.f ? p[e] : 0.f;
      s += p[e];
    }
    *reinterpret_cast<uint4*>(pre + oc) = pack8<T>(p);
  }
  const float t = block_sum(s, s_red);
  if (threadIdx.x == 0) add_bsum<Sum>(bsum, gc, t);
}

// rowsum[gc][i] = sum_j x[i][j] (valid block), one warp per row
template <typename T>
__global__ void __launch_bounds__(256)
plane_rowsum_kernel(const T* __restrict__ x, float* __restrict__ rowsum, int C, Geo geo, const int32_t* __restrict__ npg) {
  const int gc = blockIdx.y, g = gc / C;
  const int n = graph_n(npg, g, geo.N);
  const int i = blockIdx.x * 8 + threadIdx.x / 32, lane = threadIdx.x % 32;
  if (i >= geo.N) return;
  float s = 0.f;
  if (i < n) {
    const int pj_end = phys_k_end(n, geo.TN1);
    for (int pj0 = lane * 8; pj0 < pj_end; pj0 += 256) {
      const uint32_t vm = valid8(pj0, n, geo);
      float p[8];
      unpack8<T>(*reinterpret_cast<const uint4*>(x + (long)gc * geo.PSC + (long)i * geo.NPC + pj0), p);
#pragma unroll
      for (int e = 0; e < 8; ++e)
        if (vm & (1u << e)) s += p[e];
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  }
  if (lane == 0) rowsum[(long)gc * geo.N + i] = s;
}

// colsum[gc][pj] = sum_i x[i][pj] (valid block; 0 at holes and beyond the graph), one thread per physical column
template <typename T>
__global__ void __launch_bounds__(256)
plane_colsum_kernel(const T* __restrict__ x, float* __restrict__ colsum, int C, Geo geo, const int32_t* __restrict__ npg) {
  const int gc = blockIdx.y, g = gc / C;
  const int n = graph_n(npg, g, geo.N);
  const int pj = blockIdx.x * blockDim.x + threadIdx.x;
  if (pj >= geo.NPC) return;
  const bool hole = (pj & (geo.BN - 1)) == geo.BN - 1;
  const int j = pj - (pj >> geo.BNLOG);
  float s = 0.f;
  if (!hole && j < n) {
    const T* col = x + (long)gc * geo.PSC + pj;
    for (int i = 0; i < n; ++i) s += Elem<T>::to_float(col[(long)i * geo.NPC]);
  }
  colsum[(long)gc * geo.NPC + pj] = s;
}

// ColumnMaxPooling of the training path: emb[g][c][i] = max_j (a z[i][j] + s), arg = physical column of the maximum
// (smallest column on ties); rows >= n -> 0 / -1.  One warp per row.  emb is (G, co_real, N), arg (G, C, N).
template <typename T>
__global__ void __launch_bounds__(256)
colmax16_kernel(const T* __restrict__ z, const float* __restrict__ coef, float* __restrict__ emb, int32_t* __restrict__ arg,
                int C, int co_real, Geo geo, const int32_t* __restrict__ npg) {
  const int gc = blockIdx.y, g = gc / C, c = gc % C;
  const int n = graph_n(npg, g, geo.N);
  const int i = blockIdx.x * 8 + threadIdx.x / 32, lane = threadIdx.x % 32;
  if (i >= geo.N) return;
  float best = -INFINITY;
  int bj = 0x7fffffff;
  const float a = coef[2 * (long)gc], sft = coef[2 * (long)gc + 1];
  const float sgn = a >= 0.f ? 1.f : -1.f;
  if (i < n) {
    const int pj_end = phys_k_end(n, geo.TN1);
    for (int pj0 = lane * 8; pj0 < pj_end; pj0 += 256) {
      const uint32_t vm = valid8(pj0, n, geo);
      float p[8];
      unpack8<T>(*reinterpret_cast<const uint4*>(z + (long)gc * geo.PSC + (long)i * geo.NPC + pj0), p);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float v = sgn * p[e];
        if ((vm & (1u << e)) && v > best) { best = v; bj = pj0 + e; }
      }
    }
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
      if (ov > best || (ov == best && oj < bj)) { best = ov; bj = oj; }
    }
  }
  if (lane == 0) {
    if (c < co_real) emb[((long)g * co_real + c) * geo.N + i] = i < n ? fmaf(a, sgn * best, sft) : 0.f;
    arg[(long)gc * geo.N + i] = (i < n && bj != 0x7fffffff) ? bj : -1;   // a row of NaNs has no arg-max: no gradient
  }
}

// loss scale of the 16-bit backward: the power of two that brings max |d emb| to [2^(t-1), 2^t), t = target_log2
__global__ void __launch_bounds__(1024)
grad_scale_kernel(const float* __restrict__ demb, long total, float* __restrict__ scale, int target_log2) {
  __shared__ float s_red[32];
  float m = 0.f;
  for (long i = threadIdx.x; i < total; i += blockDim.x) m = fmaxf(m, fabsf(demb[i]));
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (threadIdx.x % 32 == 0) s_red[threadIdx.x / 32] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 32; ++w) m = fmaxf(m, s_red[w]);
    float sc = 1.f;
    if (m > 0.f && isfinite(m)) {
      int e;
      frexpf(m, &e);                       // m = f * 2^e, f in [0.5, 1)
      int k = target_log2 - e;             // m * 2^k in [2^(t-1), 2^t)
      k = k < -24 ? -24 : (k > 40 ? 40 : k);
      sc = ldexpf(1.f, k);
    }
    scale[0] = sc;
  }
}

// dy of the last block's output: zero planes (memset by the caller) + scale * d emb at the pooling arg-max; demb is
// (G, co_real, N), the padded channels get no gradient
template <typename T>
__global__ void pool_scatter_kernel(const float* __restrict__ demb, const int32_t* __restrict__ arg, const float* __restrict__ scale,
                                    T* __restrict__ dy, int C, int co_real, Geo geo, long total) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int a = arg[idx];
  if (a < 0) return;
  const long gc = idx / geo.N;
  const int i = (int)(idx % geo.N);
  const int c = (int)(gc % C);
  if (c >= co_real) return;
  dy[gc * geo.PSC + (long)i * geo.NPC + a] = Elem<T>::from_float(scale[0] * demb[((gc / C) * co_real + c) * geo.N + i]);
}

// wt[r][dst_col0 + c] = w[c][col0 + r]   (r < rows, c < co): transposed (slices of) conv weights for the data gradients.
// w has its real shape (co_real, cin_total); the stored slice is zero beyond co_real columns and rows_real rows.
__global__ void transpose_slice_kernel(const float* __restrict__ w, float* __restrict__ wt, int co, int co_real, int cin_total,
                                       int col0, int rows, int rows_real, int dst_pitch, int dst_col0) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * co) return;
  const int r = idx / co, c = idx % co;
  wt[r * dst_pitch + dst_col0 + c] = c < co_real && r < rows_real ? w[c * cin_total + col0 + r] : 0.f;
}

// hidden-layer parameter gradients: dW[co][ci] += inv * P[co][ldp], db[co] += inv * sum_g bsum[g][co]; real (co, ci) out of
// the stored C channels of bsum
__global__ void wgrad_combine_hidden_kernel(const float* __restrict__ P, int ldp, const float* __restrict__ bsum, float* dW, float* db,
                                            const float* __restrict__ scale, int G, int C, int co, int ci) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const float inv = 1.f / scale[0];
  if (idx < co * ci) dW[idx] += inv * P[(idx / ci) * ldp + idx % ci];
  if (idx < co && db) {
    float s = 0.f;
    for (int g = 0; g < G; ++g) s += bsum[(long)g * C + idx];
    db[idx] += inv * s;
  }
}

// first-layer parameter gradients through the per-graph GraphNorm fold (see the header of this file):
//   dW[co][ci] += inv * sum_g ( P_g[co][k(ci)] a_src[g][ci] + bsum[g][co] s_src[g][ci] ),  db[co] += inv * sum_g bsum[g][co]
// for the real entries only: real column (s ? cr_0 : 0) + ch of dW is channel ch of source s, stored at k = koff_s + ch
struct CombineFirstArgs {
  const float* P;          // [G][co][ldp]
  const float* bsum;       // [G][co]
  const float* coef[2];    // per source [G][c_s][2] or null
  int c[2], cr[2], koff[2], nsrc;
  int G, co, co_real, ldp;
  float* dW;               // (co_real, cr0 + cr1)
  float* db;
  const float* scale;
};
__global__ void wgrad_combine_first_kernel(CombineFirstArgs a) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int cin = a.cr[0] + (a.nsrc > 1 ? a.cr[1] : 0);
  const float inv = 1.f / a.scale[0];
  if (idx < a.co_real * cin) {
    const int co = idx / cin, col = idx % cin;
    const int s = col < a.cr[0] ? 0 : 1;
    const int chn = col - (s ? a.cr[0] : 0);
    const int k = a.koff[s] + chn;
    float acc = 0.f;
    for (int g = 0; g < a.G; ++g) {
      const float av = a.coef[s] ? a.coef[s][((long)g * a.c[s] + chn) * 2] : 1.f;
      const float sv = a.coef[s] ? a.coef[s][((long)g * a.c[s] + chn) * 2 + 1] : 0.f;
      acc = fmaf(a.P[((long)g * a.co + co) * a.ldp + k], av, acc);
      acc = fmaf(a.bsum[(long)g * a.co + co], sv, acc);
    }
    a.dW[idx] += inv * acc;
  }
  if (idx < a.co_real && a.db) {
    float s = 0.f;
    for (int g = 0; g < a.G; ++g) s += a.bsum[(long)g * a.co + idx];
    a.db[idx] += inv * s;
  }
}

// =============================================================================================
// tc_wgrad_kernel: P[g][co][ci] (+)= sum_px A[g][co][px] * B[g][ci][px]  -- the weight gradient of a 1x1 conv.
//   A = output-gradient planes (layout C, co <= 128 channels), B = the layer's input planes (one or two sources,
//   Nw = padded channel count, multiple of 16, <= 128); both operands K-major (K = 64 pixels per stage, TMA boxes of
//   64 pixels x channels, rows beyond the channel count zero-filled by the tensor map), M = 128, N = Nw, fp32
//   accumulation in TMEM over the CTA's pixel range, atomicAdd of the accumulator tile at the end.
//   Work item = (graph, split of its pixel range); out_stride_g = 0 accumulates all graphs into one matrix.
//   OrderedSum: every item stores its tile to its own record out[item][co][Nw] (zeros for an empty pixel range) with
//   plain stores, and launch_wgrad sums the records in item order.
// Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer, warps 2-5 = epilogue.
// =============================================================================================
struct WgradArgs {
  int G, S;            // graphs, splits per graph
  int co, Nw, k0, nsrc;
  float* out;
  long out_stride_g;
  Geo geo;
  const int32_t* n_per_graph;
};
// A stage holds only the rows the tensor maps deliver: co_pad = round_up(co, 8) rows of A (the MMA still reads 128 rows:
// rows >= co_pad are whatever the ring holds, they only feed accumulator lanes nobody reads) and Nw rows of B.  With
// 32-channel layers a stage is 8 KB, and the ring is as deep as shared memory allows: the kernel is a pure
// streaming reduction and needs tens of KB in flight per SM.
constexpr int kWgMaxStages = 16;
constexpr size_t kWgRingBytes = 160 * 1024;
constexpr size_t kWgSmemBytes = kWgRingBytes + 128 * 128 + (2 * kWgMaxStages + 4) * 8 + 16;   // + slack the last stage's 128-row read may touch

template <typename T, typename Sum>
__global__ void __launch_bounds__(192, 1)
tc_wgrad_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b0,
                const __grid_constant__ CUtensorMap map_b1, const WgradArgs args) {
  extern __shared__ uint8_t smem_wg[];
  uint8_t* smem = smem_wg;
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kWgRingBytes + 128 * 128);
  uint64_t* full = bars;
  uint64_t* empty = bars + kWgMaxStages;
  uint64_t* tmem_full = bars + 2 * kWgMaxStages;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;         // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  const int warp = uniform_warp_idx(), lane = threadIdx.x % 32;
  const Geo geo = args.geo;
  const int Nw = args.Nw;
  const int co_pad = (args.co + 7) & ~7;
  const uint32_t stage_tx = (uint32_t)(co_pad + Nw) * 128u;
  const uint32_t stage_bytes = (stage_tx + 1023u) & ~1023u;
  const int kWgStages = min(kWgMaxStages, (int)(kWgRingBytes / stage_bytes));
  const int items = args.G * args.S;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kWgStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], 4); }
    fence_barrier_init();
  }
  // rows of a stage the tensor maps never write are read by the 128-row MMA: give them finite contents once
  for (uint32_t i = threadIdx.x; i < (uint32_t)((kWgRingBytes + 128 * 128) / 16); i += blockDim.x)
    reinterpret_cast<uint4*>(smem)[i] = make_uint4(0u, 0u, 0u, 0u);
  fence_proxy_async_smem();
  if (warp == 0) tmem_alloc(tmem_slot, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // pixel range of an item: 64-pixel steps [lo, hi) of the graph's covered rows
  auto item_range = [&](int item, int& g, int& lo, int& hi) {
    g = item / args.S;
    const int sp = item % args.S;
    const int steps = (int)(((long)rows_cover(args.n_per_graph, g, geo) * geo.NPC + 63) / 64);
    const int per = (steps + args.S - 1) / args.S;
    lo = sp * per;
    hi = min(steps, lo + per);
  };

  if (warp == 0) {
    if (lane == 0) { prefetch_tensormap(&map_a); prefetch_tensormap(&map_b0); }
    int stage = 0;
    uint32_t phase = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      int g, lo, hi;
      item_range(item, g, lo, hi);
      for (int st = lo; st < hi; ++st) {
        mbar_wait(&empty[stage], phase ^ 1);
        uint8_t* sa = smem + (size_t)stage * stage_bytes;
        uint8_t* sb = sa + (size_t)co_pad * 128;
        mbar_arrive_expect_tx_e(&full[stage], stage_tx);
        tma_load_3d_e(sa, &map_a, &full[stage], st * 64, 0, g);
        tma_load_3d_e(sb, &map_b0, &full[stage], st * 64, 0, g);
        if (args.nsrc > 1) tma_load_3d_e(sb + (size_t)args.k0 * 128, &map_b1, &full[stage], st * 64, 0, g);
        if (++stage == kWgStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = make_idesc(Elem<T>::kFmt, /*A K-major*/ 0, /*B K-major*/ 0, 128, Nw);
    const uint64_t a_d0 = smem_desc_sw128(smem_u32(smem), 16u, 1024u);
    const uint64_t b_d0 = smem_desc_sw128(smem_u32(smem) + (uint32_t)co_pad * 128u, 16u, 1024u);
    const uint32_t a_lo0 = (uint32_t)a_d0, a_hi = (uint32_t)(a_d0 >> 32);
    const uint32_t b_lo0 = (uint32_t)b_d0, b_hi = (uint32_t)(b_d0 >> 32);
    int stage = 0;
    uint32_t phase = 0;
    int as = 0;
    uint32_t aphase = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      int g, lo, hi;
      item_range(item, g, lo, hi);
      mbar_wait(&tmem_empty[as], aphase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(as * 128);
      for (int st = lo; st < hi; ++st) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        const uint32_t a_lo = a_lo0 + (uint32_t)stage * (stage_bytes >> 4);
        const uint32_t b_lo = b_lo0 + (uint32_t)stage * (stage_bytes >> 4);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          mma_ss2_e(d_tmem, a_lo + (uint32_t)k * (32u >> 4), a_hi, b_lo + (uint32_t)k * (32u >> 4), b_hi, idesc,
                    (st > lo || k > 0) ? 1u : 0u);
        mma_commit_e(&empty[stage]);
        if (++stage == kWgStages) { stage = 0; phase ^= 1; }
      }
      mma_commit_e(&tmem_full[as]);     // also for an empty range: the epilogue then adds nothing (see below)
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
  } else {
    const int quad = warp % 4;
    int as = 0;
    uint32_t aphase = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      int g, lo, hi;
      item_range(item, g, lo, hi);
      mbar_wait(&tmem_full[as], aphase);
      tc_fence_after();
      const int r = quad * 32 + lane;
      if constexpr (Sum::kOrdered) {
        if (quad * 32 < args.co) {                   // warp-uniform
          const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * 128);
          float4* dst = reinterpret_cast<float4*>(args.out + ((long)item * args.co + r) * Nw);
#pragma unroll 1
          for (int c0 = 0; c0 < Nw; c0 += 16) {
            uint32_t rr[16] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
            if (hi > lo) {                           // warp-uniform; an empty range leaves the accumulator unwritten
              tmem_ld16(taddr + (uint32_t)c0, rr);
              tmem_wait_ld();
            }
            if (r < args.co) {
#pragma unroll
              for (int u = 0; u < 4; ++u)
                dst[c0 / 4 + u] = make_float4(__uint_as_float(rr[4 * u]), __uint_as_float(rr[4 * u + 1]),
                                              __uint_as_float(rr[4 * u + 2]), __uint_as_float(rr[4 * u + 3]));
            }
          }
        }
      } else if (hi > lo && quad * 32 < args.co) {          // warp-uniform
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * 128);
        float* dst = args.out + (long)g * args.out_stride_g + (long)r * Nw;
#pragma unroll 1
        for (int c0 = 0; c0 < Nw; c0 += 16) {
          uint32_t rr[16];
          tmem_ld16(taddr + (uint32_t)c0, rr);
          tmem_wait_ld();
          if (r < args.co) {
#pragma unroll
            for (int u = 0; u < 16; ++u) atomicAdd(dst + c0 + u, __uint_as_float(rr[u]));
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[as]);
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 0) {
    __syncwarp();
    tmem_dealloc(tmem_base, 256);
  }
}

// =============================================================================================
// tc_bmm_bwd_kernel: the two data gradients of the per-(graph, channel) N x N matmul (layers.py:161-162).
//   MODE 1: dY1[i][k] = alpha (dM Y2^T)[i][k] + beta rowsum(dM)[i]      alpha, beta = GraphNorm (a2, s2) of Y2
//           A = dM (layout C) K-major, B = Y2 (layout B: physical rows k + k/(BN-1)) K-major, K = physical column.
//           The output column index is Y2's physical row = layout C's physical column: the result IS layout C.
//   MODE 2: dY2[k][j] = alpha (Y1^T dM)[k][j] + beta colsum(dM)[j]      alpha, beta = (a1, s1) of Y1
//           A = Y1 (layout A, ones rows zeroed beforehand) MN-major, B = dM (layout C) MN-major; K runs over the 127-row
//           logical tiles: K chunk (rt, h) pairs Y1's physical rows 128 rt + 64 h .. +63 with dM's logical rows
//           127 rt + 64 h .. +63 (the last pair of h = 1 multiplies the zeroed ones row).  Output rows come out in Y1's
//           physical column numbering; the epilogue stores them at their logical row (a hole can only be the last row
//           of a warp's 32: 31-row store box), so the result is layout C as well.
//   Both: 128 x BN tiles, TMA ring, two TMEM accumulator stages, epilogue through swizzled shared memory + TMA store.
// =============================================================================================
template <typename T>
struct BmmBwdArgs {
  int G, C;
  Geo geo;
  const float* coef;      // [G*C][2] (alpha, beta) or null (1, 0)
  const float* vec;       // MODE 1: rowsum [G*C][N];  MODE 2: colsum [G*C][NPC]
  const int32_t* n_per_graph;
};

template <typename T, int BN, int MODE>
__global__ void __launch_bounds__(192, 1)
tc_bmm_bwd_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                  const __grid_constant__ CUtensorMap map_o32, const __grid_constant__ CUtensorMap map_o31,
                  const BmmBwdArgs<T> args) {
  using Cfg = MatmulCfg<BN>;
  constexpr int kStages = Cfg::kStages;
  constexpr uint32_t kTmemCols = (2 * BN <= 128) ? 128 : (2 * BN <= 256 ? 256 : 512);
  extern __shared__ uint8_t smem_bb[];
  uint8_t* smem = smem_bb;
  if ((smem_u32(smem) & 1023u) != 0u) __trap();
  uint8_t* s_store = smem + (size_t)kStages * Cfg::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_store + Cfg::kStoreBytes + 2 * BN * sizeof(float));
  uint64_t* full = bars;
  uint64_t* empty = bars + kStages;
  uint64_t* tmem_full = bars + 2 * kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  const int warp = uniform_warp_idx(), lane = threadIdx.x % 32;
  const Geo geo = args.geo;

  // tiles per plane: M tiles x N tiles (per graph size)
  auto m_tiles = [&](int n) { return MODE == 1 ? (n + 127) / 128 : (phys_k_end(n, geo.TN1) + 127) / 128; };
  auto n_tiles = [&](int n) { return (n + geo.TN1 - 1) / geo.TN1; };
  long total = 0;
  for (int g = 0; g < args.G; ++g) {
    const int n = graph_n(args.n_per_graph, g, geo.N);
    total += (long)m_tiles(n) * n_tiles(n) * args.C;
  }
  struct Walk {
    int g = 0, n = 0, mt = 0, nt = 0;
    long base = 0, tiles_g = 0;
  };
  auto walk_set = [&](Walk& w) {
    w.n = graph_n(args.n_per_graph, w.g, geo.N);
    w.mt = m_tiles(w.n);
    w.nt = n_tiles(w.n);
    w.tiles_g = (long)w.mt * w.nt * args.C;
  };
  auto walk_locate = [&](Walk& w, long t, int& q, int& m, int& nn) {
    while (t >= w.base + w.tiles_g) { w.base += w.tiles_g; ++w.g; walk_set(w); }
    const long local = t - w.base;
    const int per_plane = w.mt * w.nt;
    q = w.g * args.C + (int)(local / per_plane);
    const int rem = (int)(local % per_plane);
    m = rem / w.nt;
    nn = rem % w.nt;
  };
  // number of K stages of a tile
  auto k_stages = [&](int n) {
    if (MODE == 1) return (phys_k_end(n, geo.TN1) + 63) / 64;
    const int rt = (n + kTM1 - 1) / kTM1;
    const int last = n - (rt - 1) * kTM1;          // logical rows in the last tile
    return 2 * (rt - 1) + (last > 64 ? 2 : 1);
  };

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
    if (lane == 0) { prefetch_tensormap(&map_a); prefetch_tensormap(&map_b); }
    Walk w;
    walk_set(w);
    int stage = 0;
    uint32_t phase = 0;
    for (long t = blockIdx.x; t < total; t += gridDim.x) {
      int q, m, nn;
      walk_locate(w, t, q, m, nn);
      const int kts = k_stages(w.n);
      for (int kt = 0; kt < kts; ++kt) {
        mbar_wait(&empty[stage], phase ^ 1);
        uint8_t* sa = smem + (size_t)stage * Cfg::kStageBytes;
        uint8_t* sb = sa + 128 * 128;
        mbar_arrive_expect_tx_e(&full[stage], (uint32_t)Cfg::kStageBytes);
        if (MODE == 1) {
          tma_load_3d_e(sa, &map_a, &full[stage], kt * 64, m * 128, q);          // dM rows x 64 physical columns
          tma_load_3d_e(sb, &map_b, &full[stage], kt * 64, nn * BN, q);          // Y2 physical rows x 64 physical columns
        } else {
          const int rt = kt >> 1, h = kt & 1;
          for (int u = 0; u < 2; ++u)                                            // Y1: 64 rows (K) x 128 physical columns (M)
            tma_load_3d_e(sa + (size_t)u * 8192, &map_a, &full[stage], m * 128 + u * 64, rt * 128 + h * 64, q);
          for (int u = 0; u < BN / 64; ++u)                                      // dM: 64 logical rows (K) x BN columns
            tma_load_3d_e(sb + (size_t)u * 8192, &map_b, &full[stage], nn * BN + u * 64, rt * kTM1 + h * 64, q);
        }
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = make_idesc(Elem<T>::kFmt, MODE == 1 ? 0 : 1, MODE == 1 ? 0 : 1, 128, BN);
    const uint64_t a_d0 = MODE == 1 ? smem_desc_sw128(smem_u32(smem), 16u, 1024u) : smem_desc_sw128(smem_u32(smem), 8192u, 1024u);
    const uint64_t b_d0 = MODE == 1 ? smem_desc_sw128(smem_u32(smem) + 128 * 128, 16u, 1024u)
                                    : smem_desc_sw128(smem_u32(smem) + 128 * 128, 8192u, 1024u);
    const uint32_t a_lo0 = (uint32_t)a_d0, a_hi = (uint32_t)(a_d0 >> 32);
    const uint32_t b_lo0 = (uint32_t)b_d0, b_hi = (uint32_t)(b_d0 >> 32);
    constexpr uint32_t kstep = MODE == 1 ? (32u >> 4) : (2048u >> 4);
    Walk w;
    walk_set(w);
    int stage = 0;
    uint32_t phase = 0;
    int as = 0;
    uint32_t aphase = 0;
    for (long t = blockIdx.x; t < total; t += gridDim.x) {
      int q, m, nn;
      walk_locate(w, t, q, m, nn);
      const int kts = k_stages(w.n);
      mbar_wait(&tmem_empty[as], aphase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(as * BN);
      for (int kt = 0; kt < kts; ++kt) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        const uint32_t a_lo = a_lo0 + (uint32_t)stage * (Cfg::kStageBytes >> 4);
        const uint32_t b_lo = b_lo0 + (uint32_t)stage * (Cfg::kStageBytes >> 4);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          mma_ss2_e(d_tmem, a_lo + (uint32_t)k * kstep, a_hi, b_lo + (uint32_t)k * kstep, b_hi, idesc,
                    (kt > 0 || k > 0) ? 1u : 0u);
        mma_commit_e(&empty[stage]);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      mma_commit_e(&tmem_full[as]);
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
  } else {
    const int quad = warp % 4;
    Walk w;
    walk_set(w);
    int as = 0;
    uint32_t aphase = 0;
    int sbuf = 0;
    for (long t = blockIdx.x; t < total; t += gridDim.x) {
      int q, m, nn;
      walk_locate(w, t, q, m, nn);
      const int n = w.n;
      float alpha = 1.f, beta = 0.f;
      if (args.coef) { alpha = args.coef[2 * q]; beta = args.coef[2 * q + 1]; }
      const int r = quad * 32 + lane;
      const int prow = m * 128 + r;                    // MODE 1: logical row i; MODE 2: physical row numbering (layout B)
      int lrow = prow;
      bool row_ok;
      if (MODE == 1) {
        row_ok = prow < n;
      } else {
        const bool hole_row = (prow & (BN - 1)) == BN - 1;
        lrow = prow - (prow >> geo.BNLOG);
        row_ok = !hole_row && lrow < n;
      }
      float rterm = 0.f;
      if (MODE == 1 && row_ok) rterm = beta * args.vec[(long)q * geo.N + prow];
      mbar_wait(&tmem_full[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * BN);
      const int jlog0 = nn * geo.TN1;
      // store box of this warp's 32 rows: logical start row; 31 rows when the last one is a hole row (MODE 2)
      const int p0 = m * 128 + quad * 32;
      const int store_row = MODE == 1 ? p0 : p0 - (p0 >> geo.BNLOG);
      const bool box31 = MODE == 2 && (((p0 + 31) & (BN - 1)) == BN - 1);
      const CUtensorMap* mo = box31 ? &map_o31 : &map_o32;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 64) {
        if (jlog0 + c0 >= n) break;
        uint8_t* buf = s_store + (size_t)(quad * 2 + sbuf) * 4096;
        if (lane == 0) bulk_wait_group_read1();
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
            float t0 = rterm, t1 = rterm;
            if (MODE == 2) {
              t0 = beta * args.vec[(long)q * geo.NPC + nn * BN + ca];
              t1 = beta * args.vec[(long)q * geo.NPC + nn * BN + cb];
            }
            float x0 = fmaf(alpha, __uint_as_float(rr[2 * u]), t0);
            float x1 = fmaf(alpha, __uint_as_float(rr[2 * u + 1]), t1);
            if (!row_ok || ca == BN - 1 || jlog0 + ca >= n) x0 = 0.f;
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
          tma_store_3d(mo, buf, nn * BN + c0, store_row, q);
          bulk_commit_group();
        }
        sbuf ^= 1;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[as]);
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
    if (lane == 0) bulk_wait_group0();
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
// host side of the training path
// =============================================================================================
// pixel splits per graph of the weight-gradient GEMM (about two work items per SM)
int wgrad_splits(int G, const Geo& geo) {
  const int steps = (int)((geo.PSC + 63) / 64);
  return std::max(1, std::min(steps / 8, ceil_div(2 * num_sms(), G)));
}

// out (+)= the weight-gradient GEMM; rec: deterministic mode, room for G * wgrad_splits(G) records of co x Nw floats
// (the kernel stores each work item's tile there and out is OVERWRITTEN with their fixed-order sum), or null (atomics
// into out, which the caller has zeroed)
template <typename T>
int launch_wgrad(const T* gplanes, int co, const T* src0, int c0, const T* src1, int c1, float* out, long out_stride_g,
                 int G, const Geo& geo, const int32_t* npg, float* rec, cudaStream_t st) {
  const int k0 = round_up(c0, 16), k1 = src1 ? round_up(c1, 16) : 0;
  FGNN_CHECK_ARG(co <= 128 && k0 + k1 <= 128, "weight-gradient GEMM supports <= 128 channels per side (got %d x %d)", co, k0 + k1);
  CUtensorMap ma, mb0, mb1;
  if (int e = pixel_map(&ma, gplanes, co, G, geo, (co + 7) & ~7)) return e;
  if (int e = pixel_map(&mb0, src0, c0, G, geo, k0)) return e;
  if (src1) {
    if (int e = pixel_map(&mb1, src1, c1, G, geo, k1)) return e;
  } else {
    mb1 = mb0;
  }
  WgradArgs a{};
  a.G = G;
  a.S = wgrad_splits(G, geo);
  a.co = co;
  a.Nw = k0 + k1;
  a.k0 = k0;
  a.nsrc = src1 ? 2 : 1;
  a.out = rec ? rec : out;
  a.out_stride_g = out_stride_g;
  a.geo = geo;
  a.n_per_graph = npg;
  const int grid = std::min(num_sms(), G * a.S);
  if (!rec) {
    FGNN_CUDA(cudaFuncSetAttribute(tc_wgrad_kernel<T, AtomicSum>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWgSmemBytes));
    prof::begin(prof::kGlue, st);
    tc_wgrad_kernel<T, AtomicSum><<<grid, 192, kWgSmemBytes, st>>>(ma, mb0, mb1, a);
    prof::end(prof::kGlue, st);
    FGNN_LAUNCHED();
    return FGNN_OK;
  }
  FGNN_CUDA(cudaFuncSetAttribute(tc_wgrad_kernel<T, OrderedSum>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWgSmemBytes));
  prof::begin(prof::kGlue, st);
  tc_wgrad_kernel<T, OrderedSum><<<grid, 192, kWgSmemBytes, st>>>(ma, mb0, mb1, a);
  FGNN_LAUNCHED();
  // per graph over its splits (first layers: out [G][co][Nw]), or over all items in (graph, split) order (one matrix)
  const int w = co * a.Nw;
  const int ret = out_stride_g ? sum_records(rec, out, (long)G * w, a.S, w, false, st) : sum_records(rec, out, w, G * a.S, w, false, st);
  prof::end(prof::kGlue, st);
  return ret;
}

// mode 1: out = alpha (a b^T) + beta rowsum, a = dM (layout C), b = Y2 (layout B);  mode 2: out = alpha (a^T b) + beta colsum,
// a = Y1 (layout A, ones rows zeroed), b = dM (layout C).  out: layout C.
template <typename T>
int launch_bmm_bwd(int mode, const T* a, const T* b, T* out, const float* coef, const float* vec, int G, int C,
                   const Geo& geo, const int32_t* npg, cudaStream_t st) {
  CUtensorMap ma, mb, mo32, mo31;
  const uint64_t planes = (uint64_t)G * C;
  if (mode == 1) {
    if (int e = plane_map(&ma, a, kLayoutC, geo, planes, 128)) return e;
    if (int e = plane_map(&mb, b, kLayoutB, geo, planes, geo.BN)) return e;
  } else {
    if (int e = plane_map(&ma, a, kLayoutA, geo, planes, 64)) return e;
    if (int e = plane_map(&mb, b, kLayoutC, geo, planes, 64)) return e;
  }
  if (int e = plane_map(&mo32, out, kLayoutC, geo, planes, 32)) return e;
  if (int e = plane_map(&mo31, out, kLayoutC, geo, planes, 31)) return e;
  BmmBwdArgs<T> args{G, C, geo, coef, vec, npg};
  const int grid = num_sms();
  return with_bn(geo, [&](auto bn) -> int {
    constexpr int BN = decltype(bn)::value;
    auto kernel = mode == 1 ? tc_bmm_bwd_kernel<T, BN, 1> : tc_bmm_bwd_kernel<T, BN, 2>;
    const size_t smem = MatmulCfg<BN>::kSmemBytes;
    prof::begin(prof::kMatmul, st);
    FGNN_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<grid, 192, smem, st>>>(ma, mb, mo32, mo31, args);
    prof::end(prof::kMatmul, st);
    FGNN_LAUNCHED();
    return FGNN_OK;
  });
}

// Two workspace layouts for the 16-bit training entry points.  Both hold the 16-bit input planes of the whole batch
// first, outside the range that every pass zeroes, and cut the batch into passes of tp.G graphs.
//   PASSES     the workspace holds every activation of one pass (carve_train: about 51 plane sets per graph at depth 3,
//              4 blocks; 107 GB for 64 graphs at N = 500, C = 64).  When the whole batch fits T as one pass, it is one
//              pass: the forward leaves every activation in the workspace until the backward.  Otherwise the passes are
//              `chunk` graphs.  The forward runs pass by pass and keeps only emb; the backward computes the loss scale
//              once over the whole d emb, then per pass re-runs that pass's forward from the input planes and runs the
//              block-stack backward on it (about one extra training forward per step).  Parameter gradients accumulate
//              across passes as they do across calls.
//   CHECKPOINT chosen by the caller (FGNN_CHECKPOINT_BLOCKS), and then always in passes of `chunk` graphs.  The
//              workspace holds, for the whole batch, the input planes, every block's pre-norm output Z3[b], every MLP's
//              GraphNorm coefficients and statistics and the pooling arg-max; and, for one pass, ONE block's
//              intermediates (H, Y1, Y2, MULT, shared by all blocks) and the backward scratch: about nb + 3 D + 11 plane
//              sets per graph instead of 51.  The forward runs pass by pass, block by block.  The backward, per pass and
//              for b = nb-1 .. 0, re-runs block b's forward from Z3[b-1] (the input planes for b = 0) up to, not
//              including, mlp3's last conv, whose output Z3[b] and statistics are kept, then runs block b's backward
//              (about one extra forward per step).
// T = FGNN_TC_TRAIN_WS_GB GiB when set (0: the batch is always cut into passes of `chunk`, and one that fits a single
// pass is not re-run); otherwise half the current device's memory, because a siamese step holds two embedder
// workspaces (x1, x2) until backward; unlimited when no device can be queried (host-only workspace queries).
// chunk = FGNN_TC_CHUNK when set (as for inference), else the largest pass whose own part of the carve fits FGNN_TC_WS_GB
// (default 16) GiB, never less than one graph; the passes are equal, the last one may be shorter.
// The plan is a pure function of (parameter shapes, G, N, flags, T, FGNN_TC_WS_GB, FGNN_TC_CHUNK).  fgnn_embed_bwd derives
// it again from the same arguments and must reach the forward call's answer: neither the variables nor the device may
// change between the two calls.
struct TrainPlan {
  Geo geo;
  int C, cin0, D, nb;
  int c_emb;        // real channels of the embeddings (the last block's c_out)
  int G;            // graphs of one pass: the whole batch or `chunk` (pass_plan lowers it for a short last pass)
  int batch;        // graphs of the call
  bool checkpoint;  // FGNN_CHECKPOINT_BLOCKS: block-level checkpoints, one block's intermediates at a time
  bool det;         // deterministic mode: OrderedSum kernels, and room for their records in the carve
};

// Without checkpoints the workspace keeps every activation of a pass, and a pass holds at least one graph (some 15 GB
// at N = 2048, C = 32), so training stops at the padded size the inference path had before it was extended to kMaxN.
// The checkpoint plan (about 55 GB for one graph at N = 4096, C = 64) trains up to kMaxN.
constexpr int kMaxTrainN = 1024;

struct TrainBuf {
  // kept from forward to backward (xin for the whole call; the rest for the current pass, except on the checkpoint
  // plan: Z3, coef, gnstat and arg for the whole call, the other planes for one block of the current pass, H[b] ..
  // MULT[b] the same buffers for every b)
  void* xin;
  void* H[FGNN_MAX_BLOCKS][3][FGNN_MAX_DEPTH];
  void *Y1[FGNN_MAX_BLOCKS], *Y2[FGNN_MAX_BLOCKS], *MULT[FGNN_MAX_BLOCKS], *Z3[FGNN_MAX_BLOCKS];
  float* coef[FGNN_MAX_BLOCKS][3];
  float* gnstat[FGNN_MAX_BLOCKS][3];
  int32_t* arg;
  size_t planes_begin, planes_end;       // byte range of the plane buffers above (ragged batches zero all of it)
  // scratch of both passes
  void* wf;
  float* bf;
  double* stat_acc;
  float* zeros;
  float* wt[2];
  // backward scratch
  void *A0, *A1, *B0, *B1, *DM, *DX3[2], *DX12[2], *DY1, *DY2;
  size_t bwd_begin, bwd_end;
  double* gacc;
  float *bc, *bsum[2], *rowsum, *colsum, *P, *Pglob, *scale;
  // deterministic mode only (else null): OrderedSum records of the conv-chain statistics, the GraphNorm backward
  // sums [GC][kPlaneCtas][2], the bias-gradient sums [GC][kPlaneCtas] and the weight-gradient GEMM [items][C][128]
  double *stat_rec, *gacc_rec;
  float *bsum_rec, *wg_rec;
};

// CTAs per plane of the plane reductions (gn_bwd_stats / gn_bwd_apply / relu_mask)
constexpr int kPlaneCtas = 32;

size_t carve_train(const TrainPlan& tp, Arena& ar, TrainBuf& B) {
  const Geo& geo = tp.geo;
  const size_t G = tp.G, C = tp.C;
  const size_t actC = G * C * geo.stride(kLayoutC);
  // the batch's input planes come first, outside the plane range that every pass zeroes
  B.xin = ar.take<uint16_t>((size_t)tp.batch * tp.cin0 * geo.stride(kLayoutC), 1024);
  if (tp.checkpoint) {   // the block checkpoints of the whole batch, also outside that range
    const size_t BC = (size_t)tp.batch * C;
    for (int b = 0; b < tp.nb; ++b) B.Z3[b] = ar.take<uint16_t>(BC * geo.stride(kLayoutC), 1024);
    for (int b = 0; b < tp.nb; ++b)
      for (int m = 0; m < 3; ++m) {
        B.coef[b][m] = ar.take<float>(BC * 2);
        B.gnstat[b][m] = ar.take<float>(BC * 4);
      }
    B.arg = ar.take<int32_t>(BC * geo.N);
  }
  B.planes_begin = align_up(ar.off, 1024);
  const int sets = tp.checkpoint ? 1 : tp.nb;
  for (int b = 0; b < sets; ++b) {
    for (int m = 0; m < 3; ++m)
      for (int l = 0; l < tp.D - 1; ++l) B.H[b][m][l] = ar.take<uint16_t>(actC, 1024);
    B.Y1[b] = ar.take<uint16_t>(G * C * geo.stride(kLayoutA), 1024);
    B.Y2[b] = ar.take<uint16_t>(G * C * geo.stride(kLayoutB), 1024);
    B.MULT[b] = ar.take<uint16_t>(actC, 1024);
    if (!tp.checkpoint) B.Z3[b] = ar.take<uint16_t>(actC, 1024);
  }
  for (int b = sets; b < tp.nb; ++b) {
    for (int m = 0; m < 3; ++m)
      for (int l = 0; l < tp.D - 1; ++l) B.H[b][m][l] = B.H[0][m][l];
    B.Y1[b] = B.Y1[0];
    B.Y2[b] = B.Y2[0];
    B.MULT[b] = B.MULT[0];
  }
  B.planes_end = ar.off;
  if (!tp.checkpoint) {
    for (int b = 0; b < tp.nb; ++b)
      for (int m = 0; m < 3; ++m) {
        B.coef[b][m] = ar.take<float>(G * C * 2);
        B.gnstat[b][m] = ar.take<float>(G * C * 4);
      }
    B.arg = ar.take<int32_t>(G * C * geo.N);
  }
  B.wf = ar.take<uint16_t>(G * 2 * C * 256, 1024);
  B.bf = ar.take<float>(G * 2 * C);
  B.stat_acc = ar.take<double>(G * 2 * C * 2);
  B.zeros = ar.take<float>(512);
  B.wt[0] = ar.take<float>(256 * 256);
  B.wt[1] = ar.take<float>(256 * 256);
  B.bwd_begin = align_up(ar.off, 1024);
  void** bp[] = {&B.A0, &B.A1, &B.B0, &B.B1, &B.DM, &B.DX3[0], &B.DX3[1], &B.DX12[0], &B.DX12[1], &B.DY1, &B.DY2};
  for (void** q : bp) *q = ar.take<uint16_t>(actC, 1024);
  B.bwd_end = ar.off;
  B.gacc = ar.take<double>(G * C * 2);
  B.bc = ar.take<float>(G * C * 4);
  B.bsum[0] = ar.take<float>(G * C);
  B.bsum[1] = ar.take<float>(G * C);
  B.rowsum = ar.take<float>(G * C * geo.N);
  B.colsum = ar.take<float>(G * C * geo.NPC);
  B.P = ar.take<float>(G * C * 128);
  B.Pglob = ar.take<float>(128 * 128);
  B.scale = ar.take<float>(4);
  B.stat_rec = tp.det ? ar.take<double>(stat_rec_doubles(tp.G, tp.C, geo)) : nullptr;
  B.gacc_rec = tp.det ? ar.take<double>(G * C * kPlaneCtas * 2) : nullptr;
  B.bsum_rec = tp.det ? ar.take<float>(G * C * kPlaneCtas) : nullptr;
  // a pass of g <= G graphs has g * wgrad_splits(g) < g + 2 num_sms() work items, each at most C x 128
  B.wg_rec = tp.det ? ar.take<float>((G + 2 * (size_t)num_sms()) * C * 128) : nullptr;
  return align_up(ar.off, 1024);
}

size_t train_workspace_bytes(const TrainPlan& tp) {
  Arena ar(nullptr, 0);
  TrainBuf B;
  return carve_train(tp, ar, B);
}

// T of the plan selection, in bytes (see TrainPlan)
size_t one_pass_limit() {
  if (const char* v = getenv("FGNN_TC_TRAIN_WS_GB")) return (size_t)(std::min(std::max(atof(v), 0.0), 1e9) * (double)(1ull << 30));
  static size_t cache[64] = {0};   // per device: the query is not free and runs three times per embedder call
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();            // no device: leave no error behind for a later launch check
    return SIZE_MAX;
  }
  if (dev >= 0 && dev < 64 && cache[dev]) return cache[dev];
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
    cudaGetLastError();
    return SIZE_MAX;
  }
  const size_t t = prop.totalGlobalMem / 2;
  if (dev >= 0 && dev < 64) cache[dev] = t;
  return t;
}

int make_train_plan(const fgnn_embed_params& p, int G, int N, bool det, bool ckpt, TrainPlan& tp) {
  if (ckpt && N > kMaxN)
    return fail(FGNN_ERR_UNSUPPORTED, "16-bit training with block checkpoints supports N <= %d (got %d)", kMaxN, N);
  if (!ckpt && N > kMaxTrainN)
    return fail(FGNN_ERR_UNSUPPORTED, "16-bit training supports N <= %d (got %d): its workspace holds every activation of at "
                "least one graph; embed larger graphs with the inference path (N <= %d), or train them with block "
                "checkpoints (FGNN_CHECKPOINT_BLOCKS, Network.set_checkpoint_blocks)", kMaxTrainN, N, kMaxN);
  Plan pl;
  if (int e = make_plan(p, G, N, pl)) return e;
  tp.geo = pl.geo;
  tp.C = pl.C;
  tp.cin0 = pl.cin0;
  tp.nb = p.num_blocks;
  tp.c_emb = p.block[p.num_blocks - 1].mlp3.c_out;
  tp.G = G;
  tp.batch = G;
  tp.checkpoint = ckpt;
  tp.det = det;
  tp.D = p.block[0].mlp1.depth;
  for (int b = 0; b < p.num_blocks; ++b) {
    const fgnn_block_params& bp = p.block[b];
    if (bp.mlp1.depth != tp.D || bp.mlp2.depth != tp.D || bp.mlp3.depth != tp.D)
      return fail(FGNN_ERR_UNSUPPORTED, "16-bit training needs the same depth_of_mlp in every MLP");
  }
  if (tp.D < 1 || tp.D > FGNN_MAX_DEPTH) return fail(FGNN_ERR_INVALID, "bad depth %d", tp.D);
  if (tp.cin0 > 64) return fail(FGNN_ERR_UNSUPPORTED, "original_features_num %d > 64 unsupported", tp.cin0);
  if ((long)G * tp.C > 65535) return fail(FGNN_ERR_UNSUPPORTED, "16-bit training: G * C = %ld planes exceed one call's grid (split the batch)", (long)G * tp.C);
  if (!ckpt && train_workspace_bytes(tp) <= one_pass_limit()) return FGNN_OK;   // the whole batch in one pass
  int chunk = env_int("FGNN_TC_CHUNK", 0);
  if (chunk <= 0) {   // the largest pass whose own carve (batch = 0: without the batch-wide part) fits the budget, or 1
    const size_t budget = (size_t)std::max(1, env_int("FGNN_TC_WS_GB", 16)) << 30;
    TrainPlan q = tp;
    q.batch = 0;
    int lo = 1, hi = G;
    while (lo < hi) {
      q.G = lo + (hi - lo + 1) / 2;
      if (train_workspace_bytes(q) <= budget) lo = q.G; else hi = q.G - 1;
    }
    chunk = lo;
  }
  chunk = std::min(chunk, G);
  const int passes = (G + chunk - 1) / chunk;
  tp.G = (G + passes - 1) / passes;
  return FGNN_OK;
}

// the plan of the pass that starts at graph g0: the same carve, launches over the pass's graphs only
TrainPlan pass_plan(const TrainPlan& tp, int g0) {
  TrainPlan pp = tp;
  pp.G = std::min(tp.G, tp.batch - g0);
  return pp;
}

// the buffers of the pass that starts at graph g0: its graphs' part of the batch-wide buffers (the input planes, and on
// the checkpoint plan the checkpoints), B's own for the rest (they hold one pass)
TrainBuf pass_bufs(const TrainPlan& tp, const TrainBuf& B, int g0) {
  TrainBuf V = B;
  V.xin = static_cast<uint16_t*>(B.xin) + (size_t)g0 * tp.cin0 * tp.geo.PSC;
  if (!tp.checkpoint) return V;
  const size_t gc = (size_t)g0 * tp.C;
  for (int b = 0; b < tp.nb; ++b) {
    V.Z3[b] = static_cast<uint16_t*>(B.Z3[b]) + gc * tp.geo.PSC;
    for (int m = 0; m < 3; ++m) {
      V.coef[b][m] = B.coef[b][m] + gc * 2;
      V.gnstat[b][m] = B.gnstat[b][m] + gc * 4;
    }
  }
  V.arg = B.arg + gc * tp.geo.N;
  return V;
}

// Zero what a pass's producers never write but later reads cover, before every pass's forward.  Ragged batch: all the
// kept planes and the backward scratch (rows beyond a graph's covered range are never written, the GEMM K loops read
// them, and an earlier pass's larger graph leaves data there).  Otherwise: the physical rows / column chunks the
// producers skip.  The batch-wide part of the workspace lies before planes_begin and is not touched.
int zero_pass(const TrainPlan& tp, const TrainBuf& B, void* ws, bool ragged, cudaStream_t st) {
  const Geo& geo = tp.geo;
  const size_t GC = (size_t)tp.G * tp.C;
  char* base = static_cast<char*>(ws);
  if (ragged) {
    FGNN_CUDA(cudaMemsetAsync(base + B.planes_begin, 0, B.planes_end - B.planes_begin, st));
    FGNN_CUDA(cudaMemsetAsync(base + B.bwd_begin, 0, B.bwd_end - B.bwd_begin, st));
  } else {
    for (int b = 0; b < (tp.checkpoint ? 1 : tp.nb); ++b) {   // checkpoint: one set of planes shared by all blocks
      FGNN_CUDA(cudaMemsetAsync(B.Y1[b], 0, GC * geo.PSA * 2, st));
      FGNN_CUDA(cudaMemsetAsync(B.Y2[b], 0, GC * geo.PSB * 2, st));
      FGNN_CUDA(cudaMemsetAsync(B.MULT[b], 0, GC * geo.PSC * 2, st));
    }
    FGNN_CUDA(cudaMemsetAsync(B.DY1, 0, GC * geo.PSC * 2, st));
    FGNN_CUDA(cudaMemsetAsync(B.DY2, 0, GC * geo.PSC * 2, st));
  }
  return FGNN_OK;
}

// a depth-1 launch of the conv-chain kernel on the training scratch, as every 1x1 conv of training is: one MLP, one
// source, outputs in layout C until the caller sets otherwise
template <typename T>
MlpGroup<T> conv_group(const TrainBuf& B) {
  MlpGroup<T> M{};
  M.nmlp = M.nsrc = 1;
  M.wf = reinterpret_cast<T*>(B.wf);
  M.bf = B.bf;
  M.stat_acc = B.stat_acc;
  M.stat_rec = B.stat_rec;
  return M;
}

// layer l of mp as a depth-1 launch (a missing bias reads as zeros); its last layer finalises mp's GraphNorm
MlpLayers layer(const fgnn_mlp_params& mp, int l, const float* zeros) {
  return {mp.w[l], {mp.b[l] ? mp.b[l] : zeros}, 1, mp.c_out, l == mp.depth - 1 ? &mp : nullptr};
}

// a data-gradient conv: wt is a transposed weight zero-padded by transpose_slice_kernel to (C, C per source); no bias, no GraphNorm
MlpLayers transposed(const float* wt, const TrainBuf& B, int C) { return {wt, {B.zeros}, 1, C, nullptr}; }

// input of block b: the input planes xin for b = 0, else the previous block's pre-norm output and its GraphNorm fold
template <typename T>
Src<T> block_in(const fgnn_embed_params& p, const TrainPlan& tp, const TrainBuf& B, int b) {
  if (b == 0) return {reinterpret_cast<const T*>(B.xin), tp.cin0, tp.cin0, nullptr};
  return {reinterpret_cast<const T*>(B.Z3[b - 1]), tp.C, p.block[b - 1].mlp3.c_out, B.coef[b - 1][2]};
}

// training forward of block b of one pass (tp.G graphs): writes its hidden activations, Y1, Y2, MULT, Z3[b] and the
// GraphNorm statistics of its MLPs into B.  z3 = false stops before mlp3's last conv (the checkpoint plan's backward:
// Z3[b] and its statistics are kept, never rewritten).
template <typename T>
int train_fwd_block(const fgnn_embed_params& p, const TrainPlan& tp, const TrainBuf& B, int b, bool z3,
                    const int32_t* npg, cudaStream_t st) {
  const Geo& geo = tp.geo;
  const int G = tp.G, C = tp.C, D = tp.D;
  const Src<T> in = block_in<T>(p, tp, B, b);
  const fgnn_block_params& bp = p.block[b];
  const int co = bp.mlp1.c_out;
  const fgnn_mlp_params* mlps[2] = {&bp.mlp1, &bp.mlp2};
  T* y12[2] = {reinterpret_cast<T*>(B.Y1[b]), reinterpret_cast<T*>(B.Y2[b])};
  const Layout mode12[2] = {kLayoutA, kLayoutB};
  for (int l = 0; l < D; ++l) {
    const bool last = l == D - 1;
    const int nmlp = l == 0 ? 2 : 1;   // mlp1 and mlp2 share the block input: one launch of their first layers
    for (int m0 = 0; m0 < 2; m0 += nmlp) {
      MlpGroup<T> M = conv_group<T>(B);
      M.nmlp = nmlp;
      M.src[0] = l == 0 ? in : Src<T>{reinterpret_cast<const T*>(B.H[b][m0][l - 1]), C, co, nullptr};
      for (int j = 0; j < nmlp; ++j) {
        const int m = m0 + j;
        M.mlp[j] = layer(*mlps[m], l, B.zeros);
        M.out[j] = last ? y12[m] : reinterpret_cast<T*>(B.H[b][m][l]);
        M.out_mode[j] = last ? mode12[m] : kLayoutC;
        M.ones[j] = last ? 1 : 0;
        if (last) { M.coef[j] = B.coef[b][m]; M.gnstat[j] = B.gnstat[b][m]; }
      }
      M.relu_out = !last;
      if (int e = run_mlp_group<T>(M, C, G, geo, npg, st)) return e;
    }
  }
  T* mult = reinterpret_cast<T*>(B.MULT[b]);
  if (int e = launch_matmul<T>(y12[0], y12[1], mult, B.coef[b][0], B.coef[b][1], G, C, geo, npg, st)) return e;
  for (int l = 0; l < (z3 ? D : D - 1); ++l) {
    const bool last = l == D - 1;
    MlpGroup<T> M = conv_group<T>(B);
    M.src[0] = Src<T>{l == 0 ? mult : reinterpret_cast<const T*>(B.H[b][2][l - 1]), C, co, nullptr};
    if (l == 0) { M.src[1] = in; M.nsrc = 2; }
    M.mlp[0] = layer(bp.mlp3, l, B.zeros);
    M.out[0] = reinterpret_cast<T*>(last ? B.Z3[b] : B.H[b][2][l]);
    if (last) { M.coef[0] = B.coef[b][2]; M.gnstat[0] = B.gnstat[b][2]; }
    M.relu_out = !last;
    if (int e = run_mlp_group<T>(M, C, G, geo, npg, st)) return e;
  }
  return FGNN_OK;
}

// training forward of one pass (tp.G graphs): their input planes B.xin -> emb (tp.G, C, N), and in B everything the
// backward reads
template <typename T>
int train_fwd_pass(const fgnn_embed_params& p, const TrainPlan& tp, const TrainBuf& B, float* emb, const int32_t* npg,
                   cudaStream_t st) {
  const Geo& geo = tp.geo;
  for (int b = 0; b < tp.nb; ++b)
    if (int e = train_fwd_block<T>(p, tp, B, b, true, npg, st)) return e;
  {
    const Src<T> out = block_in<T>(p, tp, B, tp.nb);
    dim3 grid((unsigned)((geo.N + 7) / 8), tp.G * tp.C);
    colmax16_kernel<T><<<grid, 256, 0, st>>>(out.x, out.coef, emb, B.arg, tp.C, out.c_real, geo, npg);
    FGNN_LAUNCHED();
  }
  return FGNN_OK;
}

template <typename T>
int embed_fwd_train_t(const fgnn_embed_params& p, bool det, bool ckpt, const float* x, float* emb, int G, int N,
                      const int32_t* npg, void* ws, size_t ws_bytes, cudaStream_t st) {
  TrainPlan tp;
  if (int e = make_train_plan(p, G, N, det, ckpt, tp)) return e;
  Arena ar(ws, ws_bytes);
  TrainBuf B;
  const size_t need = carve_train(tp, ar, B);
  if (need > ws_bytes) return fail(FGNN_ERR_WORKSPACE, "training workspace too small: %zu < %zu", ws_bytes, need);
  const Geo& geo = tp.geo;
  FGNN_CUDA(cudaMemsetAsync(B.zeros, 0, 512 * sizeof(float), st));
  if (tp.checkpoint && npg)   // ragged: the batch's checkpoints once, as zero_pass does for a pass's planes
    for (int b = 0; b < tp.nb; ++b) FGNN_CUDA(cudaMemsetAsync(B.Z3[b], 0, (size_t)G * tp.C * geo.PSC * sizeof(T), st));
  {   // the whole batch's input planes, every pixel (padding and holes included) written
    dim3 grid((unsigned)std::min(N, 256), G * tp.cin0);
    to_planes_c_kernel<T><<<grid, 256, 0, st>>>(x, reinterpret_cast<T*>(B.xin), tp.cin0, geo, npg);
    FGNN_LAUNCHED();
  }
  for (int g0 = 0; g0 < G; g0 += tp.G) {
    const TrainPlan pp = pass_plan(tp, g0);
    if (int e = zero_pass(pp, B, ws, npg != nullptr, st)) return e;
    if (int e = train_fwd_pass<T>(p, pp, pass_bufs(tp, B, g0), emb + (size_t)g0 * tp.c_emb * N, npg ? npg + g0 : nullptr,
                                  st)) return e;
  }
  return FGNN_OK;
}

// backward of one MlpBlock_Real.  dy = dya (+ dyb) in layout C is the gradient of the NORMALISED output; z the stored
// pre-norm output (layout zmode).  bufs[0..1]: ping-pong planes; on return *g0 (one of them) holds the gradient of the
// first conv's output, which the caller turns into the data gradient of the MLP's sources.
template <typename T>
struct MlpBwd {
  const fgnn_mlp_params* mp;
  const fgnn_mlp_grads* gr;
  const T* dya;
  const T* dyb;
  const T* z;
  Layout zmode;
  const float* coef;
  const float* gnstat;
  void* const* H;               // hidden activations h_0 .. h_{D-2} (layout C)
  int co_real;                  // real output channels (mp's c_out)
  Src<T> src[2];
  int nsrc;
  T* bufs[2];
};

template <typename T>
int mlp_bwd(const MlpBwd<T>& a, const TrainPlan& tp, const TrainBuf& B, const int32_t* npg, cudaStream_t st, T** g0) {
  const Geo& geo = tp.geo;
  const int G = tp.G, C = tp.C, D = tp.D;
  const int GC = G * C;
  const dim3 pgrid((unsigned)std::max<long>(1, std::min<long>(kPlaneCtas, (geo.PSC / 8 + 255) / 256)), GC);
  const bool det = tp.det;
  // bias-gradient sums of the plane kernels: atomics into bsum[bi] (zeroed), or records reduced into it
  auto bsum_begin = [&](int bi) -> int {
    if (!det) FGNN_CUDA(cudaMemsetAsync(B.bsum[bi], 0, (size_t)GC * sizeof(float), st));
    return FGNN_OK;
  };
  auto bsum_end = [&](int bi) -> int { return det ? sum_records(B.bsum_rec, B.bsum[bi], GC, (int)pgrid.x, 1, false, st) : FGNN_OK; };
  prof::begin(prof::kStats, st);
  if (det) {
    gn_bwd_stats_kernel<T, OrderedSum><<<pgrid, 256, 0, st>>>(a.dya, a.dyb, a.z, a.zmode, B.gacc_rec, C, geo, npg);
    FGNN_LAUNCHED();
    if (int e = sum_records(B.gacc_rec, B.gacc, (long)GC * 2, (int)pgrid.x, 2, false, st)) return e;
  } else {
    FGNN_CUDA(cudaMemsetAsync(B.gacc, 0, (size_t)GC * 2 * sizeof(double), st));
    gn_bwd_stats_kernel<T, AtomicSum><<<pgrid, 256, 0, st>>>(a.dya, a.dyb, a.z, a.zmode, B.gacc, C, geo, npg);
    FGNN_LAUNCHED();
  }
  gn_bwd_coef_kernel<<<ceil_div(GC, 256), 256, 0, st>>>(B.gacc, a.coef, a.gnstat, B.bc, C, geo.N, npg, GC);
  FGNN_LAUNCHED();
  gn_param_grad_kernel<<<ceil_div(C, 64), 64, 0, st>>>(B.gacc, a.gnstat, a.gr->gn_w, a.gr->gn_b, B.scale, G, C, a.co_real);
  FGNN_LAUNCHED();
  int bi = 0;                                           // bsum[bi] = per-(graph, channel) sum of the current gradient
  if (int e = bsum_begin(bi)) return e;
  if (det) gn_bwd_apply_kernel<T, OrderedSum><<<pgrid, 256, 0, st>>>(a.dya, a.dyb, a.z, a.zmode, B.bc, a.bufs[0], B.bsum_rec, C, geo, npg);
  else gn_bwd_apply_kernel<T, AtomicSum><<<pgrid, 256, 0, st>>>(a.dya, a.dyb, a.z, a.zmode, B.bc, a.bufs[0], B.bsum[bi], C, geo, npg);
  FGNN_LAUNCHED();
  if (int e = bsum_end(bi)) return e;
  prof::end(prof::kStats, st);
  T* curg = a.bufs[0];
  for (int l = D - 1; l >= 1; --l) {
    const T* hin = reinterpret_cast<const T*>(a.H[l - 1]);
    // weight / bias gradient of layer l (all graphs into one matrix)
    if (!det) FGNN_CUDA(cudaMemsetAsync(B.Pglob, 0, 128 * 128 * sizeof(float), st));
    if (int e = launch_wgrad<T>(curg, C, hin, C, nullptr, 0, B.Pglob, 0, G, geo, npg, B.wg_rec, st)) return e;
    wgrad_combine_hidden_kernel<<<ceil_div(C * C, 256), 256, 0, st>>>(B.Pglob, round_up(C, 16), B.bsum[bi], a.gr->w[l], a.gr->b[l],
                                                                      B.scale, G, C, a.co_real, a.co_real);
    FGNN_LAUNCHED();
    // data gradient: pre = W_l^T g, then the ReLU mask of h_{l-1}
    transpose_slice_kernel<<<ceil_div(C * C, 256), 256, 0, st>>>(a.mp->w[l], B.wt[0], C, a.co_real, a.co_real, 0, C, a.co_real, C, 0);
    FGNN_LAUNCHED();
    T* nxt = (curg == a.bufs[0]) ? a.bufs[1] : a.bufs[0];
    MlpGroup<T> M = conv_group<T>(B);
    M.src[0] = Src<T>{curg, C, C, nullptr};
    M.mlp[0] = transposed(B.wt[0], B, C);
    M.out[0] = nxt;
    if (int e = run_mlp_group<T>(M, C, G, geo, npg, st)) return e;
    bi ^= 1;
    if (int e = bsum_begin(bi)) return e;
    prof::begin(prof::kStats, st);
    if (det) relu_mask_kernel<T, OrderedSum><<<pgrid, 256, 0, st>>>(nxt, hin, B.bsum_rec, C, geo, npg);
    else relu_mask_kernel<T, AtomicSum><<<pgrid, 256, 0, st>>>(nxt, hin, B.bsum[bi], C, geo, npg);
    FGNN_LAUNCHED();
    if (int e = bsum_end(bi)) return e;
    prof::end(prof::kStats, st);
    curg = nxt;
  }
  // first layer: per-graph pixel GEMM, combined through the per-graph GraphNorm fold of the sources
  {
    const int k0 = round_up(a.src[0].c, 16), k1 = a.nsrc > 1 ? round_up(a.src[1].c, 16) : 0;
    const int Nw = k0 + k1;
    if (!det) FGNN_CUDA(cudaMemsetAsync(B.P, 0, (size_t)G * C * Nw * sizeof(float), st));
    if (int e = launch_wgrad<T>(curg, C, a.src[0].x, a.src[0].c, a.nsrc > 1 ? a.src[1].x : nullptr, a.src[1].c, B.P, (long)C * Nw, G,
                                geo, npg, B.wg_rec, st)) return e;
    CombineFirstArgs ca{};
    ca.P = B.P;
    ca.bsum = B.bsum[bi];
    for (int s = 0; s < a.nsrc; ++s) { ca.coef[s] = a.src[s].coef; ca.c[s] = a.src[s].c; ca.cr[s] = a.src[s].c_real; }
    ca.koff[0] = 0;
    ca.koff[1] = k0;
    ca.nsrc = a.nsrc;
    ca.G = G;
    ca.co = C;
    ca.co_real = a.co_real;
    ca.ldp = Nw;
    ca.dW = a.gr->w[0];
    ca.db = a.gr->b[0];
    ca.scale = B.scale;
    const int cin = ca.c[0] + ca.c[1];
    wgrad_combine_first_kernel<<<ceil_div(std::max(C * cin, C), 256), 256, 0, st>>>(ca);
    FGNN_LAUNCHED();
  }
  *g0 = curg;
  return FGNN_OK;
}

// block-stack backward of one pass (tp.G graphs) whose forward state is in B: demb (tp.G, C, N), scaled by *B.scale.
// On the checkpoint plan B holds the pass's checkpoints, and each block's forward is re-run just before its backward.
template <typename T>
int train_bwd_pass(const fgnn_embed_params& p, const fgnn_embed_grads& gr, const TrainPlan& tp, const TrainBuf& B,
                   const float* demb, const int32_t* npg, cudaStream_t st) {
  const Geo& geo = tp.geo;
  const int G = tp.G, N = geo.N, C = tp.C, GC = G * C;
  const size_t plane_bytes = (size_t)GC * geo.PSC * sizeof(T);
  // gradient of the last block's normalised output: zero planes + the pooling scatter
  T* dOutA = reinterpret_cast<T*>(B.DX3[tp.nb & 1]);
  const T* dOutB = nullptr;
  FGNN_CUDA(cudaMemsetAsync(dOutA, 0, plane_bytes, st));
  {
    const long total = (long)GC * N;
    pool_scatter_kernel<T><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(demb, B.arg, B.scale, dOutA, C, tp.c_emb, geo, total);
    FGNN_LAUNCHED();
  }
  for (int b = tp.nb - 1; b >= 0; --b) {
    // checkpoint plan: block b's intermediates, re-derived from its kept input into the planes all blocks share
    if (tp.checkpoint)
      if (int e = train_fwd_block<T>(p, tp, B, b, false, npg, st)) return e;
    const fgnn_block_params& bp = p.block[b];
    const fgnn_block_grads& bg = gr.block[b];
    const Src<T> in = block_in<T>(p, tp, B, b);
    const int co = bp.mlp1.c_out;
    T* A[2] = {reinterpret_cast<T*>(B.A0), reinterpret_cast<T*>(B.A1)};
    T* Bb[2] = {reinterpret_cast<T*>(B.B0), reinterpret_cast<T*>(B.B1)};
    T* DM = reinterpret_cast<T*>(B.DM);
    T* dx3 = reinterpret_cast<T*>(B.DX3[b & 1]);
    T* dx12 = reinterpret_cast<T*>(B.DX12[b & 1]);
    // ---- mlp3 ----
    T* g3 = nullptr;
    {
      MlpBwd<T> a{};
      a.mp = &bp.mlp3; a.gr = &bg.mlp3;
      a.dya = dOutA; a.dyb = dOutB;
      a.z = reinterpret_cast<const T*>(B.Z3[b]); a.zmode = kLayoutC;
      a.coef = B.coef[b][2]; a.gnstat = B.gnstat[b][2];
      a.H = B.H[b][2];
      a.co_real = co;
      a.src[0] = Src<T>{reinterpret_cast<const T*>(B.MULT[b]), C, co, nullptr}; a.src[1] = in; a.nsrc = 2;
      a.bufs[0] = A[0]; a.bufs[1] = A[1];
      if (int e = mlp_bwd<T>(a, tp, B, npg, st, &g3)) return e;
      // data gradients of the two sources: d mult = W0[:, :co]^T g, d cur = W0[:, co:]^T g (not needed for the raw input)
      const int cin = co + in.c_real;
      transpose_slice_kernel<<<ceil_div(C * C, 256), 256, 0, st>>>(bp.mlp3.w[0], B.wt[0], C, co, cin, 0, C, co, C, 0);
      FGNN_LAUNCHED();
      MlpGroup<T> M = conv_group<T>(B);
      M.src[0] = Src<T>{g3, C, C, nullptr};
      M.mlp[0] = transposed(B.wt[0], B, C);
      M.out[0] = DM;
      if (b > 0) {
        transpose_slice_kernel<<<ceil_div(C * C, 256), 256, 0, st>>>(bp.mlp3.w[0], B.wt[1], C, co, cin, co, C, in.c_real, C, 0);
        FGNN_LAUNCHED();
        M.nmlp = 2;
        M.mlp[1] = transposed(B.wt[1], B, C);
        M.out[1] = dx3;
      }
      if (int e = run_mlp_group<T>(M, C, G, geo, npg, st)) return e;
    }
    // ---- matmul ----
    {
      prof::begin(prof::kStats, st);
      plane_rowsum_kernel<T><<<dim3((unsigned)((N + 7) / 8), GC), 256, 0, st>>>(DM, B.rowsum, C, geo, npg);
      FGNN_LAUNCHED();
      plane_colsum_kernel<T><<<dim3((unsigned)((geo.NPC + 255) / 256), GC), 256, 0, st>>>(DM, B.colsum, C, geo, npg);
      FGNN_LAUNCHED();
      zero_inserted_rows_kernel<T><<<dim3(4, GC), 256, 0, st>>>(reinterpret_cast<T*>(B.Y1[b]), geo, kLayoutA);
      FGNN_LAUNCHED();
      prof::end(prof::kStats, st);
      if (int e = launch_bmm_bwd<T>(1, DM, reinterpret_cast<const T*>(B.Y2[b]), reinterpret_cast<T*>(B.DY1), B.coef[b][1], B.rowsum,
                                    G, C, geo, npg, st)) return e;
      if (int e = launch_bmm_bwd<T>(2, reinterpret_cast<const T*>(B.Y1[b]), DM, reinterpret_cast<T*>(B.DY2), B.coef[b][0], B.colsum,
                                    G, C, geo, npg, st)) return e;
    }
    // ---- mlp1 / mlp2 ----
    T* g12[2] = {nullptr, nullptr};
    for (int m = 0; m < 2; ++m) {
      MlpBwd<T> a{};
      a.mp = m == 0 ? &bp.mlp1 : &bp.mlp2;
      a.gr = m == 0 ? &bg.mlp1 : &bg.mlp2;
      a.dya = reinterpret_cast<const T*>(m == 0 ? B.DY1 : B.DY2); a.dyb = nullptr;
      a.z = reinterpret_cast<const T*>(m == 0 ? B.Y1[b] : B.Y2[b]); a.zmode = m == 0 ? kLayoutA : kLayoutB;
      a.coef = B.coef[b][m]; a.gnstat = B.gnstat[b][m];
      a.H = B.H[b][m];
      a.co_real = co;
      a.src[0] = in; a.nsrc = 1;
      a.bufs[0] = m == 0 ? A[0] : Bb[0];
      a.bufs[1] = m == 0 ? A[1] : Bb[1];
      if (int e = mlp_bwd<T>(a, tp, B, npg, st, &g12[m])) return e;
    }
    if (b > 0) {
      // d cur (through mlp1 and mlp2) = [W0_1^T | W0_2^T] [g1; g2]: one two-source conv
      transpose_slice_kernel<<<ceil_div(C * C, 256), 256, 0, st>>>(bp.mlp1.w[0], B.wt[0], C, co, in.c_real, 0, C, in.c_real, 2 * C, 0);
      FGNN_LAUNCHED();
      transpose_slice_kernel<<<ceil_div(C * C, 256), 256, 0, st>>>(bp.mlp2.w[0], B.wt[0], C, co, in.c_real, 0, C, in.c_real, 2 * C, C);
      FGNN_LAUNCHED();
      MlpGroup<T> M = conv_group<T>(B);
      M.src[0] = Src<T>{g12[0], C, C, nullptr};
      M.src[1] = Src<T>{g12[1], C, C, nullptr};
      M.nsrc = 2;
      M.mlp[0] = transposed(B.wt[0], B, C);
      M.out[0] = dx12;
      if (int e = run_mlp_group<T>(M, C, G, geo, npg, st)) return e;
      dOutA = dx3;
      dOutB = dx12;
    }
  }
  return FGNN_OK;
}

template <typename T>
int embed_bwd_t(const fgnn_embed_params& p, const fgnn_embed_grads& gr, bool det, bool ckpt, const float* demb, int grad_scale_log2,
                int G, int N, const int32_t* npg, void* ws, size_t ws_bytes, cudaStream_t st) {
  TrainPlan tp;
  if (int e = make_train_plan(p, G, N, det, ckpt, tp)) return e;
  Arena ar(ws, ws_bytes);
  TrainBuf B;
  const size_t need = carve_train(tp, ar, B);
  if (need > ws_bytes) return fail(FGNN_ERR_WORKSPACE, "training workspace too small: %zu < %zu", ws_bytes, need);
  // one loss scale for the whole batch, whatever the passes
  grad_scale_kernel<<<1, 1024, 0, st>>>(demb, (long)G * tp.c_emb * N, B.scale, grad_scale_log2);
  FGNN_LAUNCHED();
  const bool passes = tp.G < G;   // else the forward's single pass is still in the workspace
  for (int g0 = 0; g0 < G; g0 += tp.G) {
    const TrainPlan pp = pass_plan(tp, g0);
    const TrainBuf V = pass_bufs(tp, B, g0);
    const int32_t* npg_p = npg ? npg + g0 : nullptr;
    // the pass's planes (on the checkpoint plan: the shared block planes) and the backward scratch hold other data than
    // this pass's forward left: zero them as the forward did
    if (passes || tp.checkpoint)
      if (int e = zero_pass(pp, B, ws, npg != nullptr, st)) return e;
    // re-derive the pass's activations; its embeddings land in rowsum, which the backward rewrites before reading it
    if (passes && !tp.checkpoint)
      if (int e = train_fwd_pass<T>(p, pp, V, V.rowsum, npg_p, st)) return e;
    if (int e = train_bwd_pass<T>(p, gr, pp, V, demb + (size_t)g0 * tp.c_emb * N, npg_p, st)) return e;
  }
  return FGNN_OK;
}
