// On-device synthetic graph pairs (SURVEY 8(f) row 4): the reference draws a graph W from a generator
// (loaders/data_generator.py:39-68: "ErdosRenyi" = networkx.erdos_renyi_graph, "Regular" = networkx.random_regular_graph
// with d = int(p N), +1 if N d is odd) and a noisy copy W_noise = W (1 - N1) + (1 - W) N2 with N1 ~ ER(noise),
// N2 ~ ER(p noise / (1 - p)) (noise_erdos_renyi, data_generator.py:79-87).  Here both adjacency matrices of every pair
// are produced on the device as uint8 (G,N,N) batches -- the input format of fgnn_embed_fwd_adjacency_u8 /
// fgnn_features_from_adjacency_u8 -- from a counter-based generator (same seed -> same graphs).  Parity with the
// reference is distributional (edge density, exact degrees, flip rates, triangle counts), not bitwise.
//   Erdos-Renyi: one Bernoulli(p) per unordered vertex pair.
//   Regular:     the switch chain on simple d-regular graphs: start from a randomly relabelled circulant graph and apply
//                kSwapsPerEdge * |E| double-edge-swap proposals (u,v),(s,t) -> (u,t),(s,v), rejected when they would
//                create a loop or a parallel edge (its stationary distribution is uniform over simple d-regular graphs).
//                One CTA per graph; the n x ceil(n/32)-word adjacency bitmap sits in shared memory up to N = 1264 and in the
//                caller's workspace (L2-resident) above; the chain itself is sequential (one thread), so its time grows
//                with |E| = n d / 2 (10 |E| proposals; not measured at large n).
// N <= 4096 (vertex numbers are packed as 16-bit halves of an edge word, and the Regular workspace grows as G N^2).
#include "fgnn_common.cuh"

namespace fgnn {
namespace gen {
namespace {

constexpr int kSwapsPerEdge = 10;
constexpr int kMaxN = 4096;
constexpr size_t kSmemCap = 200 * 1024;   // dynamic shared memory the Regular kernel asks for at most

__host__ __device__ inline uint64_t mix64(uint64_t x) {   // splitmix64 finaliser
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
// uniform in [0,1) for (seed, graph, stream, unordered pair)
__device__ inline float u01(uint64_t seed, int g, int stream, int i, int j) {
  const uint64_t key = ((uint64_t)(uint32_t)g << 40) ^ ((uint64_t)(uint32_t)stream << 32) ^ ((uint64_t)(uint32_t)i << 16) ^ (uint64_t)(uint32_t)j;
  return (float)(mix64(mix64(seed) ^ key) >> 40) * (1.0f / 16777216.0f);
}
__device__ inline int graph_n(const int32_t* npg, int g, int N) { return npg ? npg[g] : N; }

// adj1 = ER(p) (when make_w) and adj2 = noisy copy of adj1; one thread per entry of the upper triangle, mirrored.
__global__ void er_pairs_kernel(uint8_t* __restrict__ adj1, uint8_t* __restrict__ adj2, int N, const int32_t* __restrict__ npg,
                                float p, float noise, float pe2, uint64_t seed, int make_w) {
  const int g = blockIdx.z;
  const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
  if (j >= N) return;
  const int n = graph_n(npg, g, N);
  const size_t ij = ((size_t)g * N + i) * N + j;
  if (i >= n || j >= n || i == j) {
    if (make_w) adj1[ij] = 0;
    adj2[ij] = 0;
    return;
  }
  const int a = min(i, j), b = max(i, j);
  uint8_t w;
  if (make_w) {
    w = u01(seed, g, 0, a, b) < p ? 1 : 0;
    adj1[ij] = w;
  } else {
    w = adj1[ij];
  }
  const bool n1 = u01(seed, g, 1, a, b) < noise, n2 = u01(seed, g, 2, a, b) < pe2;
  adj2[ij] = w ? (n1 ? 0 : 1) : (n2 ? 1 : 0);
}

struct Rng {   // sequential stream of the chain thread
  uint64_t s;
  __device__ uint32_t next() { s = mix64(s); return (uint32_t)(s >> 32); }
  __device__ uint32_t below(uint32_t n) { return (uint32_t)(((uint64_t)next() * n) >> 32); }
};

__global__ void __launch_bounds__(256, 1)
regular_kernel(uint8_t* __restrict__ adj, int N, const int32_t* __restrict__ npg, float p, uint64_t seed,
               uint32_t* __restrict__ edges_ws, long edges_per_graph, int edges_in_smem, uint32_t* __restrict__ bits_ws) {
  extern __shared__ uint32_t sm[];
  const int g = blockIdx.x;
  const int n = graph_n(npg, g, N);
  int d = (int)(p * (float)n);
  if ((n * d) & 1) d += 1;
  if (d > n - 1) d = n - 1 - (((n - 1) * n) & 1);   // cannot exceed the complete graph
  const int words = (n + 31) / 32;                   // bitmap row pitch
  // [n][words]: in shared memory, or this graph's slice of the workspace (bits_ws, row pitch ceil(N/32))
  uint32_t* bits = bits_ws ? bits_ws + (size_t)g * N * ((N + 31) / 32) : sm;
  uint16_t* perm = reinterpret_cast<uint16_t*>(bits_ws ? sm : bits + (size_t)n * words);   // [n]
  uint32_t* edges = edges_in_smem ? reinterpret_cast<uint32_t*>(perm + ((n + 1) & ~1)) : edges_ws + (size_t)g * edges_per_graph;
  for (int k = threadIdx.x; k < n * words; k += blockDim.x) bits[k] = 0u;
  if (threadIdx.x == 0) {
    Rng r{mix64(seed ^ (0xD1B54A32D192ED03ull * (uint64_t)(g + 1)))};
    for (int k = 0; k < n; ++k) perm[k] = (uint16_t)k;
    for (int k = n - 1; k > 0; --k) {               // Fisher-Yates relabelling of the circulant start
      const int q = (int)r.below((uint32_t)(k + 1));
      const uint16_t t = perm[k]; perm[k] = perm[q]; perm[q] = t;
    }
  }
  __syncthreads();
  auto set_bit = [&](int u, int v) { atomicOr(&bits[u * words + (v >> 5)], 1u << (v & 31)); atomicOr(&bits[v * words + (u >> 5)], 1u << (u & 31)); };
  auto clr_bit = [&](int u, int v) { bits[u * words + (v >> 5)] &= ~(1u << (v & 31)); bits[v * words + (u >> 5)] &= ~(1u << (u & 31)); };
  auto has = [&](int u, int v) { return (bits[u * words + (v >> 5)] >> (v & 31)) & 1u; };
  // circulant d-regular graph: i ~ i + k (k = 1 .. d/2), plus the antipode when d is odd (n is even then)
  const int half = d / 2;
  const int E = n * d / 2;
  for (int e = threadIdx.x; e < n * half; e += blockDim.x) {
    const int i = e / half, k = e % half + 1;
    const int u = perm[i], v = perm[(i + k) % n];
    set_bit(u, v);
    edges[e] = ((uint32_t)u << 16) | (uint32_t)v;
  }
  if (d & 1)
    for (int i = threadIdx.x; i < n / 2; i += blockDim.x) {
      const int u = perm[i], v = perm[i + n / 2];
      set_bit(u, v);
      edges[n * half + i] = ((uint32_t)u << 16) | (uint32_t)v;
    }
  __syncthreads();
  if (threadIdx.x == 0 && E >= 2) {
    Rng r{mix64(seed ^ (0xA24BAED4963EE407ull * (uint64_t)(g + 1)))};
    const long attempts = (long)kSwapsPerEdge * E;
    for (long a = 0; a < attempts; ++a) {
      const uint32_t e1 = r.below((uint32_t)E), e2 = r.below((uint32_t)E);
      if (e1 == e2) continue;
      uint32_t x = edges[e1], y = edges[e2];
      int u = (int)(x >> 16), v = (int)(x & 0xffffu), s = (int)(y >> 16), t = (int)(y & 0xffffu);
      if (r.next() & 1u) { const int q = s; s = t; t = q; }          // random orientation of the second edge
      if (u == t || s == v || u == s || v == t) continue;            // loop, or the swap would change nothing
      if (has(u, t) || has(s, v)) continue;                          // parallel edge
      clr_bit(u, v); clr_bit(s, t);
      bits[u * words + (t >> 5)] |= 1u << (t & 31); bits[t * words + (u >> 5)] |= 1u << (u & 31);
      bits[s * words + (v >> 5)] |= 1u << (v & 31); bits[v * words + (s >> 5)] |= 1u << (s & 31);
      edges[e1] = ((uint32_t)u << 16) | (uint32_t)t;
      edges[e2] = ((uint32_t)s << 16) | (uint32_t)v;
    }
  }
  __syncthreads();
  uint8_t* out = adj + (size_t)g * N * N;
  for (long k = threadIdx.x; k < (long)N * N; k += blockDim.x) {
    const int i = (int)(k / N), j = (int)(k % N);
    out[k] = (i < n && j < n) ? (uint8_t)has(i, j) : 0;
  }
}

size_t regular_bitmap_bytes(int n) { return (size_t)n * ((n + 31) / 32) * 4; }
bool regular_bitmap_in_smem(int n) { return regular_bitmap_bytes(n) + (size_t)((n + 1) & ~1) * 2 + 16 <= kSmemCap; }
size_t regular_edges_per_graph(int n) { return (size_t)n * n / 2 + 16; }

size_t regular_smem(int n, bool with_bitmap, bool with_edges, long E) {
  return (with_bitmap ? regular_bitmap_bytes(n) : 0) + (size_t)((n + 1) & ~1) * 2 + (with_edges ? (size_t)E * 4 : 0) + 16;
}

}  // namespace
}  // namespace gen
}  // namespace fgnn

extern "C" size_t fgnn_generate_workspace_bytes(int32_t G, int32_t N, int32_t generator) {
  using namespace fgnn::gen;
  if (generator != 1 || N < 1) return 256;
  // edge lists and, above N = 1264, adjacency bitmaps when they do not fit on chip
  const size_t bitmaps = regular_bitmap_in_smem(N) ? 0 : (size_t)G * regular_bitmap_bytes(N);
  return fgnn::align_up((size_t)G * regular_edges_per_graph(N) * sizeof(uint32_t) + bitmaps, 256);
}

extern "C" int fgnn_generate_pairs_u8(uint8_t* adj1, uint8_t* adj2, int32_t G, int32_t N, const int32_t* n_per_graph,
                                      int32_t generator, float edge_density, float noise, uint64_t seed, void* workspace,
                                      size_t workspace_bytes, void* stream) {
  using namespace fgnn;
  using namespace fgnn::gen;
  cudaStream_t st = (cudaStream_t)stream;
  FGNN_CHECK_ARG(adj1 && adj2, "null pointer");
  FGNN_CHECK_ARG(G >= 1 && G <= 65535 && N >= 2 && N <= kMaxN, "graph generator supports G <= 65535 and 2 <= N <= %d (got G=%d N=%d)",
                 kMaxN, G, N);
  FGNN_CHECK_ARG(edge_density > 0.f && edge_density < 1.f && noise >= 0.f && noise <= 1.f, "edge_density %f / noise %f out of range",
                 (double)edge_density, (double)noise);
  FGNN_CHECK_ARG(generator == 0 || generator == 1, "generator must be 0 (ErdosRenyi) or 1 (Regular); BarabasiAlbert is not built");
  const float pe2 = edge_density * noise / (1.f - edge_density);
  if (generator == 1) {
    FGNN_CHECK_ARG(workspace && workspace_bytes >= fgnn_generate_workspace_bytes(G, N, 1), "generator workspace too small");
    const long E = (long)regular_edges_per_graph(N);
    const long e_max = (long)N * ((int)(edge_density * N) + 1) / 2 + 1;
    const bool bits_in_smem = regular_bitmap_in_smem(N);
    const bool in_smem = regular_smem(N, bits_in_smem, true, e_max) <= kSmemCap;
    const size_t smem = regular_smem(N, bits_in_smem, in_smem, e_max);
    uint32_t* edges_ws = static_cast<uint32_t*>(workspace);
    uint32_t* bits_ws = bits_in_smem ? nullptr : edges_ws + (size_t)G * E;
    FGNN_CUDA(cudaFuncSetAttribute(regular_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    regular_kernel<<<G, 256, smem, st>>>(adj1, N, n_per_graph, edge_density, seed, edges_ws, E, in_smem ? 1 : 0, bits_ws);
    FGNN_LAUNCHED();
  }
  dim3 grid((N + 127) / 128, N, G);
  er_pairs_kernel<<<grid, 128, 0, st>>>(adj1, adj2, N, n_per_graph, edge_density, noise, pe2, seed, generator == 0 ? 1 : 0);
  FGNN_LAUNCHED();
  return FGNN_OK;
}
