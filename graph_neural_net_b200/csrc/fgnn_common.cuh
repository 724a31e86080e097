// Shared host/device helpers for libfgnn_b200 (internal; the public ABI is include/fgnn_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>
#include "../../include/fgnn_b200.h"

namespace fgnn {

extern thread_local char g_last_error[512];
extern thread_local int64_t g_launches;

inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap);
  va_end(ap);
  return code;
}

#define FGNN_CHECK_ARG(cond, ...) \
  do {                            \
    if (!(cond)) return ::fgnn::fail(FGNN_ERR_INVALID, __VA_ARGS__); \
  } while (0)

#define FGNN_CUDA(call)                                                                      \
  do {                                                                                       \
    cudaError_t e__ = (call);                                                                \
    if (e__ != cudaSuccess)                                                                  \
      return ::fgnn::fail(FGNN_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                          __FILE__, __LINE__);                                               \
  } while (0)

// every kernel launch in the library goes through this so gpu_launches is an honest count
#define FGNN_LAUNCHED()                                                                      \
  do {                                                                                       \
    ++::fgnn::g_launches;                                                                    \
    cudaError_t e__ = cudaGetLastError();                                                    \
    if (e__ != cudaSuccess)                                                                  \
      return ::fgnn::fail(FGNN_ERR_CUDA, "kernel launch failed: %s (%s:%d)",                 \
                          cudaGetErrorString(e__), __FILE__, __LINE__);                      \
  } while (0)

// Optional per-kernel-class device timing (CUDA events on the launching stream); off by default.
namespace prof {
enum Kind { kMlp = 0, kMatmul = 1, kStats = 2, kGlue = 3, kNumKinds = 4 };
void begin(Kind k, cudaStream_t st);
void end(Kind k, cudaStream_t st);
}  // namespace prof

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// How a kernel whose CTAs produce partial sums of the same value combines them (DESIGN.md §7.1).
//   AtomicSum   (default) each partial is added with a floating-point atomic, in whatever order the CTAs finish;
//   OrderedSum  (FGNN_DETERMINISTIC) each partial is stored to its own record, at an index fixed by the launch, and a
//               reduce kernel sums the records in a fixed order: the result does not depend on scheduling.
// The tag is a template argument of every such kernel, so the modes are separate instantiations: the default ones keep
// their code, and the OrderedSum ones contain no floating-point atomic (tests/test_deterministic_cpu.py checks the SASS).
struct AtomicSum { static constexpr bool kOrdered = false; };
struct OrderedSum { static constexpr bool kOrdered = true; };

namespace {
// out[o][e] = (out[o][e] +) sum_{r < nrec} rec[o][r][e], r ascending, in double: the fixed-order sum of OrderedSum
// records.  o < nout / w, e < w.
template <typename R, typename O>
__global__ void sum_records_kernel(const R* __restrict__ rec, O* __restrict__ out, long nout, int nrec, int w, int accumulate) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= nout) return;
  const R* p = rec + (idx / w) * nrec * w + idx % w;
  double s = 0.0;
  for (int r = 0; r < nrec; ++r) s += (double)p[(long)r * w];
  out[idx] = accumulate ? (O)(out[idx] + (O)s) : (O)s;
}

template <typename R, typename O>
int sum_records(const R* rec, O* out, long nout, int nrec, int w, bool accumulate, cudaStream_t st) {
  if (nout <= 0) return FGNN_OK;
  sum_records_kernel<R, O><<<(unsigned)((nout + 255) / 256), 256, 0, st>>>(rec, out, nout, nrec, w, accumulate ? 1 : 0);
  FGNN_LAUNCHED();
  return FGNN_OK;
}
}  // namespace

// Bump allocator over a caller-provided workspace.
struct Arena {
  char* base;
  size_t size;
  size_t off = 0;
  bool dry;  // dry run: only measure
  Arena(void* p, size_t n) : base(static_cast<char*>(p)), size(n), dry(p == nullptr) {}
  template <typename T>
  T* take(size_t count, size_t align = 256) {
    off = align_up(off, align);
    T* r = dry ? nullptr : reinterpret_cast<T*>(base + off);
    off += count * sizeof(T);
    return r;
  }
  bool ok() const { return dry || off <= size; }
};

}  // namespace fgnn
