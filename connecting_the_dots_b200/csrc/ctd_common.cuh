// Shared helpers of libctd_b200: status/error plumbing, launch accounting, small device utilities, and the winner-take-all
// rule of the stereo-matching ops (WtaRun, wta_store).
#pragma once
#include <cuda_runtime.h>
#include <limits.h>
#include <math_constants.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/ctd_b200.h"

#define CTD_API extern "C" __attribute__((visibility("default")))

namespace ctd {

// thread-local last-error message (ctd_last_error)
char* err_buf();
int fail(int code, const char* fmt, ...);
void count_launch(int n = 1);

// Stream-ordered scratch memory from a library-owned pool per device that keeps its memory between calls (no
// torch dependency, no synchronisation, usable under CUDA-graph capture).  nullptr when unavailable.
void* scratch_alloc(size_t bytes, cudaStream_t st);
void scratch_free(void* p, cudaStream_t st);

// Ticket + block-partial workspace for kernels that end with finish_masked_sums (ownership rules in ctd_core.cu): a
// static slot private to the stream (eager) or to the captured call (graph capture), else stream-ordered scratch
// memory with its ticket zeroed on the stream.  ms_acquire returns false only when no memory can be had at all;
// ms_release goes right after the kernel launch.
constexpr int MS_EAGER = 32, MS_GRAPH = 96, MS_MAXBLK = 4096;
struct MsSlot {
  unsigned* ticket;
  double* partials;
  void* scratch;
};
bool ms_acquire(size_t nblocks, cudaStream_t st, MsSlot* s);
void ms_release(MsSlot* s, cudaStream_t st);

// Check the launch that was just issued (no synchronisation, like a normal async API).
int check_launch(const char* what);

#define CTD_REQUIRE(cond, ...)                                   \
  do {                                                           \
    if (!(cond)) return ::ctd::fail(CTD_ERR_INVALID, __VA_ARGS__); \
  } while (0)

#define CTD_CUDA(call)                                                                           \
  do {                                                                                           \
    cudaError_t e__ = (call);                                                                    \
    if (e__ != cudaSuccess)                                                                      \
      return ::ctd::fail(CTD_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, \
                         __LINE__);                                                              \
  } while (0)

static inline cudaStream_t as_stream(ctd_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

__host__ __device__ __forceinline__ int clampi(int v, int lo, int hi) {
  return v < lo ? lo : (v > hi ? hi : v);
}

__host__ __device__ __forceinline__ int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// bare MUFU.RSQ (x is always >= eps > 0 where this is used)
__device__ __forceinline__ float rsqrt_approx(float x) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// read-only 128-bit load
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// the same load pinned in program order (the compiler may not sink it towards its use)
__device__ __forceinline__ float4 ldg4_volatile(const float* p) {
  float4 v;
  asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}

// Two global sums (the caller's masked-mean numerator and denominator, model/networks.py:377) produced by a kernel
// that has other work to do: every thread of the block (a whole number of warps) passes its share, the block's partial goes to
// `partials[2 * block]`, and the last block to arrive (ticket counter, zero before the launch) adds all partials in
// index order in fp64 and writes out2 -- deterministic for a given grid, no floating-point atomics.
__device__ __forceinline__ void finish_masked_sums(double num, double den, double* __restrict__ partials,
                                                   unsigned* __restrict__ ticket, float* __restrict__ out2) {
  __shared__ double s_num[32], s_den[32];  // one per warp, up to 1024 threads
  __shared__ bool s_last;
  const unsigned bid = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
  const unsigned nblocks = gridDim.x * gridDim.y * gridDim.z;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    num += __shfl_xor_sync(0xffffffffu, num, o);
    den += __shfl_xor_sync(0xffffffffu, den, o);
  }
  if ((threadIdx.x & 31) == 0) {
    s_num[threadIdx.x >> 5] = num;
    s_den[threadIdx.x >> 5] = den;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
      a += s_num[w];
      b += s_den[w];
    }
    partials[2 * bid] = a;
    partials[2 * bid + 1] = b;
    __threadfence();
    s_last = atomicAdd(ticket, 1u) == nblocks - 1;
  }
  __syncthreads();
  if (s_last) {  // block-uniform: the whole block adds the partials (fixed assignment and order)
    __threadfence();
    double a = 0.0, b = 0.0;
    for (unsigned i = threadIdx.x; i < nblocks; i += blockDim.x) {
      a += __ldcg(partials + 2 * i);
      b += __ldcg(partials + 2 * i + 1);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    __syncthreads();  // s_num / s_den of the first phase have been consumed
    if ((threadIdx.x & 31) == 0) {
      s_num[threadIdx.x >> 5] = a;
      s_den[threadIdx.x >> 5] = b;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      a = 0.0;
      b = 0.0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
        a += s_num[w];
        b += s_den[w];
      }
      out2[0] = (float)a;
      out2[1] = (float)b;
      *ticket = 0;
    }
  }
}

__device__ __forceinline__ bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// [a, a + na) and [b, b + nb) (bytes) share no byte; a null pointer or an empty range overlaps nothing
inline bool ranges_disjoint(const void* a, size_t na, const void* b, size_t nb) {
  const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b;
  return !a || !b || na == 0 || nb == 0 || x + na <= y || y + nb <= x;
}

// A kernel launched with more than 48 KB of dynamic shared memory has to opt in.  The attribute belongs to the device,
// so it is set on every call (a process may use several GPUs).
template <typename Kernel>
int raise_smem_limit(Kernel kernel, size_t bytes, const char* op) {
  if (bytes > 48 * 1024 && cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
    return fail(CTD_ERR_CUDA, "%s: cannot raise the shared-memory limit to %zu bytes", op, bytes);
  return CTD_OK;
}

// the value below every other: -inf for floating point, INT_MIN for int
template <typename T>
__device__ __forceinline__ T lowest();
template <>
__device__ __forceinline__ float lowest<float>() { return -CUDART_INF_F; }
template <>
__device__ __forceinline__ double lowest<double>() { return -CUDART_INF; }
template <>
__device__ __forceinline__ int lowest<int>() { return INT_MIN; }

// Winner-take-all over scores fed in order d = 0, 1, ...: best = the largest score, bd = the first d that reached it
// (d*), cm and cp = the scores at d* - 1 and d* + 1 (cp is caught on the step after d* while d* stands).  The lowest()
// sentinels make d = 0 an ordinary step: any score beats them, and a column of lowest() keeps d* = 0.  Selects only.
template <typename V>
struct WtaRun {
  V best, prev, cm, cp;
  int bd;
  __device__ __forceinline__ void init() {
    best = prev = lowest<V>();
    cm = cp = 0;
    bd = 0;
  }
  // returns whether v is a new best (bd and best are then d and v; read bd before the call for the old d*)
  __device__ __forceinline__ bool step(V v, int d) {
    cp = d - 1 == bd ? v : cp;
    const bool nb = v > best;
    cm = nb ? prev : cm;
    bd = nb ? d : bd;
    best = nb ? v : best;
    prev = v;
    return nb;
  }
};

// three-point parabola through the scores at d* - 1, d*, d* + 1: vertex offset in [-0.5, 0.5], 0 unless the peak is strict
// (den < 0); fp64 with disparity_from_volume's operation order
__device__ __forceinline__ double wta_subpixel(double cm, double c0, double cp) {
  const double den = cm - 2.0 * c0 + cp;
  if (!(den < 0.0)) return 0.0;
  return fmin(fmax((cm - cp) / (2.0 * den), -0.5), 0.5);
}

// The winner-take-all outputs of pixel px (either pointer may be null): score = c0, the score at d* = bd, and disp = d*
// plus, with subpixel, the parabola's offset through cm, c0, cp where 0 < d* < lim - 1 (lim: the number of disparities
// the pixel has).
template <typename T>
__device__ __forceinline__ void wta_store(T* disp, T* score, int64_t px, int bd, T c0, T cm, T cp, int lim, int subpixel) {
  if (score) score[px] = c0;
  if (disp) {
    const double delta = subpixel && bd > 0 && bd < lim - 1 ? wta_subpixel((double)cm, (double)c0, (double)cp) : 0.0;
    disp[px] = (T)((double)bd + delta);
  }
}

}  // namespace ctd
