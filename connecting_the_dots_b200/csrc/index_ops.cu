// ProjNN, NN and CrossCheck for sm_100a: the bit-exact index ops.
//
// Reference semantics: torchext/ext/ext.h:65-117 (ProjNNFunctor), :13-46 (NNFunctor<T,3>),
// :48-63 (CrossCheckFunctor).  The reference's CPU build contains no fused multiply-adds, so this
// file is compiled with -fmad=false and keeps the reference's association order; float->int
// conversions follow x86 cvttsd2si (NaN / out of range -> INT_MIN), which is what the CPU extension
// does and what makes non-finite projections come out as -1.
#include <algorithm>

#include "ctd_common.cuh"

namespace ctd {

extern int g_force_generic;

// ------------------------------------------------------------------------------------------
// ProjNN
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int x86_double_to_int(double v) {
  if (!(v > -2147483649.0 && v < 2147483648.0)) return INT32_MIN;
  return (int)v;
}

constexpr int PN_THREADS = 256;

template <typename T>
__global__ void __launch_bounds__(PN_THREADS)
proj_nn_kernel(const T* __restrict__ xyz0, const T* __restrict__ xyz1, const T* __restrict__ K,
               int64_t* __restrict__ out, int64_t total, int H, int W, int ps) {
  __shared__ T pts[PN_THREADS * 3];
  const int tid = threadIdx.x;
  const int64_t i0 = (int64_t)blockIdx.x * PN_THREADS;
  const int64_t nvalid = min((int64_t)PN_THREADS, total - i0);
  // coalesced staging of this block's 256 query points (channels-last xyz: 3 values per pixel)
  for (int j = tid; j < nvalid * 3; j += PN_THREADS) pts[j] = __ldg(xyz0 + i0 * 3 + j);
  T k[9];
#pragma unroll
  for (int j = 0; j < 9; ++j) k[j] = __ldg(K + j);
  __syncthreads();
  if (tid >= nvalid) return;
  const int64_t i = i0 + tid;
  const int64_t hw = (int64_t)H * W;
  const int64_t b = i / hw;
  const T x = pts[tid * 3 + 0], y = pts[tid * 3 + 1], z = pts[tid * 3 + 2];
  const T den = k[6] * x + k[7] * y + k[8] * z;
  const T u = (k[0] * x + k[1] * y + k[2] * z) / den;
  const T v = (k[3] * x + k[4] * y + k[5] * z) / den;
  const int u0 = x86_double_to_int((double)u + 0.5);
  const int v0 = x86_double_to_int((double)v + 0.5);
  int64_t best = -1;
  T best_d = (T)1e9;
  const int half = ps / 2;
  for (int pv = 0; pv < ps; ++pv) {
    const int v1 = (int)((int64_t)(v0 + pv) - half);
    if (v1 < 0 || v1 >= H) continue;
    for (int pu = 0; pu < ps; ++pu) {
      const int u1 = (int)((int64_t)(u0 + pu) - half);
      if (u1 < 0 || u1 >= W) continue;
      const int64_t j = (b * H + v1) * W + u1;
      const T* q = xyz1 + j * 3;
      const T qx = __ldg(q), qy = __ldg(q + 1), qz = __ldg(q + 2);
      const T dd = (x - qx) * (x - qx) + (y - qy) * (y - qy) + (z - qz) * (z - qz);
      if (dd < best_d) {
        best_d = dd;
        best = j;
      }
    }
  }
  out[i] = best;
}

// ------------------------------------------------------------------------------------------
// NN (brute force, 3-D)
// ------------------------------------------------------------------------------------------
constexpr int NN_THREADS = 128;
constexpr int NN_QPT = 4;      // queries per thread
constexpr int NN_TILE = 1024;  // in1 points staged per shared-memory tile

// SPLIT: in1 is divided over blockIdx.y; partial minima meet in `out` (pre-set to all ones = -1) as
// (distance bits << 32 | index) through atomicMin, so equal distances resolve to the lowest index
// exactly like the reference's strict '<' scan.  Only used for float (distance bits fit 32).
template <typename T, bool SPLIT>
__global__ void __launch_bounds__(NN_THREADS)
nn_kernel(const T* __restrict__ in0, const T* __restrict__ in1, int64_t* __restrict__ out, int64_t N0,
          int64_t N1, int64_t chunk) {
  __shared__ __align__(16) T tile[NN_TILE * 4];
  const int tid = threadIdx.x;
  const int64_t q0 = ((int64_t)blockIdx.x * NN_THREADS + tid) * NN_QPT;
  T qx[NN_QPT], qy[NN_QPT], qz[NN_QPT], best_d[NN_QPT];
  int64_t best[NN_QPT];
#pragma unroll
  for (int m = 0; m < NN_QPT; ++m) {
    const int64_t q = min(q0 + m, N0 - 1);
    qx[m] = __ldg(in0 + q * 3 + 0);
    qy[m] = __ldg(in0 + q * 3 + 1);
    qz[m] = __ldg(in0 + q * 3 + 2);
    best_d[m] = (T)1e9;
    best[m] = -1;
  }
  const int64_t c0 = (int64_t)blockIdx.y * chunk, c1 = min(N1, c0 + chunk);
  for (int64_t t0 = c0; t0 < c1; t0 += NN_TILE) {
    const int cnt = (int)min((int64_t)NN_TILE, c1 - t0);
    __syncthreads();
    for (int j = tid; j < cnt * 3; j += NN_THREADS) tile[(j / 3) * 4 + j % 3] = __ldg(in1 + t0 * 3 + j);
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < cnt; ++j) {
      const T bx = tile[j * 4 + 0], by = tile[j * 4 + 1], bz = tile[j * 4 + 2];
#pragma unroll
      for (int m = 0; m < NN_QPT; ++m) {
        const T dx = qx[m] - bx, dy = qy[m] - by, dz = qz[m] - bz;
        const T dist = dx * dx + dy * dy + dz * dz;  // ((0 + dx^2) + dy^2) + dz^2, no FMA
        if (dist < best_d[m]) {
          best_d[m] = dist;
          best[m] = t0 + j;
        }
      }
    }
  }
#pragma unroll
  for (int m = 0; m < NN_QPT; ++m) {
    if (q0 + m >= N0) continue;
    if (SPLIT) {
      if (best[m] >= 0) {
        const unsigned long long key =
            ((unsigned long long)__float_as_uint((float)best_d[m]) << 32) | (unsigned long long)best[m];
        atomicMin(reinterpret_cast<unsigned long long*>(out) + q0 + m, key);
      }
    } else {
      out[q0 + m] = best[m];
    }
  }
}

__global__ void nn_unpack_kernel(int64_t* out, int64_t N0) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N0) return;
  const int64_t v = out[i];
  if (v != -1) out[i] = v & 0xffffffffll;
}

// ------------------------------------------------------------------------------------------
// CrossCheck
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint8_t crosscheck_one(int64_t a, int64_t i, const int64_t* __restrict__ in1, int64_t N1) {
  const int j = (int)(uint32_t)(uint64_t)a;  // `int idx1 = in0[idx0]`: int64 -> int32 truncation
  if (j < 0 || j >= N1) return 0;
  const int64_t bck = __ldg(in1 + j);
  return (uint8_t)(bck >= 0 && bck == i);
}

__global__ void __launch_bounds__(256)
crosscheck_kernel(const int64_t* __restrict__ in0, const int64_t* __restrict__ in1, uint8_t* __restrict__ out,
                  int64_t N0, int64_t N1, int vec) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i >= N0) return;
  if (vec && i + 3 < N0) {
    const longlong2 a = __ldg(reinterpret_cast<const longlong2*>(in0 + i));
    const longlong2 b = __ldg(reinterpret_cast<const longlong2*>(in0 + i + 2));
    uchar4 r;
    r.x = crosscheck_one(a.x, i + 0, in1, N1);
    r.y = crosscheck_one(a.y, i + 1, in1, N1);
    r.z = crosscheck_one(b.x, i + 2, in1, N1);
    r.w = crosscheck_one(b.y, i + 3, in1, N1);
    *reinterpret_cast<uchar4*>(out + i) = r;
  } else {
    for (int64_t k = i; k < min(i + 4, N0); ++k) out[k] = crosscheck_one(__ldg(in0 + k), k, in1, N1);
  }
}

// Fixed patch size (1, 2, 3, 5, 7, 9), images below 2^31 / 3 pixels: the PS x PS scan is unrolled, the in-image
// test of every candidate is done up front and all its loads are issued before the first comparison (PS^2 gathers
// in flight instead of one), indices are 32-bit inside the image.  Same arithmetic and scan order as above: an
// absent candidate gets distance +inf, which never passes the strict `<` against 1e9 or anything below it.
template <typename T, int PS>
__global__ void __launch_bounds__(PN_THREADS)
proj_nn_fixed_kernel(const T* __restrict__ xyz0, const T* __restrict__ xyz1, const T* __restrict__ K,
                     int64_t* __restrict__ out, int64_t total, int H, int W) {
  __shared__ T pts[PN_THREADS * 3];
  const int tid = threadIdx.x;
  const int64_t i0 = (int64_t)blockIdx.x * PN_THREADS;
  const int nvalid = (int)min((int64_t)PN_THREADS, total - i0);
  for (int j = tid; j < nvalid * 3; j += PN_THREADS) pts[j] = __ldg(xyz0 + i0 * 3 + j);
  T k[9];
#pragma unroll
  for (int j = 0; j < 9; ++j) k[j] = __ldg(K + j);
  __syncthreads();
  if (tid >= nvalid) return;
  const int64_t i = i0 + tid;
  const unsigned hw = (unsigned)H * (unsigned)W;
  const int64_t b = i / hw;
  const T* img1 = xyz1 + b * (int64_t)hw * 3;
  const T x = pts[tid * 3 + 0], y = pts[tid * 3 + 1], z = pts[tid * 3 + 2];
  const T den = k[6] * x + k[7] * y + k[8] * z;
  const T u = (k[0] * x + k[1] * y + k[2] * z) / den;
  const T v = (k[3] * x + k[4] * y + k[5] * z) / den;
  const int u0 = x86_double_to_int((double)u + 0.5);
  const int v0 = x86_double_to_int((double)v + 0.5);
  constexpr int half = PS / 2;
  // INT_MIN (x86's answer to NaN / out of range) must stay far outside the image after the offsets are added
  const int ub = u0 < -(1 << 30) ? -(1 << 30) : u0 - half, vb = v0 < -(1 << 30) ? -(1 << 30) : v0 - half;
  T best_d = (T)1e9;
  int best = -1;
  if (ub >= 0 && vb >= 0 && ub + PS <= W && vb + PS <= H) {
    // The whole patch lies inside the image (all but the queries that project next to the border): no per-candidate
    // tests, one row pointer per patch row with compile-time offsets behind it, and the winner remembered by its
    // position in the scan (a constant per candidate) instead of its pixel index.  Same scan order, same strict <.
    const T* row = img1 + (unsigned)(vb * W + ub) * 3u;
    int bestc = -1;
#pragma unroll
    for (int pv = 0; pv < PS; ++pv) {
      T q[3 * PS];
#pragma unroll
      for (int j = 0; j < 3 * PS; ++j) q[j] = __ldg(row + j);
#pragma unroll
      for (int pu = 0; pu < PS; ++pu) {
        const T dd = (x - q[3 * pu]) * (x - q[3 * pu]) + (y - q[3 * pu + 1]) * (y - q[3 * pu + 1]) + (z - q[3 * pu + 2]) * (z - q[3 * pu + 2]);
        if (dd < best_d) {
          best_d = dd;
          bestc = pv * PS + pu;
        }
      }
      row += (unsigned)W * 3u;
    }
    if (bestc >= 0) best = (vb + bestc / PS) * W + (ub + bestc % PS);
  } else {
#pragma unroll
    for (int pv = 0; pv < PS; ++pv) {
      const int v1 = vb + pv;
      const bool vok = v1 >= 0 && v1 < H;
      T qx[PS], qy[PS], qz[PS];
#pragma unroll
      for (int pu = 0; pu < PS; ++pu) {
        const int u1 = ub + pu;
        const bool ok = vok && u1 >= 0 && u1 < W;
        const T* q = img1 + (unsigned)(ok ? v1 * W + u1 : 0) * 3u;
        qx[pu] = ok ? __ldg(q) : (T)INFINITY;
        qy[pu] = ok ? __ldg(q + 1) : (T)0;
        qz[pu] = ok ? __ldg(q + 2) : (T)0;
      }
#pragma unroll
      for (int pu = 0; pu < PS; ++pu) {
        const T dd = (x - qx[pu]) * (x - qx[pu]) + (y - qy[pu]) * (y - qy[pu]) + (z - qz[pu]) * (z - qz[pu]);
        if (dd < best_d) {
          best_d = dd;
          best = (vb + pv) * W + (ub + pu);
        }
      }
    }
  }
  out[i] = best < 0 ? (int64_t)-1 : b * (int64_t)hw + best;
}

template <typename T>
static int proj_nn_impl(const T* xyz0, const T* xyz1, const T* K, int64_t* out, int64_t B, int64_t H, int64_t W,
                        int ps, cudaStream_t st) {
  CTD_REQUIRE(B >= 0 && H >= 0 && W >= 0, "proj_nn: negative size");
  CTD_REQUIRE(H <= INT32_MAX && W <= INT32_MAX, "proj_nn: image too large");
  CTD_REQUIRE(ps >= 0 && ps <= 4096, "proj_nn: patch_size %d out of range", ps);
  const int64_t total = B * H * W;
  if (total == 0) return CTD_OK;
  CTD_REQUIRE(xyz0 && xyz1 && K && out, "proj_nn: null pointer");
  CTD_REQUIRE(cdiv(total, PN_THREADS) <= INT32_MAX, "proj_nn: too many pixels");
  const unsigned grid = (unsigned)cdiv(total, PN_THREADS);
  const bool fixed = !g_force_generic && H * W < ((int64_t)1 << 31) / 3;
#define CTD_PN_CASE(PS)                                                                                             \
  case PS:                                                                                                          \
    proj_nn_fixed_kernel<T, PS><<<grid, PN_THREADS, 0, st>>>(xyz0, xyz1, K, out, total, (int)H, (int)W);           \
    count_launch();                                                                                                 \
    return check_launch("proj_nn(fixed)");
  if (fixed) switch (ps) {
      CTD_PN_CASE(1)
      CTD_PN_CASE(2)
      CTD_PN_CASE(3)
      CTD_PN_CASE(5)
      CTD_PN_CASE(7)
      CTD_PN_CASE(9)
      default: break;
    }
#undef CTD_PN_CASE
  proj_nn_kernel<T><<<grid, PN_THREADS, 0, st>>>(xyz0, xyz1, K, out, total, (int)H, (int)W, ps);
  count_launch();
  return check_launch("proj_nn");
}

template <typename T>
static int nn_impl(const T* in0, const T* in1, int64_t* out, int64_t N0, int64_t N1, cudaStream_t st) {
  CTD_REQUIRE(N0 >= 0 && N1 >= 0, "nn: negative size");
  if (N0 == 0) return CTD_OK;
  CTD_REQUIRE(in0 && out && (in1 || N1 == 0), "nn: null pointer");
  const int64_t qtiles = cdiv(N0, NN_THREADS * NN_QPT);
  CTD_REQUIRE(qtiles <= INT32_MAX, "nn: too many queries");
  int64_t nchunks = 1;
  if (sizeof(T) == 4 && N1 < ((int64_t)1 << 32)) {
    nchunks = std::min<int64_t>(std::max<int64_t>(1, (2 * 148 + qtiles - 1) / qtiles), std::max<int64_t>(1, N1 / NN_TILE));
    nchunks = std::min<int64_t>(nchunks, 65535);
  }
  if (nchunks > 1) {
    const int64_t chunk = cdiv(cdiv(N1, nchunks), NN_TILE) * NN_TILE;
    nchunks = cdiv(N1, chunk);
    CTD_CUDA(cudaMemsetAsync(out, 0xFF, (size_t)N0 * sizeof(int64_t), st));
    nn_kernel<T, true><<<dim3((unsigned)qtiles, (unsigned)nchunks), NN_THREADS, 0, st>>>(in0, in1, out, N0, N1, chunk);
    nn_unpack_kernel<<<(unsigned)cdiv(N0, 256), 256, 0, st>>>(out, N0);
    count_launch(2);
  } else {
    nn_kernel<T, false><<<dim3((unsigned)qtiles, 1), NN_THREADS, 0, st>>>(in0, in1, out, N0, N1, std::max<int64_t>(N1, 1));
    count_launch();
  }
  return check_launch("nn");
}

}  // namespace ctd

using namespace ctd;

CTD_API int ctd_proj_nn_f32(const float* xyz0, const float* xyz1, const float* K, int64_t* out, int64_t B,
                               int64_t H, int64_t W, int ps, ctd_stream_t s) {
  return proj_nn_impl<float>(xyz0, xyz1, K, out, B, H, W, ps, as_stream(s));
}
CTD_API int ctd_proj_nn_f64(const double* xyz0, const double* xyz1, const double* K, int64_t* out, int64_t B,
                               int64_t H, int64_t W, int ps, ctd_stream_t s) {
  return proj_nn_impl<double>(xyz0, xyz1, K, out, B, H, W, ps, as_stream(s));
}
CTD_API int ctd_nn_f32(const float* in0, const float* in1, int64_t* out, int64_t N0, int64_t N1, ctd_stream_t s) {
  return nn_impl<float>(in0, in1, out, N0, N1, as_stream(s));
}
CTD_API int ctd_nn_f64(const double* in0, const double* in1, int64_t* out, int64_t N0, int64_t N1, ctd_stream_t s) {
  return nn_impl<double>(in0, in1, out, N0, N1, as_stream(s));
}
CTD_API int ctd_crosscheck(const int64_t* in0, const int64_t* in1, uint8_t* out, int64_t N0, int64_t N1,
                              ctd_stream_t s) {
  CTD_REQUIRE(N0 >= 0 && N1 >= 0, "crosscheck: negative size");
  if (N0 == 0) return CTD_OK;
  CTD_REQUIRE(in0 && out && (in1 || N1 == 0), "crosscheck: null pointer");
  const int vec = ((reinterpret_cast<uintptr_t>(in0) & 15) == 0) && ((reinterpret_cast<uintptr_t>(out) & 3) == 0);
  const int64_t blocks = cdiv(cdiv(N0, 4), 256);
  CTD_REQUIRE(blocks <= INT32_MAX, "crosscheck: too many elements");
  crosscheck_kernel<<<(unsigned)blocks, 256, 0, as_stream(s)>>>(in0, in1, out, N0, N1, vec);
  count_launch();
  return check_launch("crosscheck");
}
