// Semi-global matching over a [B,D,H,W] score volume (ctd_sgm_*) for sm_100a.
//
// Definition (include/ctd_b200.h states it in full): for each path direction r = (dy, dx) and q = p - r,
//   L_r(p, d) = V(p, d)                                   if q is outside the image (a path starts),
//   L_r(p, d) = V(p, d) + (m - M)                         otherwise, with M = max_k L_r(q, k) and
//   m = max(L_r(q, d), L_r(q, d-1) - p1, L_r(q, d+1) - p1, M - p2) over the neighbours inside [0, D).
// A = (((L_0 + L_1) + L_2) + ...) in the fixed path order (0,+1) (0,-1) (+1,0) (-1,0) [(+1,+1) (+1,-1) (-1,+1) (-1,-1)].
// There is no multiply and max is exact, so every kernel below reproduces the definition bit for bit.
//
// Kernels: one sweep of a path along a line is sequential; lines are independent.  A line's D values live in the
// registers of a group of G lanes, K consecutive disparities per lane (lane g holds d = g*K .. g*K + K-1; slots past D hold
// -inf, which every max ignores).  The neighbours d-1 and d+1 of the group's edge slots come from one shuffle each and M
// is a shuffle reduction over the group.
//   * sgm_horizontal: paths 0 and 1.  One warp (G = 32) per image row.  In [B,D,H,W] a pixel's D values are H*W apart, so
//     the row passes through per-warp shared slabs [D][WT] in tiles of WT columns: coalesced cp.async row copies in (the
//     next tile's while the current one is swept), the recurrence over the tile's columns in place, coalesced stores out.  Path 1 runs in the same warp right after path 0,
//     so the row's slice of A it read-modify-writes (D*W values) is still in L2.
//   * sgm_lines: one vertical or diagonal path.  Lines are sheared columns k = w - dx*dy*h: a diagonal line's predecessor
//     lies on the same line, so a line needs no data from its neighbours, and the 32/G lines of a warp read adjacent w.
//     Each step loads the next row's V and A before it computes the current one.  The last pass in path order also takes
//     the winner-take-all disparity and score of A: the first maximum by a reduction over the group, stored through
//     wta_store (ctd_common.cuh) with disparity_from_volume's fp64 sub-pixel offset.
// No atomics, no scratch memory, no host synchronisation: every call is capture-safe and its result does not depend on
// the launch configuration (every value is computed by the same operations in the same order whatever G, K or WT are).
#include <cuda_pipeline.h>

#include <algorithm>
#include <cmath>

#include "ctd_common.cuh"

namespace ctd {

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int SGM_MAX_D = 1024;      // 32 lanes x 32 registers per line
constexpr int SGM_HWARPS = 4;        // rows (warps) per sgm_horizontal CTA
constexpr int SGM_SLAB_BYTES = 16384;  // shared slabs per warp (two tiles)
constexpr int SGM_LTHREADS = 256;

// One step of the recurrence for the line held by a group of G lanes (this lane is g).  L holds L_r(q, .) and M its maximum
// on entry, L_r(p, .) and its maximum on exit; start: q is outside the image.  Every lane of the warp calls it.
template <typename T, int K>
__device__ __forceinline__ void sgm_step(T (&L)[K], const T (&v)[K], T& M, bool start, int g, int G, T p1, T p2) {
  const T ninf = lowest<T>();
  const T lo = __shfl_up_sync(FULL, L[K - 1], 1, G);  // L(q, g*K - 1)
  const T hi = __shfl_down_sync(FULL, L[0], 1, G);    // L(q, g*K + K)
  const T mp2 = M - p2;
  T prev = g == 0 ? ninf : lo;
  T mx = ninf;
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const T next = j + 1 < K ? L[j + 1] : (g == G - 1 ? ninf : hi);
    const T m = fmax(fmax(L[j], prev - p1), fmax(next - p1, mp2));
    prev = L[j];
    L[j] = start ? v[j] : v[j] + (m - M);
    mx = fmax(mx, L[j]);
  }
  for (int o = 1; o < G; o <<= 1) mx = fmax(mx, __shfl_xor_sync(FULL, mx, o, G));
  M = mx;
}

// slab column of (d, c): XOR-swizzled so that both the row loads (fixed d, c across lanes) and the recurrence's reads
// (fixed c, d = g*K + j across lanes) hit distinct banks
template <int K>
__device__ __forceinline__ int slab_col(int d, int c, int WT) { return c ^ ((d / K) & (WT - 1)); }

// paths (0,+1) and (0,-1) of one image row per warp: A = L0, then A = A + L1.  Two slabs a warp: the next tile's V is
// copied in with cp.async while the recurrence runs over the current one.
template <typename T, int K>
__global__ void __launch_bounds__(32 * SGM_HWARPS)
sgm_horizontal(const T* __restrict__ vol, T* __restrict__ agg, int64_t B, int D, int H, int W, int WT, T p1, T p2) {
  extern __shared__ __align__(16) unsigned char sgm_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T* slabs = reinterpret_cast<T*>(sgm_smem) + (size_t)warp * 2 * D * WT;
  const T ninf = lowest<T>();
  const int64_t plane = (int64_t)H * W, nrows = B * H;
  const int ntiles = (W + WT - 1) / WT, wshift = __ffs(WT) - 1;
  for (int64_t row = (int64_t)blockIdx.x * SGM_HWARPS + warp; row < nrows; row += (int64_t)gridDim.x * SGM_HWARPS) {
    const int64_t b = row / H, off = b * D * plane + (row - b * H) * W;
    const T* vrow = vol + off;
    T* arow = agg + off;
    for (int pass = 0; pass < 2; ++pass) {
      // tile t of this pass covers columns [w0, w0 + wn); pass 1 walks the tiles right to left
      auto fetch = [&](int t) {
        if (t < ntiles) {
          T* slab = slabs + (t & 1) * D * WT;
          const int w0 = (pass == 0 ? t : ntiles - 1 - t) * WT, wn = min(WT, W - w0);
          for (int i = lane; i < D * WT; i += 32) {
            const int d = i >> wshift, c = i & (WT - 1);
            if (c < wn) __pipeline_memcpy_async(slab + d * WT + slab_col<K>(d, c, WT), vrow + d * plane + w0 + c, sizeof(T));
          }
        }
        __pipeline_commit();
      };
      T L[K], M = 0;
#pragma unroll
      for (int j = 0; j < K; ++j) L[j] = ninf;
      fetch(0);
      for (int t = 0; t < ntiles; ++t) {
        fetch(t + 1);  // the slab it fills was released by tile t - 1's last __syncwarp
        __pipeline_wait_prior(1);
        __syncwarp();
        T* slab = slabs + (t & 1) * D * WT;
        const int w0 = (pass == 0 ? t : ntiles - 1 - t) * WT, wn = min(WT, W - w0);
        for (int i = 0; i < wn; ++i) {
          const int c = pass == 0 ? i : wn - 1 - i;
          T v[K];
#pragma unroll
          for (int j = 0; j < K; ++j) {
            const int d = lane * K + j;
            v[j] = d < D ? slab[d * WT + slab_col<K>(d, c, WT)] : ninf;
          }
          sgm_step<T, K>(L, v, M, t == 0 && i == 0, lane, 32, p1, p2);
#pragma unroll
          for (int j = 0; j < K; ++j) {
            const int d = lane * K + j;
            if (d < D) slab[d * WT + slab_col<K>(d, c, WT)] = L[j];
          }
        }
        __syncwarp();
#pragma unroll 16
        for (int i = lane; i < D * WT; i += 32) {
          const int d = i >> wshift, c = i & (WT - 1);
          if (c < wn) {
            T* a = arow + d * plane + w0 + c;
            const T x = slab[d * WT + slab_col<K>(d, c, WT)];
            *a = pass == 0 ? x : *a + x;  // L0 + L1 (addition commutes exactly)
          }
        }
        __syncwarp();
      }
    }
  }
}

// one vertical or diagonal path (dy = +-1): A = A + L_r; WTA: also disp / score of the final A (either may be null)
template <typename T, int K, bool WTA>
__global__ void __launch_bounds__(SGM_LTHREADS)
sgm_lines(const T* __restrict__ vol, T* __restrict__ agg, T* __restrict__ disp, T* __restrict__ score, int64_t B, int D,
          int H, int W, int dy, int dx, int G, T p1, T p2, int subpixel) {
  const T ninf = lowest<T>();
  const int s = dx * dy;  // pixel (h, w) lies on line k = w - s*h
  const int64_t plane = (int64_t)H * W;
  const int64_t nk = W + (s != 0 ? (int64_t)H - 1 : 0), kmin = s > 0 ? -(int64_t)(H - 1) : 0;
  const int lane = threadIdx.x & 31, g = lane & (G - 1), lpw = 32 / G;
  const int64_t nwarps = cdiv(B * nk, lpw);
  for (int64_t wi = ((int64_t)blockIdx.x * SGM_LTHREADS + threadIdx.x) >> 5; wi < nwarps;
       wi += (int64_t)gridDim.x * (SGM_LTHREADS / 32)) {
    const int64_t line = wi * lpw + lane / G;
    const int64_t b = line / nk;
    const int64_t k = kmin + (line - b * nk);
    // rows of the line inside the image: 0 <= k + s*h < W
    int hlo = H, hhi = -1;
    if (line < B * nk) {
      const int64_t lo = s > 0 ? -k : (s < 0 ? k - W + 1 : 0), hi = s > 0 ? W - 1 - k : (s < 0 ? k : H - 1);
      hlo = (int)(lo > 0 ? lo : 0);
      hhi = (int)(hi < H - 1 ? hi : H - 1);
    }
    const int wlo = __reduce_min_sync(FULL, hlo), whi = __reduce_max_sync(FULL, hhi);
    if (wlo > whi) continue;  // warp-uniform
    const int hstart = dy > 0 ? hlo : hhi, nsteps = whi - wlo + 1;
    const T* vb = vol + b * D * plane;
    T* ab = agg + b * D * plane;
    auto load = [&](int h, T(&v)[K], T(&a)[K]) {
      const bool in = h >= hlo && h <= hhi;
      const int64_t o = (int64_t)h * W + (k + (int64_t)s * h);
#pragma unroll
      for (int j = 0; j < K; ++j) {
        const int d = g * K + j;
        const bool ok = in && d < D;
        v[j] = ok ? vb[d * plane + o] : ninf;
        a[j] = ok ? ab[d * plane + o] : (T)0;
      }
    };
    T L[K], M = 0, v[K], a[K];
#pragma unroll
    for (int j = 0; j < K; ++j) L[j] = ninf;
    int h = dy > 0 ? wlo : whi;
    load(h, v, a);
    for (int step = 0; step < nsteps; ++step, h += dy) {
      T vn[K], an[K];
      if (step + 1 < nsteps) load(h + dy, vn, an);
      sgm_step<T, K>(L, v, M, h == hstart, g, G, p1, p2);
      const bool in = h >= hlo && h <= hhi;
      const int64_t o = (int64_t)h * W + (k + (int64_t)s * h);
#pragma unroll
      for (int j = 0; j < K; ++j) {
        const int d = g * K + j;
        a[j] = a[j] + L[j];
        if (in && d < D) ab[d * plane + o] = a[j];
      }
      if (WTA) {
        // the first maximum of A over d: lane-local, then over the group (larger value, then smaller d)
        T best = ninf;
        int bd = D;
#pragma unroll
        for (int j = 0; j < K; ++j) {
          const int d = g * K + j;
          if (d < D && (bd == D || a[j] > best)) best = a[j], bd = d;
        }
        for (int o2 = 1; o2 < G; o2 <<= 1) {
          const T ob = __shfl_xor_sync(FULL, best, o2, G);
          const int od = __shfl_xor_sync(FULL, bd, o2, G);
          if (ob > best || (ob == best && od < bd)) best = ob, bd = od;
        }
        bd = min(bd, D - 1);  // only a non-finite column can leave it at D
        T cm = 0, cp = 0;
#pragma unroll
        for (int j = 0; j < K; ++j) {
          const int d = g * K + j;
          if (d == bd - 1) cm = a[j];
          if (d == bd + 1) cp = a[j];
        }
        cm = __shfl_sync(FULL, cm, max(bd - 1, 0) / K, G);
        cp = __shfl_sync(FULL, cp, min(bd + 1, D - 1) / K, G);
        if (in && g == 0) wta_store<T>(disp, score, b * plane + o, bd, best, cm, cp, D, subpixel);
      }
#pragma unroll
      for (int j = 0; j < K; ++j) v[j] = vn[j], a[j] = an[j];
    }
  }
}

int pow2_at_least(int64_t x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

template <typename T, int K>
int horizontal_launch(const T* vol, T* agg, int64_t B, int D, int H, int W, T p1, T p2, cudaStream_t st) {
  int WT = 32;
  while (WT > 1 && (size_t)2 * D * WT * sizeof(T) > SGM_SLAB_BYTES) WT >>= 1;
  const size_t smem = (size_t)SGM_HWARPS * 2 * D * WT * sizeof(T);
  auto kernel = sgm_horizontal<T, K>;
  const int rs = raise_smem_limit(kernel, smem, "sgm");
  if (rs != CTD_OK) return rs;
  const int64_t grid = std::min<int64_t>(cdiv(B * H, SGM_HWARPS), INT32_MAX);
  kernel<<<(unsigned)grid, 32 * SGM_HWARPS, smem, st>>>(vol, agg, B, D, H, W, WT, p1, p2);
  count_launch();
  return check_launch("sgm(horizontal)");
}

template <typename T, int K>
int lines_launch(const T* vol, T* agg, T* disp, T* score, int64_t B, int D, int H, int W, int dy, int dx, int G, T p1, T p2,
                 int subpixel, bool wta, cudaStream_t st) {
  const int64_t nk = W + (dx != 0 ? (int64_t)H - 1 : 0);
  const int64_t grid = std::min<int64_t>(cdiv(cdiv(B * nk, 32 / G), SGM_LTHREADS / 32), INT32_MAX);
  auto kernel = wta ? sgm_lines<T, K, true> : sgm_lines<T, K, false>;
  kernel<<<(unsigned)grid, SGM_LTHREADS, 0, st>>>(vol, agg, disp, score, B, D, H, W, dy, dx, G, p1, p2, subpixel);
  count_launch();
  return check_launch(wta ? "sgm(lines, winner-take-all)" : "sgm(lines)");
}

#define CTD_SGM_BY_K(K, CALL)      \
  switch (K) {                     \
    case 1: return CALL(1);        \
    case 2: return CALL(2);        \
    case 4: return CALL(4);        \
    case 8: return CALL(8);        \
    case 16: return CALL(16);      \
    default: return CALL(32);      \
  }

}  // namespace

template <typename T>
static int sgm_impl(const T* vol, T* agg, T* disp, T* score, int64_t B, int64_t D, int64_t H, int64_t W, double p1, double p2,
                    int paths, int subpixel, cudaStream_t st) {
  CTD_REQUIRE(paths == 4 || paths == 8, "sgm: paths must be 4 or 8, got %d", paths);
  const T tp1 = (T)p1, tp2 = (T)p2;
  CTD_REQUIRE(std::isfinite(tp1) && std::isfinite(tp2), "sgm: penalties must be finite in the volume's dtype");
  CTD_REQUIRE(tp1 >= 0 && tp2 >= tp1, "sgm: penalties must satisfy 0 <= p1 <= p2 (p1 = %g, p2 = %g)", p1, p2);
  CTD_REQUIRE(B >= 0 && D >= 0 && H >= 0 && W >= 0, "sgm: negative size");
  CTD_REQUIRE(H <= INT32_MAX && W <= INT32_MAX, "sgm: dimension too large");
  if (B * H * W == 0) return CTD_OK;
  CTD_REQUIRE(D >= 1, "sgm: the volume has no disparities (D = 0)");
  CTD_REQUIRE(D <= SGM_MAX_D, "sgm: at most %d disparities, got %lld", SGM_MAX_D, (long long)D);
  CTD_REQUIRE(vol && agg, "sgm: null pointer");
  const size_t n = (size_t)(B * D * H * W) * sizeof(T);
  CTD_REQUIRE(ranges_disjoint(agg, n, vol, n), "sgm: agg overlaps vol");
  const int d = (int)D, h = (int)H, w = (int)W;
  // horizontal: a warp per row
  const int kh = pow2_at_least(cdiv(D, 32));
#define CTD_SGM_H(K) horizontal_launch<T, K>(vol, agg, B, d, h, w, tp1, tp2, st)
  const int rc = [&]() -> int { CTD_SGM_BY_K(kh, CTD_SGM_H) }();
#undef CTD_SGM_H
  if (rc != CTD_OK) return rc;
  // vertical and diagonal: 8 lanes per line (4 adjacent lines per warp, 32-byte row segments) while a lane holds at most
  // 16 floats or 8 doubles (more spill: the kernel keeps four such arrays), then wider groups
  const int kmax = sizeof(T) == 4 ? 16 : 8;
  int G = 8, kl = pow2_at_least(cdiv(D, 8));
  if (kl > kmax) kl = kmax, G = pow2_at_least(cdiv(D, kmax));
  if (G > 32) G = 32, kl = pow2_at_least(cdiv(D, 32));
  static const int dirs[6][2] = {{1, 0}, {-1, 0}, {1, 1}, {1, -1}, {-1, 1}, {-1, -1}};
  const int npass = paths - 2;
  for (int i = 0; i < npass; ++i) {
    const bool wta = i == npass - 1 && (disp || score);
    const int dy = dirs[i][0], dx = dirs[i][1];
#define CTD_SGM_L(K) lines_launch<T, K>(vol, agg, disp, score, B, d, h, w, dy, dx, G, tp1, tp2, subpixel, wta, st)
    const int r = [&]() -> int { CTD_SGM_BY_K(kl, CTD_SGM_L) }();
#undef CTD_SGM_L
    if (r != CTD_OK) return r;
  }
  return CTD_OK;
}

}  // namespace ctd

CTD_API int ctd_sgm_f32(const float* vol, float* agg, float* disp, float* score, int64_t B, int64_t D, int64_t H, int64_t W,
                        double p1, double p2, int paths, int subpixel, ctd_stream_t s) {
  return ctd::sgm_impl<float>(vol, agg, disp, score, B, D, H, W, p1, p2, paths, subpixel, ctd::as_stream(s));
}
CTD_API int ctd_sgm_f64(const double* vol, double* agg, double* disp, double* score, int64_t B, int64_t D, int64_t H,
                        int64_t W, double p1, double p2, int paths, int subpixel, ctd_stream_t s) {
  return ctd::sgm_impl<double>(vol, agg, disp, score, B, D, H, W, p1, p2, paths, subpixel, ctd::as_stream(s));
}
