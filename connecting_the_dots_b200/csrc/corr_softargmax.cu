// Differentiable correlation soft-argmax disparity (ctd_corr_softargmax_fwd_* / _bwd_*) for sm_100a: the DispNetC /
// FlowNet 1-D correlation of two feature maps followed by a soft-argmax over d, forward and backward fused so that the
// B x D x H x W score volume is never written.
//
// Definition (include/ctd_b200.h states it in full): for pixel (b,h,w), Dw = min(D, w + 1) and, for d < Dw,
// s_d = (sum_c f0[b,c,h,w] * f1[b,c,h,w-d]) / C; lse = logsumexp_d(s_d / tau), p_d = exp(s_d / tau - lse),
// disp = sum_d d * p_d; d disp / d s_d = p_d (d - disp) / tau.
//
// Every launch takes one chunk of TW = 128 pixels of one image row per CTA (4 warps; a lane owns 4 consecutive pixels).
// Disparities go in groups of DG = 4 * DT; warp g takes the tile [d0 + g*DT, d0 + (g+1)*DT) of a group, so the four warps
// share one staged window of the partner row.  Channels are staged in slabs of up to CS; scores of a tile stay in
// registers (4 x DT accumulators per lane) until every slab is added.  Shared-memory reads are 16-byte vector loads: a
// lane reads its 4 own pixels and a DT + 4 wide window of the partner row per channel for 4 x DT FMAs.
//   corr_fwd: online softmax per pixel and warp (running max, sum of exp and d-weighted sum), the four warps' states
//             combined in a fixed order at the end; writes disp and lse (the saved state of the backward).
//   corr_bwd<to_f1 = false>: grad_f0 of a chunk of pixels w.  Scores of (w, d) are recomputed, a_d(w) = grad_disp(w) *
//             exp(s_d/tau - lse(w)) * (d - disp(w)) / (tau C) goes to shared memory, and grad_f0[c,w] += a_d(w) f1[c,w-d]
//             with a warp owning a quarter of the channels of the slab for all pixels and disparities.
//   corr_bwd<to_f1 = true>: grad_f1 of a chunk of columns x, the mirror image: the pairs are (x + d, d), the per-pixel
//             state of the pixels x + d is staged with the partner window, grad_f1[c,x] += a_d(x+d) f0[c,x+d].
// Contributions that cross a chunk border are recomputed by the chunk that owns the output, so there are no atomics and
// the gradients are bit-identical from run to run.  More than CS channels repeat the score pass once per output slab.
// No scratch memory, no host synchronisation, 64-bit indexing over the batch: every call is capture-safe.
#include <algorithm>
#include <cmath>

#include "ctd_common.cuh"

namespace ctd {

namespace {

constexpr int CA_NW = 4;              // warps per CTA, one disparity tile each
constexpr int CA_THREADS = 32 * CA_NW;
constexpr int CA_TW = 128;            // pixels per CTA: 32 lanes x 4

template <typename T>
struct CaCfg;
template <>
struct CaCfg<float> {
  static constexpr int DT = 16, CS = 32;
};
template <>
struct CaCfg<double> {
  static constexpr int DT = 8, CS = 16;
};

// 4 consecutive values from shared memory at a 4-element boundary (16-byte loads)
__device__ __forceinline__ void lds4(const float* p, float (&r)[4]) {
  const float4 v = *reinterpret_cast<const float4*>(p);
  r[0] = v.x;
  r[1] = v.y;
  r[2] = v.z;
  r[3] = v.w;
}
__device__ __forceinline__ void lds4(const double* p, double (&r)[4]) {
  const double2 a = *reinterpret_cast<const double2*>(p), b = *reinterpret_cast<const double2*>(p + 2);
  r[0] = a.x;
  r[1] = a.y;
  r[2] = b.x;
  r[3] = b.y;
}
__device__ __forceinline__ void sts4(float* p, const float (&r)[4]) {
  *reinterpret_cast<float4*>(p) = make_float4(r[0], r[1], r[2], r[3]);
}
__device__ __forceinline__ void sts4(double* p, const double (&r)[4]) {
  *reinterpret_cast<double2*>(p) = make_double2(r[0], r[1]);
  *reinterpret_cast<double2*>(p + 2) = make_double2(r[2], r[3]);
}

// The DT + 4 wide window of a partner row that a lane reads for one disparity tile.  Pixel k of the lane and disparity j
// of the tile meet the partner at win[DT + k - j] (f0 side: column w - d) or at win[k + j] (f1 side: column x + d).
template <typename T, int DT>
__device__ __forceinline__ void load_window(const T* p, T (&win)[DT + 4]) {
#pragma unroll
  for (int q = 0; q < DT + 4; q += 4) {
    T r[4];
    lds4(p + q, r);
#pragma unroll
    for (int i = 0; i < 4; ++i) win[q + i] = r[i];
  }
}

template <bool MIRROR, int DT>
__device__ __forceinline__ constexpr int win_index(int k, int j) {
  return MIRROR ? k + j : DT + k - j;
}

// The row chunk a CTA works on
struct CaChunk {
  int64_t b;
  int h, w0;
};
__device__ __forceinline__ CaChunk ca_chunk(int64_t blk, int H, int nchunk) {
  const int64_t row = blk / nchunk;
  return {row / H, (int)(row % H), (int)(blk % nchunk) * CA_TW};
}

// Stage channels [c0, c0 + cs) of src's row (b, h), columns [x_lo, x_lo + width), into dst[c][width]; 0 outside [0, W).
template <typename T>
__device__ __forceinline__ void stage_rows(T* dst, const T* __restrict__ src, int64_t b, int c0, int cs, int C, int H, int W,
                                           int h, int x_lo, int width) {
  for (int i = threadIdx.x; i < cs * width; i += CA_THREADS) {
    const int c = i / width, x = x_lo + i % width;
    dst[i] = x >= 0 && x < W ? src[(((b * C) + c0 + c) * H + h) * (int64_t)W + x] : T(0);
  }
}

// acc[k][j] += sum over the staged channels of self[c][4 lane + k] * partner[c][win_index(k, j)], partner rows read from
// part + off (off: the tile's offset in the group window)
template <typename T, int DT, bool MIRROR>
__device__ __forceinline__ void add_scores(T (&acc)[4][DT], const T* self, const T* part, int cs, int lane, int off) {
  constexpr int NX = CA_TW + CA_NW * DT;
  for (int c = 0; c < cs; ++c) {
    T s4[4], win[DT + 4];
    lds4(self + c * CA_TW + 4 * lane, s4);
    load_window<T, DT>(part + c * NX + off + 4 * lane, win);
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int j = 0; j < DT; ++j) acc[k][j] = fma(s4[k], win[win_index<MIRROR, DT>(k, j)], acc[k][j]);
  }
}

template <typename T>
__device__ __forceinline__ T ca_exp(T x);
template <>
__device__ __forceinline__ float ca_exp<float>(float x) { return expf(x); }
template <>
__device__ __forceinline__ double ca_exp<double>(double x) { return exp(x); }

template <typename T>
__global__ void __launch_bounds__(CA_THREADS)
corr_fwd(const T* __restrict__ f0, const T* __restrict__ f1, T* __restrict__ disp, T* __restrict__ lse, int64_t B, int C,
         int H, int W, int D, T scale, int64_t nblk, int nchunk) {
  constexpr int DT = CaCfg<T>::DT, CS = CaCfg<T>::CS, DG = CA_NW * DT, NX = CA_TW + DG;
  extern __shared__ __align__(16) unsigned char ca_smem[];
  const int cs_max = min(C, CS);
  T* self = reinterpret_cast<T*>(ca_smem);  // [cs_max][TW]
  T* part = self + cs_max * CA_TW;          // [cs_max][NX]; after the last group [3][NW][TW] for the combine
  const int lane = threadIdx.x % 32, g = threadIdx.x / 32;
  const int nslab = (C + CS - 1) / CS, ngroup = (min(D, W) + DG - 1) / DG;
  for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
    const CaChunk ck = ca_chunk(blk, H, nchunk);
    T m[4], l[4], u[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      m[k] = lowest<T>();
      l[k] = u[k] = T(0);
    }
    for (int gi = 0; gi < ngroup; ++gi) {
      const int d0 = gi * DG;
      if (d0 > min(ck.w0 + CA_TW, W) - 1) break;  // no pixel of the chunk has these disparities
      T acc[4][DT];
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int j = 0; j < DT; ++j) acc[k][j] = T(0);
      for (int s = 0; s < nslab; ++s) {
        const int c0 = s * CS, cs = min(CS, C - c0);
        __syncthreads();  // the previous slab or group has been read
        if (nslab > 1 || gi == 0) stage_rows(self, f0, ck.b, c0, cs, C, H, W, ck.h, ck.w0, CA_TW);
        stage_rows(part, f1, ck.b, c0, cs, C, H, W, ck.h, ck.w0 - d0 - DG, NX);
        __syncthreads();
        add_scores<T, DT, false>(acc, self, part, cs, lane, (CA_NW - 1 - g) * DT);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int w = ck.w0 + 4 * lane + k;
        T v[DT], mt = lowest<T>();
#pragma unroll
        for (int j = 0; j < DT; ++j) {
          const int d = d0 + g * DT + j;
          v[j] = d < D && d <= w ? acc[k][j] * scale : lowest<T>();
          mt = fmax(mt, v[j]);
        }
        if (mt == lowest<T>()) continue;  // no disparity of this tile reaches the pixel
        const T mn = fmax(m[k], mt), r = ca_exp(m[k] - mn);
        T ls = l[k] * r, us = u[k] * r;
#pragma unroll
        for (int j = 0; j < DT; ++j) {
          const T e = ca_exp(v[j] - mn);  // 0 for the masked entries
          ls += e;
          us = fma(e, T(d0 + g * DT + j), us);
        }
        m[k] = mn;
        l[k] = ls;
        u[k] = us;
      }
    }
    __syncthreads();  // part is reused for the combine
    T* red = part;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int p = 4 * lane + k;
      red[(0 * CA_NW + g) * CA_TW + p] = m[k];
      red[(1 * CA_NW + g) * CA_TW + p] = l[k];
      red[(2 * CA_NW + g) * CA_TW + p] = u[k];
    }
    __syncthreads();
    const int p = threadIdx.x, w = ck.w0 + p;
    if (w < W) {
      T M = lowest<T>();
#pragma unroll
      for (int q = 0; q < CA_NW; ++q) M = fmax(M, red[q * CA_TW + p]);
      T L = T(0), U = T(0);
#pragma unroll
      for (int q = 0; q < CA_NW; ++q) {  // fixed order: deterministic
        const T r = ca_exp(red[q * CA_TW + p] - M);
        L = fma(red[(CA_NW + q) * CA_TW + p], r, L);
        U = fma(red[(2 * CA_NW + q) * CA_TW + p], r, U);
      }
      const int64_t px = ((int64_t)ck.b * H + ck.h) * W + w;
      disp[px] = U / L;
      lse[px] = M + log(L);
    }
  }
}

// TO_F1 = false: grad_f0 of the chunk's pixels (self f0, partner f1 at w - d).  TO_F1 = true: grad_f1 of the chunk's
// columns (self f1, partner f0 at x + d, the pixel state of x + d staged beside it).
template <typename T, bool TO_F1>
__global__ void __launch_bounds__(CA_THREADS)
corr_bwd(const T* __restrict__ f0, const T* __restrict__ f1, const T* __restrict__ disp, const T* __restrict__ lse,
         const T* __restrict__ grad_disp, T* __restrict__ grad, int64_t B, int C, int H, int W, int D, T scale, int64_t nblk,
         int nchunk) {
  constexpr int DT = CaCfg<T>::DT, CS = CaCfg<T>::CS, DG = CA_NW * DT, NX = CA_TW + DG, CPW = CS / CA_NW;
  extern __shared__ __align__(16) unsigned char ca_smem[];
  const int cs_max = min(C, CS);
  T* self = reinterpret_cast<T*>(ca_smem);  // [cs_max][TW]
  T* part = self + cs_max * CA_TW;          // [cs_max][NX]
  T* coef = part + cs_max * NX;             // [DG][TW]: a of the group, row = disparity, column = own pixel
  T* st = coef + DG * CA_TW;                // TO_F1: [3][NX] grad_disp * scale, disp, lse of the pixels x + d
  const T* fs = TO_F1 ? f1 : f0;
  const T* fp = TO_F1 ? f0 : f1;
  const int lane = threadIdx.x % 32, g = threadIdx.x / 32;
  const int nslab = (C + CS - 1) / CS, ngroup = (min(D, W) + DG - 1) / DG;
  for (int64_t blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
    const CaChunk ck = ca_chunk(blk, H, nchunk);
    const int64_t rowpx = ((int64_t)ck.b * H + ck.h) * W;
    T gk[4], dp[4], ls[4];  // TO_F1 = false: the state of the own pixels
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int w = ck.w0 + 4 * lane + k;
      const bool in = !TO_F1 && w < W;
      gk[k] = in ? grad_disp[rowpx + w] * scale : T(0);
      dp[k] = in ? disp[rowpx + w] : T(0);
      ls[k] = in ? lse[rowpx + w] : T(0);
    }
    for (int os = 0; os < nslab; ++os) {  // output channels [os * CS, os * CS + ocs)
      const int oc0 = os * CS, ocs = min(CS, C - oc0);
      T acc_g[4][CPW];
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int q = 0; q < CPW; ++q) acc_g[k][q] = T(0);
      for (int gi = 0; gi < ngroup; ++gi) {
        const int d0 = gi * DG;
        if (TO_F1 ? ck.w0 + d0 >= W : d0 > min(ck.w0 + CA_TW, W) - 1) break;
        const int x_lo = TO_F1 ? ck.w0 + d0 : ck.w0 - d0 - DG;
        const int off = TO_F1 ? g * DT : (CA_NW - 1 - g) * DT;
        T acc[4][DT];
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
          for (int j = 0; j < DT; ++j) acc[k][j] = T(0);
        for (int s = 0; s < nslab; ++s) {
          const int c0 = s * CS, cs = min(CS, C - c0);
          __syncthreads();
          if (nslab > 1 || gi == 0) stage_rows(self, fs, ck.b, c0, cs, C, H, W, ck.h, ck.w0, CA_TW);
          stage_rows(part, fp, ck.b, c0, cs, C, H, W, ck.h, x_lo, NX);
          if (TO_F1 && s == 0) {
            for (int i = threadIdx.x; i < NX; i += CA_THREADS) {
              const int x = x_lo + i;
              const bool in = x < W;
              st[i] = in ? grad_disp[rowpx + x] * scale : T(0);
              st[NX + i] = in ? disp[rowpx + x] : T(0);
              st[2 * NX + i] = in ? lse[rowpx + x] : T(0);
            }
          }
          __syncthreads();
          add_scores<T, DT, TO_F1>(acc, self, part, cs, lane, off);
        }
        // a of the warp's tile -> coef
#pragma unroll
        for (int j = 0; j < DT; ++j) {
          const int d = d0 + g * DT + j;
          T a4[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int x = ck.w0 + 4 * lane + k;  // the own pixel (grad_f0) or column (grad_f1)
            T a = T(0);
            if (TO_F1) {
              const int i = off + 4 * lane + k + j;  // pixel x + d in the state window
              if (d < D && x + d < W) a = st[i] * ca_exp(acc[k][j] * scale - st[2 * NX + i]) * (T(d) - st[NX + i]);
            } else if (d < D && d <= x && x < W) {
              a = gk[k] * ca_exp(acc[k][j] * scale - ls[k]) * (T(d) - dp[k]);
            }
            a4[k] = a;
          }
          sts4(coef + (g * DT + j) * CA_TW + 4 * lane, a4);
        }
        if (nslab > 1) {  // the partner slab of the output channels
          __syncthreads();
          stage_rows(part, fp, ck.b, oc0, ocs, C, H, W, ck.h, x_lo, NX);
        }
        __syncthreads();
        // grad[c][x] += sum_d a_d * partner[c][...]: warp g takes channels g, g + NW, ... of the output slab
#pragma unroll 1
        for (int t = 0; t < CA_NW; ++t) {
          const int toff = TO_F1 ? t * DT : (CA_NW - 1 - t) * DT;
          T a[DT][4];
#pragma unroll
          for (int j = 0; j < DT; ++j) lds4(coef + (t * DT + j) * CA_TW + 4 * lane, a[j]);
#pragma unroll
          for (int q = 0; q < CPW; ++q) {
            const int c = g + CA_NW * q;
            if (c >= ocs) break;
            T win[DT + 4];
            load_window<T, DT>(part + c * NX + toff + 4 * lane, win);
#pragma unroll
            for (int k = 0; k < 4; ++k)
#pragma unroll
              for (int j = 0; j < DT; ++j) acc_g[k][q] = fma(a[j][k], win[win_index<TO_F1, DT>(k, j)], acc_g[k][q]);
          }
        }
      }
#pragma unroll
      for (int q = 0; q < CPW; ++q) {
        const int c = g + CA_NW * q;
        if (c >= ocs) break;
        T* out = grad + (((int64_t)ck.b * C + oc0 + c) * H + ck.h) * W;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int x = ck.w0 + 4 * lane + k;
          if (x < W) out[x] = acc_g[k][q];
        }
      }
    }
  }
}

}  // namespace

template <typename T>
static size_t ca_smem_bytes(int64_t C, bool backward) {
  constexpr int DT = CaCfg<T>::DT, CS = CaCfg<T>::CS, DG = CA_NW * DT, NX = CA_TW + DG;
  const int64_t cs = std::min<int64_t>(C, CS);
  const int64_t fwd = std::max<int64_t>(cs * (CA_TW + NX), cs * CA_TW + 3 * CA_NW * CA_TW);
  return (size_t)(backward ? cs * (CA_TW + NX) + DG * CA_TW + 3 * NX : fwd) * sizeof(T);
}

// Argument checks common to both directions; *empty is set when there is nothing to compute.
static int ca_check(const char* op, int64_t B, int64_t C, int64_t H, int64_t W, int64_t D, double temperature,
                    bool* empty) {
  CTD_REQUIRE(B >= 0 && C >= 0 && H >= 0 && W >= 0 && D >= 0, "%s: negative size", op);
  CTD_REQUIRE(std::isfinite(temperature) && temperature > 0.0, "%s: temperature must be finite and > 0, got %g", op,
              temperature);
  *empty = B == 0 || H == 0 || W == 0;
  if (*empty) return CTD_OK;
  CTD_REQUIRE(C >= 1, "%s: C must be >= 1 (C = 0)", op);
  CTD_REQUIRE(D >= 1, "%s: n_disps must be >= 1 (D = 0)", op);
  // columns of a staged window reach 2 W; D only matters up to W
  CTD_REQUIRE(C <= INT32_MAX && H <= INT32_MAX && W <= INT32_MAX / 4, "%s: C, H or W exceeds the kernels' int32 range", op);
  CTD_REQUIRE(H * W <= INT64_MAX / C / B / 8, "%s: batch too large", op);
  return CTD_OK;
}

template <typename T, typename Kernel, typename... Args>
static int ca_launch(Kernel kernel, size_t smem, int64_t B, int64_t H, int64_t W, cudaStream_t st, const char* op,
                     Args... args) {
  const int r = raise_smem_limit(kernel, smem, op);
  if (r != CTD_OK) return r;
  const int nchunk = (int)cdiv(W, CA_TW);
  const int64_t nblk = B * H * nchunk;
  const unsigned grid = (unsigned)std::min<int64_t>(nblk, INT32_MAX);
  kernel<<<grid, CA_THREADS, smem, st>>>(args..., nblk, nchunk);
  count_launch();
  return check_launch(op);
}

template <typename T>
static int corr_fwd_impl(const T* f0, const T* f1, T* disp, T* lse, int64_t B, int64_t C, int64_t H, int64_t W,
                         int64_t D, double temperature, cudaStream_t st) {
  const char* op = "corr_softargmax_fwd";
  bool empty = false;
  const int rc = ca_check(op, B, C, H, W, D, temperature, &empty);
  if (rc != CTD_OK || empty) return rc;
  CTD_REQUIRE(f0 && f1 && disp && lse, "%s: null pointer", op);
  const size_t nf = (size_t)(B * C * H * W) * sizeof(T), nm = (size_t)(B * H * W) * sizeof(T);
  CTD_REQUIRE(ranges_disjoint(disp, nm, f0, nf) && ranges_disjoint(disp, nm, f1, nf), "%s: disp overlaps an input", op);
  CTD_REQUIRE(ranges_disjoint(lse, nm, f0, nf) && ranges_disjoint(lse, nm, f1, nf), "%s: lse overlaps an input", op);
  CTD_REQUIRE(ranges_disjoint(disp, nm, lse, nm), "%s: disp overlaps lse", op);
  const T scale = (T)(1.0 / ((double)C * temperature));
  return ca_launch<T>(corr_fwd<T>, ca_smem_bytes<T>(C, false), B, H, W, st, op, f0, f1, disp, lse, B, (int)C, (int)H,
                      (int)W, (int)std::min<int64_t>(D, W), scale);
}

template <typename T>
static int corr_bwd_impl(const T* f0, const T* f1, const T* disp, const T* lse, const T* grad_disp, T* grad_f0,
                         T* grad_f1, int64_t B, int64_t C, int64_t H, int64_t W, int64_t D, double temperature,
                         cudaStream_t st) {
  const char* op = "corr_softargmax_bwd";
  bool empty = false;
  const int rc = ca_check(op, B, C, H, W, D, temperature, &empty);
  if (rc != CTD_OK || empty) return rc;
  if (!grad_f0 && !grad_f1) return CTD_OK;
  CTD_REQUIRE(f0 && f1 && disp && lse && grad_disp, "%s: null pointer", op);
  const size_t nf = (size_t)(B * C * H * W) * sizeof(T), nm = (size_t)(B * H * W) * sizeof(T);
  for (T* out : {grad_f0, grad_f1}) {
    CTD_REQUIRE(ranges_disjoint(out, nf, f0, nf) && ranges_disjoint(out, nf, f1, nf) && ranges_disjoint(out, nf, disp, nm) &&
                    ranges_disjoint(out, nf, lse, nm) && ranges_disjoint(out, nf, grad_disp, nm),
                "%s: a gradient overlaps an input", op);
  }
  CTD_REQUIRE(ranges_disjoint(grad_f0, nf, grad_f1, nf), "%s: grad_f0 overlaps grad_f1", op);
  const T scale = (T)(1.0 / ((double)C * temperature));
  const int Dk = (int)std::min<int64_t>(D, W);
  const size_t smem = ca_smem_bytes<T>(C, true);
  if (grad_f0) {
    const int r = ca_launch<T>(corr_bwd<T, false>, smem, B, H, W, st, op, f0, f1, disp, lse, grad_disp, grad_f0, B, (int)C,
                               (int)H, (int)W, Dk, scale);
    if (r != CTD_OK) return r;
  }
  if (grad_f1)
    return ca_launch<T>(corr_bwd<T, true>, smem, B, H, W, st, op, f0, f1, disp, lse, grad_disp, grad_f1, B, (int)C, (int)H,
                        (int)W, Dk, scale);
  return CTD_OK;
}

}  // namespace ctd

CTD_API int ctd_corr_softargmax_fwd_f32(const float* f0, const float* f1, float* disp, float* lse, int64_t B, int64_t C,
                                        int64_t H, int64_t W, int64_t n_disps, double temperature, ctd_stream_t s) {
  return ctd::corr_fwd_impl<float>(f0, f1, disp, lse, B, C, H, W, n_disps, temperature, ctd::as_stream(s));
}
CTD_API int ctd_corr_softargmax_fwd_f64(const double* f0, const double* f1, double* disp, double* lse, int64_t B, int64_t C,
                                        int64_t H, int64_t W, int64_t n_disps, double temperature, ctd_stream_t s) {
  return ctd::corr_fwd_impl<double>(f0, f1, disp, lse, B, C, H, W, n_disps, temperature, ctd::as_stream(s));
}
CTD_API int ctd_corr_softargmax_bwd_f32(const float* f0, const float* f1, const float* disp, const float* lse,
                                        const float* grad_disp, float* grad_f0, float* grad_f1, int64_t B, int64_t C,
                                        int64_t H, int64_t W, int64_t n_disps, double temperature, ctd_stream_t s) {
  return ctd::corr_bwd_impl<float>(f0, f1, disp, lse, grad_disp, grad_f0, grad_f1, B, C, H, W, n_disps, temperature,
                                   ctd::as_stream(s));
}
CTD_API int ctd_corr_softargmax_bwd_f64(const double* f0, const double* f1, const double* disp, const double* lse,
                                        const double* grad_disp, double* grad_f0, double* grad_f1, int64_t B, int64_t C,
                                        int64_t H, int64_t W, int64_t n_disps, double temperature, ctd_stream_t s) {
  return ctd::corr_bwd_impl<double>(f0, f1, disp, lse, grad_disp, grad_f0, grad_f1, B, C, H, W, n_disps, temperature,
                                    ctd::as_stream(s));
}
