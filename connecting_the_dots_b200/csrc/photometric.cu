// PhotometricLoss forward / backward for sm_100a.
//
// Reference semantics: torchext/ext/ext.h:201-266 (forward) and :268-344 (backward), bound at
// torchext/ext/ext_cuda.cpp:92-123.  Nothing here is a translation of those functors: the
// reference runs one thread per output pixel that walks bs*bs taps in global memory and, in the
// backward, scatters with atomicAdd.  Here
//   * mse/sad forward is a separable replicate-clamped box filter of phi(es-ta) on a shared-memory
//     tile, 128-bit loads/stores;
//   * mse/sad backward is the adjoint box filter of grad_out (zero padded, border rows/columns
//     re-weighted by the clamp multiplicity) times phi'(es-ta): a gather, no atomics, no memset;
//   * census forward/backward are gathers over a shared-memory halo tile with four pixels per
//     thread so every tap row is fetched with three 128-bit shared loads; the backward uses the
//     antisymmetry of the soft census step to fold the "tap" and "centre" roles of a pixel pair
//     into one term, and keeps sign() decisions bit-identical to the reference by recomputing
//     near-ties with IEEE operations;
//   * every other case (block size != 9, fp64, tiny images) runs generic gather kernels that
//     follow the reference's operation order (this file is compiled with -fmad=false for them).
#include <algorithm>

#include "ctd_common.cuh"

namespace ctd {

extern int g_force_generic;
int box9_tma_fwd(const float* es, const float* ta, float* out, int64_t B, int64_t C, int64_t H, int64_t W, int type,
                 cudaStream_t st);
int box9_tma_bwd(const float* es, const float* ta, const float* go, float* gi, int64_t B, int64_t C, int64_t H,
                 int64_t W, int type, cudaStream_t st);
int box9_tma_fwd_bwd(const float* es, const float* ta, const float* go, float* out, float* gi, int64_t B, int64_t C,
                     int64_t H, int64_t W, int type, cudaStream_t st);
int masked_sums_launch(const float* diff, const float* mask, int64_t n, float* out2, cudaStream_t st);
int box9_tma_fwd_bwd_masked(const float* es, const float* ta, const float* go, const float* mask, float* out, float* gi,
                            float* sums2, int64_t B, int64_t C, int64_t H, int64_t W, int type, cudaStream_t st);
// census_sym.cu: every pixel pair evaluated once (forward, backward or both, optional masked sums); false = not taken.
// Two kernels serve census_mse / census_sad at block size 9: this pair-symmetric one and the tile kernels below, which
// take every call it refuses.  The choice is census_sym_launch's size rule: by default it takes forward-only and
// backward-only calls from ~6 images (CS_MIN_PIXELS) and leaves fused forward+backward calls to the tile kernels;
// ctd_set_option("census_sym", 0 / 1) sends every call to the tile kernels / to it where the shape allows.
bool census_sym_launch(const float* es, const float* ta, const float* go, float* out, float* gi, const float* mask, float* sums2,
                       int64_t B, int64_t C, int64_t H, int64_t W, int type, float eps, cudaStream_t st);

// ------------------------------------------------------------------------------------------
// generic kernels (any block size, channel count, size; float or double)
// ------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T soft_step(T x, T eps) {  // ext.h:245-246
  T q = x / sqrt(x * x + eps);
  return T(0.5) * (T(1) + q);
}

template <typename T>
__device__ __forceinline__ T sgn(T d) {
  return d < T(0) ? T(-1) : (d > T(0) ? T(1) : T(0));
}

template <typename T>
__global__ void __launch_bounds__(256)
photo_fwd_generic(const T* __restrict__ es, const T* __restrict__ ta, T* __restrict__ out, int64_t B,
                  int C, int H, int W, int bs, int type, T eps) {
  const int64_t total = B * H * W;
  const int bs2 = bs * bs, half = bs / 2;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int w = idx % W, h = (idx / W) % H;
    const int64_t n = idx / ((int64_t)W * H);
    T acc = 0;
    for (int t = 0; t < bs2; ++t) {
      const int hh = clampi(h + t / bs - half, 0, H - 1);
      const int ww = clampi(w + t % bs - half, 0, W - 1);
      for (int c = 0; c < C; ++c) {
        const int64_t base = (n * C + c) * H;
        const int64_t tap = (base + hh) * W + ww;
        T d;
        if (type <= 1) {
          d = es[tap] - ta[tap];
        } else {
          const int64_t ctr = (base + h) * W + w;
          d = soft_step(es[tap] - es[ctr], eps) - soft_step(ta[tap] - ta[ctr], eps);
        }
        acc += ((type & 1) ? fabs(d) : d * d) / T(bs2);
      }
    }
    out[idx] = acc;
  }
}

// number of window offsets delta in [-lo, hi] with clamp(p + delta, 0, n-1) == i
__device__ __forceinline__ int clamp_mult(int p, int i, int n, int lo, int hi) {
  int m = 0;
  for (int d = -lo; d <= hi; ++d) m += (clampi(p + d, 0, n - 1) == i);
  return m;
}

template <typename T>
__global__ void __launch_bounds__(256)
photo_bwd_generic(const T* __restrict__ es, const T* __restrict__ ta, const T* __restrict__ go,
                  T* __restrict__ gi, int64_t B, int C, int H, int W, int bs, int type, T eps) {
  const int64_t total = B * C * H * W;
  const int lo = bs / 2, hi = bs - 1 - lo;
  const T inv_n = T(bs * bs);
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int x = idx % W, y = (idx / W) % H;
    const int64_t nc = idx / ((int64_t)W * H);
    const int64_t n = nc / C;
    const T* esp = es + nc * H * W;
    const T* tap = ta + nc * H * W;
    const T* gop = go + n * H * W;
    const T ei = esp[(int64_t)y * W + x], ti = tap[(int64_t)y * W + x];
    T acc = 0;
    // role 1: pixel i is the (clamped) tap of centre p
    for (int py = max(0, y - hi); py <= min(H - 1, y + lo); ++py) {
      const int my = clamp_mult(py, y, H, lo, hi);
      if (!my) continue;
      for (int px = max(0, x - hi); px <= min(W - 1, x + lo); ++px) {
        const int mx = clamp_mult(px, x, W, lo, hi);
        if (!mx) continue;
        const T g0 = gop[(int64_t)py * W + px];
        T g;
        if (type <= 1) {
          const T d = ei - ti;
          g = ((type & 1) ? sgn(d) : T(2) * d) / inv_n * g0;
        } else {
          const T des = ei - esp[(int64_t)py * W + px];
          const T dta = ti - tap[(int64_t)py * W + px];
          const T d = soft_step(des, eps) - soft_step(dta, eps);
          const T gl = ((type & 1) ? sgn(d) : T(2) * d) / inv_n;
          const T s = des * des + eps;
          const T gh = T(0.5) * eps / sqrt(s * s * s);
          g = g0 * gl * gh;
        }
        acc += T(my * mx) * g;
      }
    }
    // role 2 (census only): pixel i is the centre; every tap sends -g back to it
    if (type >= 2) {
      const T g0 = gop[(int64_t)y * W + x];
      for (int t = 0; t < bs * bs; ++t) {
        const int hh = clampi(y + t / bs - lo, 0, H - 1);
        const int ww = clampi(x + t % bs - lo, 0, W - 1);
        const T des = esp[(int64_t)hh * W + ww] - ei;
        const T dta = tap[(int64_t)hh * W + ww] - ti;
        const T d = soft_step(des, eps) - soft_step(dta, eps);
        const T gl = ((type & 1) ? sgn(d) : T(2) * d) / inv_n;
        const T s = des * des + eps;
        const T gh = T(0.5) * eps / sqrt(s * s * s);
        acc -= g0 * gl * gh;
      }
    }
    gi[idx] = acc;
  }
}

// ------------------------------------------------------------------------------------------
// fast path, block size 9, fp32: mse / sad
// ------------------------------------------------------------------------------------------
constexpr int R9 = 4;                 // window radius of block size 9
constexpr int BT_W = 128, BT_H = 32;  // output tile of the box-filter kernels
constexpr int BE_W = BT_W + 2 * R9;   // 136
constexpr int BE_H = BT_H + 2 * R9;   // 40
constexpr float INV81 = 1.0f / 81.0f;

// four horizontally adjacent 9-sums from 12 consecutive values a|b|c
__device__ __forceinline__ float4 hsum9x4(const float4 a, const float4 b, const float4 c) {
  const float mid = ((a.w + b.x) + (b.y + b.z)) + (b.w + c.x);  // columns 3..8, shared by all four
  const float l12 = a.y + a.z, r910 = c.y + c.z;
  float4 o;
  o.x = mid + (a.x + l12);
  o.y = mid + (l12 + c.y);
  o.z = mid + (a.z + r910);
  o.w = mid + (r910 + c.w);
  return o;
}
__device__ __forceinline__ float4 add4(const float4 a, const float4 b) {
  return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}
__device__ __forceinline__ float4 fma4s(const float s, const float4 a, const float4 b) {
  return make_float4(fmaf(s, a.x, b.x), fmaf(s, a.y, b.y), fmaf(s, a.z, b.z), fmaf(s, a.w, b.w));
}

template <int TYPE>
__device__ __forceinline__ float phi(float d) {
  return TYPE == 0 ? d * d : fabsf(d);
}

// out = box9(phi(es - ta)) / 81 with replicate-clamped borders, summed over channels.
template <int TYPE>
__global__ void __launch_bounds__(256)
photo_fwd_box9(const float* __restrict__ es, const float* __restrict__ ta, float* __restrict__ out,
               int C, int H, int W, int vec) {
  __shared__ __align__(16) float E[BE_H][BE_W];
  __shared__ __align__(16) float Hs[BE_H][BT_W];
  const int x0 = blockIdx.x * BT_W, y0 = blockIdx.y * BT_H;
  const int64_t n = blockIdx.z;
  const int tid = threadIdx.x;
  const int64_t plane = (int64_t)H * W;
  const float* esn = es + n * C * plane;
  const float* tan = ta + n * C * plane;

  for (int ch = tid; ch < BE_H * (BE_W / 4); ch += 256) {
    const int r = ch / (BE_W / 4), k = ch % (BE_W / 4);
    const int gy = clampi(y0 - R9 + r, 0, H - 1);
    const int gx = x0 - R9 + 4 * k;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (vec && gx >= 0 && gx + 3 < W) {
      const int64_t off = (int64_t)gy * W + gx;
      for (int c = 0; c < C; ++c) {
        const float4 a = ldg4(esn + c * plane + off), b = ldg4(tan + c * plane + off);
        acc.x += phi<TYPE>(a.x - b.x);
        acc.y += phi<TYPE>(a.y - b.y);
        acc.z += phi<TYPE>(a.z - b.z);
        acc.w += phi<TYPE>(a.w - b.w);
      }
    } else {
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t off = (int64_t)gy * W + clampi(gx + j, 0, W - 1);
        float s = 0.f;
        for (int c = 0; c < C; ++c) s += phi<TYPE>(__ldg(esn + c * plane + off) - __ldg(tan + c * plane + off));
        v[j] = s;
      }
      acc = make_float4(v[0], v[1], v[2], v[3]);
    }
    *reinterpret_cast<float4*>(&E[r][4 * k]) = acc;
  }
  __syncthreads();
  for (int it = tid; it < BE_H * (BT_W / 4); it += 256) {
    const int r = it / (BT_W / 4), q = it % (BT_W / 4);
    const float4* p = reinterpret_cast<const float4*>(&E[r][4 * q]);
    *reinterpret_cast<float4*>(&Hs[r][4 * q]) = hsum9x4(p[0], p[1], p[2]);
  }
  __syncthreads();
  {
    const int q = tid % 32, rs = tid / 32;  // 4 columns x 4 rows per thread
    float4 v[12];
#pragma unroll
    for (int j = 0; j < 12; ++j) v[j] = *reinterpret_cast<const float4*>(&Hs[rs * 4 + j][4 * q]);
    const float4 mid = add4(add4(add4(v[3], v[4]), add4(v[5], v[6])), add4(v[7], v[8]));
    const float4 l12 = add4(v[1], v[2]), r910 = add4(v[9], v[10]);
    float4 o[4];
    o[0] = add4(mid, add4(v[0], l12));
    o[1] = add4(mid, add4(l12, v[9]));
    o[2] = add4(mid, add4(v[2], r910));
    o[3] = add4(mid, add4(r910, v[11]));
    const int gx = x0 + 4 * q;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gy = y0 + rs * 4 + j;
      if (gy >= H) continue;
      float* dst = out + n * plane + (int64_t)gy * W + gx;
      const float4 r = make_float4(o[j].x * INV81, o[j].y * INV81, o[j].z * INV81, o[j].w * INV81);
      if (vec) {
        if (gx < W) *reinterpret_cast<float4*>(dst) = r;
      } else {
        if (gx + 0 < W) dst[0] = r.x;
        if (gx + 1 < W) dst[1] = r.y;
        if (gx + 2 < W) dst[2] = r.z;
        if (gx + 3 < W) dst[3] = r.w;
      }
    }
  }
}

// grad_in[c] = phi'(es[c]-ta[c]) / 81 * S(grad_out), S = adjoint of the replicate-clamped 9x9 box:
// a zero-padded box sum whose first/last row and column collect the extra clamp multiplicity
// (weights 5,4,3,2,1 over the five pixels nearest the border instead of 1,1,1,1,1).
template <int TYPE>
__global__ void __launch_bounds__(256)
photo_bwd_box9(const float* __restrict__ es, const float* __restrict__ ta, const float* __restrict__ go,
               float* __restrict__ gi, int C, int H, int W, int vec) {
  __shared__ __align__(16) float G[BE_H][BE_W];
  __shared__ __align__(16) float Hs[BE_H][BT_W];
  const int x0 = blockIdx.x * BT_W, y0 = blockIdx.y * BT_H;
  const int64_t n = blockIdx.z;
  const int tid = threadIdx.x;
  const int64_t plane = (int64_t)H * W;
  const float* gon = go + n * plane;

  for (int ch = tid; ch < BE_H * (BE_W / 4); ch += 256) {
    const int r = ch / (BE_W / 4), k = ch % (BE_W / 4);
    const int gy = y0 - R9 + r, gx = x0 - R9 + 4 * k;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (gy >= 0 && gy < H) {
      if (vec && gx >= 0 && gx + 3 < W) {
        v = ldg4(gon + (int64_t)gy * W + gx);
      } else {
        if (gx + 0 >= 0 && gx + 0 < W) v.x = __ldg(gon + (int64_t)gy * W + gx + 0);
        if (gx + 1 >= 0 && gx + 1 < W) v.y = __ldg(gon + (int64_t)gy * W + gx + 1);
        if (gx + 2 >= 0 && gx + 2 < W) v.z = __ldg(gon + (int64_t)gy * W + gx + 2);
        if (gx + 3 >= 0 && gx + 3 < W) v.w = __ldg(gon + (int64_t)gy * W + gx + 3);
      }
    }
    *reinterpret_cast<float4*>(&G[r][4 * k]) = v;
  }
  __syncthreads();
  const int xr = W - 1 - x0;  // tile-local column of the last image column
  for (int it = tid; it < BE_H * (BT_W / 4); it += 256) {
    const int r = it / (BT_W / 4), q = it % (BT_W / 4);
    const float4* p = reinterpret_cast<const float4*>(&G[r][4 * q]);
    const float4 a = p[0], b = p[1], c = p[2];
    float4 o = hsum9x4(a, b, c);
    if (x0 == 0 && q == 0) o.x += 4.f * b.x + 3.f * b.y + 2.f * b.z + b.w;
    if (xr >= 0 && xr < BT_W && q == xr / 4) {
      const float* g = &G[r][xr + R9];
      const float extra = 4.f * g[0] + 3.f * g[-1] + 2.f * g[-2] + g[-3];
      const int j = xr % 4;
      if (j == 0) o.x += extra;
      if (j == 1) o.y += extra;
      if (j == 2) o.z += extra;
      if (j == 3) o.w += extra;
    }
    *reinterpret_cast<float4*>(&Hs[r][4 * q]) = o;
  }
  __syncthreads();
  {
    const int q = tid % 32, rs = tid / 32;
    float4 v[12];
#pragma unroll
    for (int j = 0; j < 12; ++j) v[j] = *reinterpret_cast<const float4*>(&Hs[rs * 4 + j][4 * q]);
    const float4 mid = add4(add4(add4(v[3], v[4]), add4(v[5], v[6])), add4(v[7], v[8]));
    const float4 l12 = add4(v[1], v[2]), r910 = add4(v[9], v[10]);
    float4 o[4];
    o[0] = add4(mid, add4(v[0], l12));
    o[1] = add4(mid, add4(l12, v[9]));
    o[2] = add4(mid, add4(v[2], r910));
    o[3] = add4(mid, add4(r910, v[11]));
    const int gx = x0 + 4 * q;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gy = y0 + rs * 4 + j;
      if (gy >= H) continue;
      float4 s = o[j];
      // output row gy sits at padded row (rs*4 + j + 4) = v[j + 4]
      if (gy == 0) s = fma4s(4.f, v[j + 4], fma4s(3.f, v[j + 5], fma4s(2.f, v[j + 6], add4(s, v[j + 7]))));
      if (gy == H - 1) s = fma4s(4.f, v[j + 4], fma4s(3.f, v[j + 3], fma4s(2.f, v[j + 2], add4(s, v[j + 1]))));
      const int64_t off = (int64_t)gy * W + gx;
      for (int c = 0; c < C; ++c) {
        const float* ep = es + (n * C + c) * plane + off;
        const float* tp = ta + (n * C + c) * plane + off;
        float* gp = gi + (n * C + c) * plane + off;
        if (vec) {
          if (gx < W) {
            const float4 e = ldg4(ep), t = ldg4(tp);
            float4 r;
            if (TYPE == 0) {
              r = make_float4(2.f * (e.x - t.x) * INV81 * s.x, 2.f * (e.y - t.y) * INV81 * s.y,
                              2.f * (e.z - t.z) * INV81 * s.z, 2.f * (e.w - t.w) * INV81 * s.w);
            } else {
              r = make_float4(sgn(e.x - t.x) * INV81 * s.x, sgn(e.y - t.y) * INV81 * s.y,
                              sgn(e.z - t.z) * INV81 * s.z, sgn(e.w - t.w) * INV81 * s.w);
            }
            *reinterpret_cast<float4*>(gp) = r;
          }
        } else {
          const float sv[4] = {s.x, s.y, s.z, s.w};
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (gx + k < W) {
              const float d = __ldg(ep + k) - __ldg(tp + k);
              gp[k] = (TYPE == 0 ? 2.f * d : sgn(d)) * INV81 * sv[k];
            }
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// fast path, block size 9, fp32: census_mse / census_sad
// ------------------------------------------------------------------------------------------
#ifndef CTD_CT_H
#define CTD_CT_H 16
#endif
constexpr int CT_W = 64, CT_H = CTD_CT_H;  // output tile; 16 rows of threads, CT_H / 16 passes
constexpr int CT_NH = CT_H / 16;
#ifndef CTD_CB_NPX
#define CTD_CB_NPX 2
#endif
constexpr int CB_NPX = CTD_CB_NPX;  // pixels per thread and pass in the census backward
#ifndef CTD_CB_MINB
#define CTD_CB_MINB 3  // resident CTAs per SM the census backward is compiled for (4 = 64 registers: measured slower / spills)
#endif
#ifndef CTD_CB_H
#define CTD_CB_H 16
#endif
constexpr int CB_H = CTD_CB_H;        // tile rows of the census backward (64 x CB_H outputs per CTA)
constexpr int CBE_H = CB_H + 8;       // its halo tile rows
static_assert(CT_H % 16 == 0, "census tile height");
constexpr int CE_W = CT_W + 2 * R9;  // 72
constexpr int CE_H = CT_H + 2 * R9;  // 40

// ---- the disparity warp in front of the loss (model/networks.py:362-371), same arithmetic as warp.cu ----------------
struct WarpArgs {
  const float* pattern;  // [Bp,1,Hp,Wp]
  float* proj;           // pattern_proj out [B,1,H,W]
  int Bp, Hp, Wp;
  float inv_w, inv_h;    // 1 / (W - 1), 1 / (H - 1)
};

struct WarpTaps {
  float nw, ne, sw, se, wy0, wy1, mult_x;  // the four pattern values (0 outside), the row weights, d ix / d gx
  float ix, iy;
  int x0, y0;
};

__device__ __forceinline__ WarpTaps warp_taps(const float* __restrict__ p, float disp, int u, int v, float inv_w, float inv_h, int Hp, int Wp) {
  WarpTaps t;
  const float gx = 2.f * __fsub_rn(__fmul_rn(__fsub_rn((float)u, disp), inv_w), 0.5f);
  const float gy = 2.f * __fsub_rn(__fmul_rn((float)v, inv_h), 0.5f);
  float ix = fmaf(gx + 1.f, (float)Wp, -1.f) / 2.f, iy = fmaf(gy + 1.f, (float)Hp, -1.f) / 2.f;
  t.mult_x = (float)Wp / 2.f;
  if (ix <= 0.f) {
    ix = 0.f;
    t.mult_x = 0.f;
  } else if (ix >= (float)(Wp - 1)) {
    ix = (float)(Wp - 1);
    t.mult_x = 0.f;
  }
  iy = fminf((float)(Hp - 1), fmaxf(iy, 0.f));
  t.ix = ix;
  t.iy = iy;
  t.x0 = (int)floorf(ix);
  t.y0 = (int)floorf(iy);
  const bool xin = t.x0 + 1 < Wp, yin = t.y0 + 1 < Hp;
  const float* r0 = p + t.y0 * Wp + t.x0;
  t.nw = __ldg(r0);
  t.ne = xin ? __ldg(r0 + 1) : 0.f;
  t.sw = yin ? __ldg(r0 + Wp) : 0.f;
  t.se = xin && yin ? __ldg(r0 + Wp + 1) : 0.f;
  t.wy1 = (float)(t.y0 + 1) - iy;
  t.wy0 = iy - (float)t.y0;
  return t;
}

// grid_sample value: ATen's nw, ne, sw, se accumulation (taps outside the pattern are skipped there; adding 0 * w is the same)
__device__ __forceinline__ float warp_value(const WarpTaps& t) {
  const float x1 = (float)(t.x0 + 1), fx0 = (float)t.x0;
  float acc = 0.f;
  acc = fmaf(t.nw, (x1 - t.ix) * t.wy1, acc);
  acc = fmaf(t.ne, (t.ix - fx0) * t.wy1, acc);
  acc = fmaf(t.sw, (x1 - t.ix) * t.wy0, acc);
  acc = fmaf(t.se, (t.ix - fx0) * t.wy0, acc);
  return acc;
}

// d pattern_proj / d disp times g (warp_bwd_kernel's sequence)
__device__ __forceinline__ float warp_grad_disp(const WarpTaps& t, float g, float inv_w) {
  float gix = 0.f;
  gix -= t.nw * t.wy1 * g;
  gix += t.ne * t.wy1 * g;
  gix -= t.sw * t.wy0 * g;
  gix += t.se * t.wy0 * g;
  return -__fmul_rn(2.f * (t.mult_x * gix), inv_w);
}

// the estimate's halo tile computed on the fly: es = pattern warped by the disparity, replicate-clamped like load_halo_tile<true>;
// the tile's own pixels are also written out as pattern_proj (the reference returns it, networks.py:378)
template <int ROWS, int OWN_H>
__device__ __forceinline__ void load_warp_tile(float (*S)[72], const WarpArgs& wa, const float* __restrict__ pat,
                                               const float* __restrict__ disp, float* __restrict__ proj, int x0, int y0, int H, int W,
                                               int tid) {
  for (int i = tid; i < ROWS * 72; i += 256) {
    const int r = i / 72, c = i % 72;
    const int uy = y0 - 4 + r, ux = x0 - 4 + c;
    const int gy = clampi(uy, 0, H - 1), gx = clampi(ux, 0, W - 1);
    const WarpTaps t = warp_taps(pat, __ldg(disp + (int64_t)gy * W + gx), gx, gy, wa.inv_w, wa.inv_h, wa.Hp, wa.Wp);
    const float v = warp_value(t);
    S[r][c] = v;
    if (r >= 4 && r < 4 + OWN_H && c >= 4 && c < 68 && uy < H && ux < W) proj[(int64_t)uy * W + ux] = v;
  }
}

// load a (CE_H x CE_W) halo tile; REPL: replicate-clamped (es, ta), else zero padded (grad_out)
template <bool REPL, int ROWS = CE_H>
__device__ __forceinline__ void load_halo_tile(float (*S)[CE_W], const float* __restrict__ src, int x0,
                                               int y0, int H, int W, int vec, int tid) {
  for (int ch = tid; ch < ROWS * (CE_W / 4); ch += 256) {
    const int r = ch / (CE_W / 4), k = ch % (CE_W / 4);
    int gy = y0 - R9 + r;
    const int gx = x0 - R9 + 4 * k;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    const bool row_ok = gy >= 0 && gy < H;
    if (REPL) gy = clampi(gy, 0, H - 1);
    if (REPL || row_ok) {
      const float* row = src + (int64_t)gy * W;
      if (vec && gx >= 0 && gx + 3 < W) {
        v = ldg4(row + gx);
      } else if (REPL) {
        v.x = __ldg(row + clampi(gx + 0, 0, W - 1));
        v.y = __ldg(row + clampi(gx + 1, 0, W - 1));
        v.z = __ldg(row + clampi(gx + 2, 0, W - 1));
        v.w = __ldg(row + clampi(gx + 3, 0, W - 1));
      } else {
        if (gx + 0 >= 0 && gx + 0 < W) v.x = __ldg(row + gx + 0);
        if (gx + 1 >= 0 && gx + 1 < W) v.y = __ldg(row + gx + 1);
        if (gx + 2 >= 0 && gx + 2 < W) v.z = __ldg(row + gx + 2);
        if (gx + 3 >= 0 && gx + 3 < W) v.w = __ldg(row + gx + 3);
      }
    }
    *reinterpret_cast<float4*>(&S[r][4 * k]) = v;
  }
}

__device__ __forceinline__ void unpack12(float* d, const float* srow) {
  const float4* p = reinterpret_cast<const float4*>(srow);
  const float4 a = p[0], b = p[1], c = p[2];
  d[0] = a.x; d[1] = a.y; d[2] = a.z; d[3] = a.w;
  d[4] = b.x; d[5] = b.y; d[6] = b.z; d[7] = b.w;
  d[8] = c.x; d[9] = c.y; d[10] = c.z; d[11] = c.w;
}

// out = sum over the window of psi(h(es_tap - es_ctr) - h(ta_tap - ta_ctr)) / 81,
// h(x) = (1 + x / sqrt(x^2 + eps)) / 2; psi = square (census_mse) or abs (census_sad).
template <int TYPE>
__global__ void __launch_bounds__(256)
photo_fwd_census9(const float* __restrict__ es, const float* __restrict__ ta, float* __restrict__ out,
                  int C, int H, int W, float eps, int vec) {
  __shared__ __align__(16) float Es[CE_H][CE_W];
  __shared__ __align__(16) float Ts[CE_H][CE_W];
  const int x0 = blockIdx.x * CT_W, y0 = blockIdx.y * CT_H;
  const int64_t n = blockIdx.z;
  const int tid = threadIdx.x;
  const int tx = tid % 16, ty = tid / 16;
  const int64_t plane = (int64_t)H * W;
  float acc[CT_NH][4] = {};
  for (int c = 0; c < C; ++c) {
    if (c) __syncthreads();
    load_halo_tile<true>(Es, es + (n * C + c) * plane, x0, y0, H, W, vec, tid);
    load_halo_tile<true>(Ts, ta + (n * C + c) * plane, x0, y0, H, W, vec, tid);
    __syncthreads();
#pragma unroll
    for (int half = 0; half < CT_NH; ++half) {
      const int yl = ty + 16 * half;
      if (y0 + yl >= H) continue;
      const float4 ec4 = *reinterpret_cast<const float4*>(&Es[yl + R9][4 * tx + R9]);
      const float4 tc4 = *reinterpret_cast<const float4*>(&Ts[yl + R9][4 * tx + R9]);
      const float ec[4] = {ec4.x, ec4.y, ec4.z, ec4.w}, tc[4] = {tc4.x, tc4.y, tc4.z, tc4.w};
#pragma unroll 1
      for (int dy = 0; dy < 9; ++dy) {
        float e[12], t[12];
        unpack12(e, &Es[yl + dy][4 * tx]);
        unpack12(t, &Ts[yl + dy][4 * tx]);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
#pragma unroll
          for (int dx = 0; dx < 9; ++dx) {
            const float des = e[k + dx] - ec[k];
            const float dta = t[k + dx] - tc[k];
            const float r1 = rsqrt_approx(fmaf(des, des, eps));
            const float r2 = rsqrt_approx(fmaf(dta, dta, eps));
            const float dd = fmaf(des, r1, -(dta * r2));  // = 2 * (h(des) - h(dta))
            if (TYPE == 2) acc[half][k] = fmaf(dd, dd, acc[half][k]);
            else acc[half][k] += fabsf(dd);
          }
        }
      }
    }
  }
  const float scale = (TYPE == 2 ? 0.25f : 0.5f) * INV81;
#pragma unroll
  for (int half = 0; half < CT_NH; ++half) {
    const int gy = y0 + ty + 16 * half, gx = x0 + 4 * tx;
    if (gy >= H) continue;
    float* dst = out + n * plane + (int64_t)gy * W + gx;
    if (vec) {
      if (gx < W)
        *reinterpret_cast<float4*>(dst) = make_float4(acc[half][0] * scale, acc[half][1] * scale,
                                                      acc[half][2] * scale, acc[half][3] * scale);
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (gx + k < W) dst[k] = acc[half][k] * scale;
    }
  }
}

// census_sad backward takes sign(h(des) - h(dta)); the fast path evaluates the difference with
// rsqrt.approx (|error| < ~1.2e-6 on dd = 2 * difference).  A pixel whose window holds a term closer to
// zero than SIGN_GUARD is not trusted: the tile pass notes it in a shared-memory list and, once the tile is
// done, the CTA's warps recompute exactly those pixels from the SAME staged tiles with the reference's own
// IEEE operation sequence (ext.h:321-330), one warp per pixel, lane l evaluating taps l, l+32, l+64 of the
// 9x9 window in both roles of the pixel.  The sign decisions -- and therefore the gradient -- then match the
// CPU extension exactly, the hot loop stays branch-free, and no second kernel, list in global memory or
// memset is involved (about one pixel in a thousand takes this path on the bench data).
constexpr float SIGN_GUARD = 3e-6f;

// (xl, yl): pixel inside the CTA's tile; Es/Ts are replicate-clamped halo tiles, Gs is zero outside the image
__device__ __forceinline__ float census_sad_bwd_exact_smem(float (*Es)[CE_W], float (*Ts)[CE_W], float (*Gs)[CE_W], int xl,
                                                           int yl, int x, int y, int H, int W, float eps, int lane) {
  const float ei = Es[yl + R9][xl + R9], ti = Ts[yl + R9][xl + R9], gc = Gs[yl + R9][xl + R9];
  float acc = 0.f;
  for (int t = lane; t < 81; t += 32) {
    const int dy = t / 9 - R9, dx = t % 9 - R9;
    const float des = ei - Es[yl + R9 + dy][xl + R9 + dx], dta = ti - Ts[yl + R9 + dy][xl + R9 + dx];
    // role "pixel is the tap of centre q": only real q (Gs is zero elsewhere), weighted by how many of q's
    // offsets clamp onto the pixel
    const float mx = x == 0 ? float(R9 + 1 - dx) : (x == W - 1 ? float(R9 + 1 + dx) : 1.f);
    const float my = y == 0 ? float(R9 + 1 - dy) : (y == H - 1 ? float(R9 + 1 + dy) : 1.f);
    const float gq = Gs[yl + R9 + dy][xl + R9 + dx] * (mx * my);
    const float s = __fadd_rn(__fmul_rn(des, des), eps);
    const float q1 = __fdiv_rn(des, __fsqrt_rn(s));
    const float q2 = __fdiv_rn(dta, __fsqrt_rn(__fadd_rn(__fmul_rn(dta, dta), eps)));
    const float d_tap = __fsub_rn(0.5f * __fadd_rn(1.f, q1), 0.5f * __fadd_rn(1.f, q2));
    // role "pixel is the centre, q the tap": des flips sign exactly, so do the quotients
    const float d_ctr = __fsub_rn(0.5f * __fadd_rn(1.f, -q1), 0.5f * __fadd_rn(1.f, -q2));
    const float r1 = rsqrt_approx(s);
    acc = fmaf(r1 * r1 * r1, sgn(d_tap) * gq - sgn(d_ctr) * gc, acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  return acc * (0.5f * eps * INV81);
}

__device__ __forceinline__ float xor_sign(float v, float s) {  // v * sign(s) for s != 0
  return __int_as_float(__float_as_int(v) ^ (__float_as_int(s) & 0x80000000));
}

// grad_in[i] = eps/(2*81) * sum_q gl(dd) * r1^3 * (M(i,q) * go[q] + go[i]) over the 9x9 window of i:
// the first summand is i as a tap of centre q (M = clamp multiplicity, 1 away from the image
// border), the second is i as the centre scattering -g back to itself; both share dd and r1
// because h(-x) = 1 - h(x).  go is zero outside the image, es/ta are replicate-clamped.
// FUSE: also accumulate the forward's psi(dd) over the same 81 (replicate-clamped) taps into facc[half][k] --
// the backward evaluates every dd the forward needs, so the loss map costs one more add per tap.
// NPX pixels per thread and pass (4: 16 rows of 16 threads, 128-bit shared loads; 2: 8 rows of 32 threads, 64-bit
// loads, fewer registers -> three CTAs per SM).
template <int NPX>
__device__ __forceinline__ void unpack_row(float* d, const float* srow) {  // NPX + 8 values from column NPX * tx
  if (NPX == 4) {
    unpack12(d, srow);
  } else {
    const float2* p = reinterpret_cast<const float2*>(srow);
#pragma unroll
    for (int q = 0; q < (NPX + 8) / 2; ++q) {
      const float2 v = p[q];
      d[2 * q] = v.x;
      d[2 * q + 1] = v.y;
    }
  }
}

template <int TYPE, bool BORDER, bool FUSE, int NPX, bool WARP = false>
__device__ __forceinline__ void census_bwd_tile(float (*Es)[CE_W], float (*Ts)[CE_W], float (*Gs)[CE_W],
                                                float* __restrict__ gi, int x0, int y0, int H, int W,
                                                float eps, int vec, int tx, int ty, unsigned short* s_fix, unsigned* s_nfix,
                                                float (*facc)[NPX], const WarpArgs* wa = nullptr, const float* __restrict__ pat = nullptr,
                                                const float* __restrict__ disp = nullptr) {
  constexpr int RPP = 256 / (CT_W / NPX);  // tile rows per pass
#pragma unroll 1
  for (int half = 0; half < CB_H / RPP; ++half) {
    const int yl = ty + RPP * half;
    const int gy = y0 + yl, gx = x0 + NPX * tx;
    if (gy >= H) continue;
    float ec[NPX], tc[NPX], gc[NPX];
#pragma unroll
    for (int k = 0; k < NPX; ++k) {
      ec[k] = Es[yl + R9][NPX * tx + R9 + k];
      tc[k] = Ts[yl + R9][NPX * tx + R9 + k];
      gc[k] = Gs[yl + R9][NPX * tx + R9 + k];
    }
    float acc[NPX], near0[NPX];  // near0 (census_sad): smallest |dd| over the window (centre tap excluded)
    // clamp multiplicity of the column / row offset d (-4..4): base + slope * d
    float bx[NPX], sx[NPX], by = 1.f, sy = 0.f;
#pragma unroll
    for (int k = 0; k < NPX; ++k) {
      acc[k] = 0.f;
      near0[k] = 1.f;
      bx[k] = 1.f;
      sx[k] = 0.f;
    }
    if (BORDER) {
#pragma unroll
      for (int k = 0; k < NPX; ++k) {
        if (gx + k == 0) { bx[k] = 5.f; sx[k] = -1.f; }
        if (gx + k == W - 1) { bx[k] = 5.f; sx[k] = 1.f; }
      }
      if (gy == 0) { by = 5.f; sy = -1.f; }
      if (gy == H - 1) { by = 5.f; sy = 1.f; }
    }
    if constexpr (NPX == 2) {
      // Two taps per instruction: Blackwell's packed fp32 pipe instructions (FADD2 / FMUL2 / FFMA2 on aligned register
      // pairs) halve the issue slots of everything around the reciprocal square roots, which is what this loop is
      // short of (80 % of the issue slots against 66 % of the XU pipe with scalar code).  A row's ten staged values
      // arrive as five aligned pairs; pixel 0 takes (0,1) .. (6,7) as tap pairs and column 8 alone, pixel 1 takes
      // (2,3) .. (8,9) and column 1 alone.  acc2 / fac2 hold the even- and odd-tap partial sums.
      float2 acc2[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
      float2 fac2[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
      const float2 eps2 = make_float2(eps, eps);
#pragma unroll 1
      for (int dy = 0; dy < 9; ++dy) {
        float2 e2[5], t2[5], g2[5];
#pragma unroll
        for (int q = 0; q < 5; ++q) {
          e2[q] = reinterpret_cast<const float2*>(&Es[yl + dy][2 * tx])[q];
          t2[q] = reinterpret_cast<const float2*>(&Ts[yl + dy][2 * tx])[q];
          g2[q] = reinterpret_cast<const float2*>(&Gs[yl + dy][2 * tx])[q];
        }
        const float my = BORDER ? fmaf(sy, float(dy - R9), by) : 1.f;
        const bool ctr_row = dy == R9 || (BORDER && ((sy < 0.f && dy < R9) || (sy > 0.f && dy > R9)));
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const float2 ec2 = make_float2(ec[k], ec[k]), tc2 = make_float2(tc[k], tc[k]), gc2 = make_float2(gc[k], gc[k]);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int dx = 2 * q + k;  // the pair's first tap; staged columns k + dx = 2 (q + k), + 1
            const float2 ev = e2[q + k], tv = t2[q + k];
            const float2 des = __fadd2_rn(ec2, make_float2(-ev.x, -ev.y));
            const float2 nta = __fadd2_rn(tv, make_float2(-tc2.x, -tc2.y));  // -(tc - t)
            const float2 s1 = __ffma2_rn(des, des, eps2), s2 = __ffma2_rn(nta, nta, eps2);
            const float2 r1 = make_float2(rsqrt_approx(s1.x), rsqrt_approx(s1.y));
            const float2 r2 = make_float2(rsqrt_approx(s2.x), rsqrt_approx(s2.y));
            const float2 dd = __ffma2_rn(des, r1, __fmul2_rn(nta, r2));
            const float2 r3 = __fmul2_rn(__fmul2_rn(r1, r1), r1);
            float2 gq = g2[q + k];
            if (BORDER) {
              const float2 wx = __ffma2_rn(make_float2(sx[k], sx[k]), make_float2(float(dx - R9), float(dx + 1 - R9)), make_float2(bx[k], bx[k]));
              gq = __fmul2_rn(gq, __fmul2_rn(wx, make_float2(my, my)));
            }
            const float2 gs = __fadd2_rn(gq, gc2);
            if (FUSE) {
              if (TYPE == 2) fac2[k] = __ffma2_rn(dd, dd, fac2[k]);
              else fac2[k] = __fadd2_rn(fac2[k], make_float2(fabsf(dd.x), fabsf(dd.y)));
            }
            if (TYPE == 2) {
              acc2[k] = __ffma2_rn(__fmul2_rn(dd, r3), gs, acc2[k]);
            } else {
              const float2 sr3 = make_float2(__uint_as_float(__float_as_uint(r3.x) | (__float_as_uint(dd.x) & 0x80000000u)),
                                             __uint_as_float(__float_as_uint(r3.y) | (__float_as_uint(dd.y) & 0x80000000u)));
              acc2[k] = __ffma2_rn(sr3, gs, acc2[k]);
              float m0 = fabsf(dd.x), m1 = fabsf(dd.y);
              if (dx == R9 || BORDER) {
                const bool cc = dx == R9 || (BORDER && (dx < R9 ? sx[k] < 0.f : sx[k] > 0.f));
                m0 = (ctr_row && cc) ? 1.f : m0;
              }
              if (dx + 1 == R9 || BORDER) {
                const bool cc = dx + 1 == R9 || (BORDER && (dx + 1 < R9 ? sx[k] < 0.f : sx[k] > 0.f));
                m1 = (ctr_row && cc) ? 1.f : m1;
              }
              near0[k] = fminf(near0[k], fminf(m0, m1));
            }
          }
          {  // the ninth tap: staged column 8 for pixel 0 (dx = 8), staged column 1 for pixel 1 (dx = 0)
            const int dx = k == 0 ? 8 : 0;
            const float ev = k == 0 ? e2[4].x : e2[0].y, tv = k == 0 ? t2[4].x : t2[0].y;
            const float des = ec[k] - ev;
            const float dta = tc[k] - tv;
            const float r1 = rsqrt_approx(fmaf(des, des, eps));
            const float r2 = rsqrt_approx(fmaf(dta, dta, eps));
            const float dd = fmaf(des, r1, -(dta * r2));
            const float r3 = r1 * r1 * r1;
            float gq = k == 0 ? g2[4].x : g2[0].y;
            if (BORDER) gq *= my * fmaf(sx[k], float(dx - R9), bx[k]);
            if (FUSE) {
              if (TYPE == 2) fac2[k].x = fmaf(dd, dd, fac2[k].x);
              else fac2[k].x += fabsf(dd);
            }
            if (TYPE == 2) {
              acc2[k].x = fmaf(dd * r3, gq + gc[k], acc2[k].x);
            } else {
              const float sr3 = __uint_as_float(__float_as_uint(r3) | (__float_as_uint(dd) & 0x80000000u));
              acc2[k].x = fmaf(sr3, gq + gc[k], acc2[k].x);
              float mag = fabsf(dd);
              if (BORDER) mag = (ctr_row && (dx < R9 ? sx[k] < 0.f : sx[k] > 0.f)) ? 1.f : mag;
              near0[k] = fminf(near0[k], mag);
            }
          }
        }
      }
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        acc[k] = acc2[k].x + acc2[k].y;
        if (FUSE) facc[half][k] += fac2[k].x + fac2[k].y;
      }
    } else {
#pragma unroll 1
    for (int dy = 0; dy < 9; ++dy) {
      float e[NPX + 8], t[NPX + 8], g[NPX + 8];
      unpack_row<NPX>(e, &Es[yl + dy][NPX * tx]);
      unpack_row<NPX>(t, &Ts[yl + dy][NPX * tx]);
      unpack_row<NPX>(g, &Gs[yl + dy][NPX * tx]);
      const float my = BORDER ? fmaf(sy, float(dy - R9), by) : 1.f;
      // rows whose clamped tap row is the pixel's own row: the centre row, and at the first / last image row
      // every window row beyond the border
      const bool ctr_row = dy == R9 || (BORDER && ((sy < 0.f && dy < R9) || (sy > 0.f && dy > R9)));
#pragma unroll
      for (int k = 0; k < NPX; ++k) {
#pragma unroll
        for (int dx = 0; dx < 9; ++dx) {
          const float des = ec[k] - e[k + dx];
          const float dta = tc[k] - t[k + dx];
          const float r1 = rsqrt_approx(fmaf(des, des, eps));
          const float r2 = rsqrt_approx(fmaf(dta, dta, eps));
          const float dd = fmaf(des, r1, -(dta * r2));
          const float r3 = r1 * r1 * r1;
          float gq = g[k + dx];
          if (BORDER) gq *= my * fmaf(sx[k], float(dx - R9), bx[k]);
          if (FUSE) {
            if (TYPE == 2) facc[half][k] = fmaf(dd, dd, facc[half][k]);
            else facc[half][k] += fabsf(dd);
          }
          if (TYPE == 2) {
            acc[k] = fmaf(dd * r3, gq + gc[k], acc[k]);
          } else {
            // sign(dd) * r3: r3 > 0, so OR-ing in dd's sign bit is one LOP3.  The centre tap (dd = +0,
            // sign(0) = 0 in the reference) comes out as +r3 * G here and is subtracted after the loop.
            const float sr3 = __uint_as_float(__float_as_uint(r3) | (__float_as_uint(dd) & 0x80000000u));
            acc[k] = fmaf(sr3, gq + gc[k], acc[k]);
            float mag = fabsf(dd);
            // a tap that clamps onto the pixel itself has dd = +0 exactly (sign 0 in the reference): not a
            // near-tie; its +r3 * G contribution is taken out after the loop
            const bool ctr_col = dx == R9 || (BORDER && (dx < R9 ? sx[k] < 0.f : sx[k] > 0.f));
            if (dx == R9 || BORDER) mag = (ctr_row && ctr_col) ? 1.f : mag;
            near0[k] = fminf(near0[k], mag);
          }
        }
      }
    }
    }
    if (TYPE == 3) {
      // self taps: the centre (counted with M(i,i) = bx*by as a tap of itself, plus once as the centre) and, at
      // the image border, the bx*by - 1 window positions outside the image that clamp back onto the pixel
      // (no real centre there, so only the "pixel as centre" half): r0^3 * gc * (2 * bx*by) in total
      const float r0 = rsqrt_approx(eps);
#pragma unroll
      for (int k = 0; k < NPX; ++k) acc[k] -= r0 * r0 * r0 * (2.f * bx[k] * by) * gc[k];
    }
    const float scale = 0.5f * eps * INV81;
    float r[NPX];
#pragma unroll
    for (int k = 0; k < NPX; ++k) {
      r[k] = acc[k] * scale;
    }
    if (TYPE == 3) {  // near-tie pixels: noted for the exact pass that follows the tile (rare)
#pragma unroll
      for (int k = 0; k < NPX; ++k)
        if (near0[k] < SIGN_GUARD && gx + k < W) s_fix[atomicAdd(s_nfix, 1u)] = (unsigned short)(yl * CT_W + NPX * tx + k);
    }
    if (WARP) {  // chain through the warp: the gradient w.r.t. the disparity leaves the kernel, not the one w.r.t. es
#pragma unroll
      for (int k = 0; k < NPX; ++k)
        if (gx + k < W) {
          const WarpTaps t = warp_taps(pat, __ldg(disp + (int64_t)gy * W + gx + k), gx + k, gy, wa->inv_w, wa->inv_h, wa->Hp, wa->Wp);
          r[k] = warp_grad_disp(t, r[k], wa->inv_w);
        }
    }
    float* dst = gi + (int64_t)gy * W + gx;
    if (vec) {
      if (gx < W) {
        if (NPX == 4) *reinterpret_cast<float4*>(dst) = make_float4(r[0], r[1], r[2], r[NPX - 1]);
        else *reinterpret_cast<float2*>(dst) = make_float2(r[0], r[1]);
      }
    } else {
#pragma unroll
      for (int k = 0; k < NPX; ++k)
        if (gx + k < W) dst[k] = r[k];
    }
  }
}

// WARP: `es` is the DISPARITY; the estimate's tile is the pattern warped by it on the fly (model/networks.py:362-371), the
// tile's own pixels go out as pattern_proj, and `gi` receives d loss / d disp (C = 1).
template <int TYPE, bool FUSE, int NPX, bool WARP = false>
__global__ void __launch_bounds__(256, NPX == 4 ? 2 : CTD_CB_MINB)
photo_bwd_census9(const float* __restrict__ es, const float* __restrict__ ta, const float* __restrict__ go,
                  float* __restrict__ gi, float* __restrict__ out, int C, int H, int W, float eps, int vec,
                  const float* __restrict__ mask, double* __restrict__ partials, unsigned* __restrict__ ticket,
                  float* __restrict__ sums2, const WarpArgs wa = WarpArgs()) {
  __shared__ __align__(16) float Es[CBE_H][CE_W];
  __shared__ __align__(16) float Ts[CBE_H][CE_W];
  __shared__ __align__(16) float Gs[CBE_H][CE_W];
  __shared__ unsigned short s_fix[CT_W * CB_H];  // tile-local indices of the near-tie pixels of this channel
  __shared__ unsigned s_nfix;
  const int x0 = blockIdx.x * CT_W, y0 = blockIdx.y * CB_H;
  const int64_t n = blockIdx.z;
  const int tid = threadIdx.x;
  constexpr int TXN = CT_W / NPX, RPP = 256 / TXN, NP = CB_H / RPP;
  static_assert(CB_H % RPP == 0, "census backward tile height");
  const int tx = tid % TXN, ty = tid / TXN;
  const int64_t plane = (int64_t)H * W;
  const bool border = x0 == 0 || y0 == 0 || x0 + CT_W >= W || y0 + CB_H >= H;
  float facc[NP][NPX] = {};
  load_halo_tile<false, CBE_H>(Gs, go + n * plane, x0, y0, H, W, vec, tid);
  for (int c = 0; c < C; ++c) {
    if (c) __syncthreads();
    if (tid == 0) s_nfix = 0;
    const float* pat = WARP ? wa.pattern + (wa.Bp == 1 ? 0 : n) * (int64_t)wa.Hp * wa.Wp : nullptr;
    const float* dpl = es + (n * C + c) * plane;  // WARP: the disparity plane
    if (WARP) load_warp_tile<CBE_H, CB_H>(Es, wa, pat, dpl, wa.proj + n * plane, x0, y0, H, W, tid);
    else load_halo_tile<true, CBE_H>(Es, es + (n * C + c) * plane, x0, y0, H, W, vec, tid);
    load_halo_tile<true, CBE_H>(Ts, ta + (n * C + c) * plane, x0, y0, H, W, vec, tid);
    __syncthreads();
    float* gic = gi + (n * C + c) * plane;
    if (border) census_bwd_tile<TYPE, true, FUSE, NPX, WARP>(Es, Ts, Gs, gic, x0, y0, H, W, eps, vec, tx, ty, s_fix, &s_nfix, facc, &wa, pat, dpl);
    else census_bwd_tile<TYPE, false, FUSE, NPX, WARP>(Es, Ts, Gs, gic, x0, y0, H, W, eps, vec, tx, ty, s_fix, &s_nfix, facc, &wa, pat, dpl);
    if (TYPE == 3) {  // exact pass over the near-tie pixels of this tile, straight from the staged tiles
      __syncthreads();
      const unsigned nfix = s_nfix;
      for (unsigned i = tid >> 5; i < nfix; i += 8) {
        const int li = s_fix[i], yl = li / CT_W, xl = li % CT_W;
        float v = census_sad_bwd_exact_smem(Es, Ts, Gs, xl, yl, x0 + xl, y0 + yl, H, W, eps, tid & 31);
        if ((tid & 31) == 0) {
          if (WARP) {
            const int64_t o = (int64_t)(y0 + yl) * W + x0 + xl;
            v = warp_grad_disp(warp_taps(pat, __ldg(dpl + o), x0 + xl, y0 + yl, wa.inv_w, wa.inv_h, wa.Hp, wa.Wp), v, wa.inv_w);
          }
          gic[(int64_t)(y0 + yl) * W + x0 + xl] = v;
        }
      }
    }
  }
  if (FUSE) {  // the loss map: sum over channels and taps, same scaling as photo_fwd_census9
    const float scale = (TYPE == 2 ? 0.25f : 0.5f) * INV81;
    float mnum = 0.f, mden = 0.f;  // optional: this thread's share of sum(mask * loss) and sum(mask)
#pragma unroll
    for (int half = 0; half < NP; ++half) {
      const int gy = y0 + ty + RPP * half, gx = x0 + NPX * tx;
      if (gy >= H) continue;
      if (mask != nullptr) {
        const float* mp = mask + n * plane + (int64_t)gy * W + gx;
        float m[NPX];
        if (vec && NPX == 2 && gx < W) {
          const float2 m2 = __ldg(reinterpret_cast<const float2*>(mp));
          m[0] = m2.x;
          m[NPX - 1] = m2.y;
        } else {
#pragma unroll
          for (int k = 0; k < NPX; ++k) m[k] = gx + k < W ? __ldg(mp + k) : 0.f;
        }
#pragma unroll
        for (int k = 0; k < NPX; ++k)
          if (gx + k < W) {
            mnum = fmaf(m[k], facc[half][k] * scale, mnum);
            mden += m[k];
          }
      }
      float* dst = out + n * plane + (int64_t)gy * W + gx;
      if (vec) {
        if (gx < W) {
          if (NPX == 4)
            *reinterpret_cast<float4*>(dst) = make_float4(facc[half][0] * scale, facc[half][1] * scale, facc[half][2] * scale,
                                                          facc[half][NPX - 1] * scale);
          else
            *reinterpret_cast<float2*>(dst) = make_float2(facc[half][0] * scale, facc[half][1] * scale);
        }
      } else {
#pragma unroll
        for (int k = 0; k < NPX; ++k)
          if (gx + k < W) dst[k] = facc[half][k] * scale;
      }
    }
    if (mask != nullptr) finish_masked_sums((double)mnum, (double)mden, partials, ticket, sums2);  // block-uniform branch
  }
}

// ------------------------------------------------------------------------------------------
// dispatch
// ------------------------------------------------------------------------------------------
static inline bool fast9_ok(int bs, int64_t H, int64_t W) {
  return !g_force_generic && bs == 9 && H >= 9 && W >= 9 && H * W < (int64_t)1 << 31;
}

static int check_common(const void* a, const void* b, const void* c, int64_t B, int64_t C, int64_t H,
                        int64_t W, int bs, int type) {
  CTD_REQUIRE(B >= 0 && C >= 0 && H >= 0 && W >= 0, "photometric: negative size");
  CTD_REQUIRE(bs >= 1 && bs <= 255, "photometric: block_size %d out of range [1,255]", bs);
  CTD_REQUIRE(type >= 0 && type <= 3, "photometric: invalid loss type %d", type);
  CTD_REQUIRE(H <= INT32_MAX && W <= INT32_MAX && C <= INT32_MAX, "photometric: dimension too large");
  if (B * C * H * W > 0) CTD_REQUIRE(a && b && c, "photometric: null pointer");
  return CTD_OK;
}

template <typename T>
static int fwd_impl(const T* es, const T* ta, T* out, int64_t B, int64_t C, int64_t H, int64_t W, int bs,
                    int type, float eps, cudaStream_t st) {
  if (int rc = check_common(es, ta, out, B, C, H, W, bs, type)) return rc;
  if (B * H * W == 0) return CTD_OK;
  const int64_t total = B * H * W;
  const int grid = (int)std::min<int64_t>(cdiv(total, 256), 148 * 64);
  photo_fwd_generic<T><<<grid, 256, 0, st>>>(es, ta, out, B, (int)C, (int)H, (int)W, bs, type, (T)eps);
  count_launch();
  return check_launch("photometric_fwd(generic)");
}

template <typename T>
static int bwd_impl(const T* es, const T* ta, const T* go, T* gi, int64_t B, int64_t C, int64_t H, int64_t W,
                    int bs, int type, float eps, cudaStream_t st) {
  if (int rc = check_common(es, ta, gi, B, C, H, W, bs, type)) return rc;
  if (B * C * H * W == 0) return CTD_OK;
  CTD_REQUIRE(go, "photometric_bwd: null grad_out");
  const int64_t total = B * C * H * W;
  const int grid = (int)std::min<int64_t>(cdiv(total, 256), 148 * 64);
  photo_bwd_generic<T><<<grid, 256, 0, st>>>(es, ta, go, gi, B, (int)C, (int)H, (int)W, bs, type, (T)eps);
  count_launch();
  return check_launch("photometric_bwd(generic)");
}

// census backward (block 9) of nb images; out != nullptr: the fused forward + backward kernel;
// mask != nullptr (fused only): also the masked-mean terms sums2 = (sum(mask * loss), sum(mask)) -- that variant
// needs scratch for the block partials [ticket | pad to 16 B][2 doubles per block] and returns false (nothing
// launched) when it cannot get it.
static bool census_bwd_launch(const float* e, const float* t, const float* g, float* o, float* out, int nb, int64_t C,
                              int64_t H, int64_t W, int type, float eps, int vec, cudaStream_t st,
                              const float* mask = nullptr, float* sums2 = nullptr) {
  dim3 grid((unsigned)cdiv(W, CT_W), (unsigned)cdiv(H, CB_H), nb);
  MsSlot ms = {nullptr, nullptr, nullptr};
  const size_t nblk = (size_t)grid.x * grid.y * grid.z;
  if (mask && !ms_acquire(nblk, st, &ms)) return false;
  unsigned* ticket = ms.ticket;
  double* partials = ms.partials;
  const int iC = (int)C, iH = (int)H, iW = (int)W;
  if (type == 2) {
    if (out) photo_bwd_census9<2, true, CB_NPX><<<grid, 256, 0, st>>>(e, t, g, o, out, iC, iH, iW, eps, vec, mask, partials, ticket, sums2);
    else photo_bwd_census9<2, false, CB_NPX><<<grid, 256, 0, st>>>(e, t, g, o, out, iC, iH, iW, eps, vec, nullptr, nullptr, nullptr, nullptr);
  } else {
    if (out) photo_bwd_census9<3, true, CB_NPX><<<grid, 256, 0, st>>>(e, t, g, o, out, iC, iH, iW, eps, vec, mask, partials, ticket, sums2);
    else photo_bwd_census9<3, false, CB_NPX><<<grid, 256, 0, st>>>(e, t, g, o, out, iC, iH, iW, eps, vec, nullptr, nullptr, nullptr, nullptr);
  }
  ms_release(&ms, st);
  return true;
}

// the whole RectifiedPatternSimilarityLoss step in ONE kernel: warp + census loss + gradient w.r.t. the disparity + masked sums
static bool census_warp_launch(const float* disp, const float* ta, const float* go, float* gd, float* out, int nb, int64_t H, int64_t W,
                               int type, float eps, int vec, cudaStream_t st, const float* mask, float* sums2, const WarpArgs& wa) {
  dim3 grid((unsigned)cdiv(W, CT_W), (unsigned)cdiv(H, CB_H), nb);
  MsSlot ms = {nullptr, nullptr, nullptr};
  const size_t nblk = (size_t)grid.x * grid.y * grid.z;
  if (mask && !ms_acquire(nblk, st, &ms)) return false;
  const int iH = (int)H, iW = (int)W;
  if (type == 2)
    photo_bwd_census9<2, true, CB_NPX, true><<<grid, 256, 0, st>>>(disp, ta, go, gd, out, 1, iH, iW, eps, vec, mask, ms.partials, ms.ticket, sums2, wa);
  else
    photo_bwd_census9<3, true, CB_NPX, true><<<grid, 256, 0, st>>>(disp, ta, go, gd, out, 1, iH, iW, eps, vec, mask, ms.partials, ms.ticket, sums2, wa);
  ms_release(&ms, st);
  return true;
}

static inline int vec_ok(int64_t W, const void* a, const void* b, const void* c, const void* d) {
  auto al = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  return W % 4 == 0 && al(a) && al(b) && al(c) && al(d);
}

}  // namespace ctd

using namespace ctd;

CTD_API int ctd_photometric_fwd_f32(const float* es, const float* ta, float* out, int64_t B, int64_t C,
                                       int64_t H, int64_t W, int bs, int type, float eps, ctd_stream_t stream) {
  cudaStream_t st = as_stream(stream);
  if (!fast9_ok(bs, H, W) || C < 1 || B < 1) return fwd_impl<float>(es, ta, out, B, C, H, W, bs, type, eps, st);
  if (int rc = check_common(es, ta, out, B, C, H, W, bs, type)) return rc;
  if (type <= 1 && box9_tma_fwd(es, ta, out, B, C, H, W, type, st)) return check_launch("photometric_fwd(tma)");
  if (type >= 2 && es && ta && out && census_sym_launch(es, ta, nullptr, out, nullptr, nullptr, nullptr, B, C, H, W, type, eps, st))
    return check_launch("photometric_fwd(census, pair-symmetric)");
  const int vec = vec_ok(W, es, ta, out, out);
  for (int64_t b0 = 0; b0 < B; b0 += 32768) {
    const int nb = (int)std::min<int64_t>(32768, B - b0);
    const float* e = es + b0 * C * H * W;
    const float* t = ta + b0 * C * H * W;
    float* o = out + b0 * H * W;
    if (type <= 1) {
      dim3 grid((unsigned)cdiv(W, BT_W), (unsigned)cdiv(H, BT_H), nb);
      if (type == 0) photo_fwd_box9<0><<<grid, 256, 0, st>>>(e, t, o, (int)C, (int)H, (int)W, vec);
      else photo_fwd_box9<1><<<grid, 256, 0, st>>>(e, t, o, (int)C, (int)H, (int)W, vec);
    } else {
      dim3 grid((unsigned)cdiv(W, CT_W), (unsigned)cdiv(H, CT_H), nb);
      if (type == 2) photo_fwd_census9<2><<<grid, 256, 0, st>>>(e, t, o, (int)C, (int)H, (int)W, eps, vec);
      else photo_fwd_census9<3><<<grid, 256, 0, st>>>(e, t, o, (int)C, (int)H, (int)W, eps, vec);
    }
    count_launch();
  }
  return check_launch("photometric_fwd");
}

CTD_API int ctd_photometric_fwd_f64(const double* es, const double* ta, double* out, int64_t B, int64_t C,
                                       int64_t H, int64_t W, int bs, int type, float eps, ctd_stream_t stream) {
  return fwd_impl<double>(es, ta, out, B, C, H, W, bs, type, eps, as_stream(stream));
}

CTD_API int ctd_photometric_bwd_f32(const float* es, const float* ta, const float* go, float* gi, int64_t B,
                                       int64_t C, int64_t H, int64_t W, int bs, int type, float eps,
                                       ctd_stream_t stream) {
  cudaStream_t st = as_stream(stream);
  if (!fast9_ok(bs, H, W) || C < 1 || B < 1) return bwd_impl<float>(es, ta, go, gi, B, C, H, W, bs, type, eps, st);
  if (int rc = check_common(es, ta, gi, B, C, H, W, bs, type)) return rc;
  CTD_REQUIRE(go, "photometric_bwd: null grad_out");
  if (type <= 1 && box9_tma_bwd(es, ta, go, gi, B, C, H, W, type, st)) return check_launch("photometric_bwd(tma)");
  if (type >= 2 && es && ta && gi && census_sym_launch(es, ta, go, nullptr, gi, nullptr, nullptr, B, C, H, W, type, eps, st))
    return check_launch("photometric_bwd(census, pair-symmetric)");
  const int vec = vec_ok(W, es, ta, go, gi);
  for (int64_t b0 = 0; b0 < B; b0 += 32768) {
    const int nb = (int)std::min<int64_t>(32768, B - b0);
    const float* e = es + b0 * C * H * W;
    const float* t = ta + b0 * C * H * W;
    const float* g = go + b0 * H * W;
    float* o = gi + b0 * C * H * W;
    if (type <= 1) {
      dim3 grid((unsigned)cdiv(W, BT_W), (unsigned)cdiv(H, BT_H), nb);
      if (type == 0) photo_bwd_box9<0><<<grid, 256, 0, st>>>(e, t, g, o, (int)C, (int)H, (int)W, vec);
      else photo_bwd_box9<1><<<grid, 256, 0, st>>>(e, t, g, o, (int)C, (int)H, (int)W, vec);
    } else {
      census_bwd_launch(e, t, g, o, nullptr, nb, C, H, W, type, eps, vec, st);
    }
    count_launch();
  }
  return check_launch("photometric_bwd");
}

// Forward and backward in one call, for callers whose grad_out does not depend on the loss map (the reference's
// RectifiedPatternSimilarityLoss, networks.py:377: grad_out = mask / sum(mask) up to a scalar).  The census
// modes run ONE kernel: the backward gather already forms every dd = 2 (h(des) - h(dta)) of the window, so the
// loss map is one more add per tap instead of a second pass over 162 reciprocal square roots per pixel.
CTD_API int ctd_photometric_fwd_bwd_f32(const float* es, const float* ta, const float* go, float* out, float* gi,
                                           int64_t B, int64_t C, int64_t H, int64_t W, int bs, int type, float eps,
                                           ctd_stream_t stream) {
  cudaStream_t st = as_stream(stream);
  if (type >= 2 && type <= 3 && fast9_ok(bs, H, W) && C >= 1 && B >= 1) {
    if (int rc = check_common(es, ta, gi, B, C, H, W, bs, type)) return rc;
    CTD_REQUIRE(go && out, "photometric_fwd_bwd: null pointer");
    if (es && ta && gi && census_sym_launch(es, ta, go, out, gi, nullptr, nullptr, B, C, H, W, type, eps, st))
      return check_launch("photometric_fwd_bwd(census, pair-symmetric)");
    const int vec = vec_ok(W, es, ta, go, gi) && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
    for (int64_t b0 = 0; b0 < B; b0 += 32768) {
      const int nb = (int)std::min<int64_t>(32768, B - b0);
      census_bwd_launch(es + b0 * C * H * W, ta + b0 * C * H * W, go + b0 * H * W, gi + b0 * C * H * W, out + b0 * H * W, nb,
                        C, H, W, type, eps, vec, st);
      count_launch();
    }
    return check_launch("photometric_fwd_bwd(census, fused)");
  }
  if (type >= 0 && type <= 1 && fast9_ok(bs, H, W) && C >= 1 && B >= 1 && es && ta && go && out && gi &&
      box9_tma_fwd_bwd(es, ta, go, out, gi, B, C, H, W, type, st))
    return check_launch("photometric_fwd_bwd(box, fused)");
  if (int rc = ctd_photometric_fwd_f32(es, ta, out, B, C, H, W, bs, type, eps, stream)) return rc;
  return ctd_photometric_bwd_f32(es, ta, go, gi, B, C, H, W, bs, type, eps, stream);
}

// ctd_photometric_fwd_bwd_f32 plus the caller's masked-mean terms sums2 = (sum(mask * out), sum(mask)) (model/networks.py:377)
// from the same pass: the loss kernels reduce their own tile and the last block to finish adds the partials.
CTD_API int ctd_photometric_fwd_bwd_masked_f32(const float* es, const float* ta, const float* go, const float* mask,
                                                  float* out, float* gi, float* sums2, int64_t B, int64_t C, int64_t H,
                                                  int64_t W, int bs, int type, float eps, ctd_stream_t stream) {
  cudaStream_t st = as_stream(stream);
  if (int rc = check_common(es, ta, gi, B, C, H, W, bs, type)) return rc;
  CTD_REQUIRE(sums2 && (B * H * W == 0 || (go && mask && out)), "photometric_fwd_bwd_masked: null pointer");
  if (B * H * W == 0) {
    CTD_CUDA(cudaMemsetAsync(sums2, 0, 2 * sizeof(float), st));
    return CTD_OK;
  }
  if (fast9_ok(bs, H, W) && C >= 1 && B >= 1 && B <= 32768) {
    if (type <= 1 && box9_tma_fwd_bwd_masked(es, ta, go, mask, out, gi, sums2, B, C, H, W, type, st))
      return check_launch("photometric_fwd_bwd_masked(box, fused)");
    if (type >= 2 && es && ta && gi && census_sym_launch(es, ta, go, out, gi, mask, sums2, B, C, H, W, type, eps, st))
      return check_launch("photometric_fwd_bwd_masked(census, pair-symmetric)");
    if (type >= 2) {
      const int vec = vec_ok(W, es, ta, go, gi) && ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(mask)) & 15) == 0;
      if (census_bwd_launch(es, ta, go, gi, out, (int)B, C, H, W, type, eps, vec, st, mask, sums2)) {
        count_launch();
        return check_launch("photometric_fwd_bwd_masked(census, fused)");
      }
    }
  }
  if (int rc = ctd_photometric_fwd_bwd_f32(es, ta, go, out, gi, B, C, H, W, bs, type, eps, stream)) return rc;
  if (int rc = masked_sums_launch(out, mask, B * H * W, sums2, st)) return rc;
  return check_launch("photometric_fwd_bwd_masked(separate)");
}

CTD_API int ctd_photometric_bwd_f64(const double* es, const double* ta, const double* go, double* gi,
                                       int64_t B, int64_t C, int64_t H, int64_t W, int bs, int type, float eps,
                                       ctd_stream_t stream) {
  return bwd_impl<double>(es, ta, go, gi, B, C, H, W, bs, type, eps, as_stream(stream));
}

// RectifiedPatternSimilarityLoss.tforward (model/networks.py:358-378) and its backward to the disparity as ONE kernel for the
// census modes, block 9: pattern_proj = grid_sample(pattern, grid(disp)) is formed inside the loss kernel's tile loader (the
// pattern is L2-resident), the loss map, the masked-mean terms and d loss / d disp for grad_out (w.r.t. the loss map; the
// caller's is mask / sum(mask) up to a scalar) come out of the same pass.  pattern [Bp,1,Hp,Wp] (Bp = 1 or B), disp / ta /
// grad_out / mask / pattern_proj / out / grad_disp [B,1,H,W]; sums2 = (sum(mask * out), sum(mask)).
CTD_API int ctd_pattern_similarity_f32(const float* pattern, const float* disp, const float* ta, const float* grad_out, const float* mask,
                                       float* pattern_proj, float* out, float* grad_disp, float* sums2, int64_t B, int64_t Bp,
                                       int64_t Hp, int64_t Wp, int64_t H, int64_t W, int type, float eps, ctd_stream_t stream) {
  cudaStream_t st = as_stream(stream);
  CTD_REQUIRE(B >= 0 && H >= 0 && W >= 0, "pattern_similarity: negative size");
  CTD_REQUIRE(type == 2 || type == 3, "pattern_similarity: the fused kernel covers census_mse (2) and census_sad (3), got %d", type);
  CTD_REQUIRE(Bp >= 1 && Hp >= 1 && Wp >= 1 && (Bp == 1 || Bp == B), "pattern_similarity: pattern batch %lld must be 1 or %lld", (long long)Bp, (long long)B);
  CTD_REQUIRE(sums2, "pattern_similarity: null sums2");
  if (B * H * W == 0) {
    CTD_CUDA(cudaMemsetAsync(sums2, 0, 2 * sizeof(float), st));
    return CTD_OK;
  }
  CTD_REQUIRE(pattern && disp && ta && grad_out && mask && pattern_proj && out && grad_disp, "pattern_similarity: null pointer");
  CTD_REQUIRE(H >= 9 && W >= 9 && H * W < ((int64_t)1 << 31) && Hp * Wp < ((int64_t)1 << 31) && B <= 32768, "pattern_similarity: size out of range");
  WarpArgs wa;
  wa.pattern = pattern;
  wa.proj = pattern_proj;
  wa.Bp = (int)Bp;
  wa.Hp = (int)Hp;
  wa.Wp = (int)Wp;
  wa.inv_w = W > 1 ? 1.f / (float)(W - 1) : INFINITY;
  wa.inv_h = H > 1 ? 1.f / (float)(H - 1) : INFINITY;
  const int vec = vec_ok(W, disp, ta, grad_out, grad_disp) && ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(mask)) & 15) == 0;
  if (!census_warp_launch(disp, ta, grad_out, grad_disp, out, (int)B, H, W, type, eps, vec, st, mask, sums2, wa))
    return fail(CTD_ERR_NOMEM, "pattern_similarity: no reduction workspace");
  count_launch();
  return check_launch("pattern_similarity(fused)");
}
