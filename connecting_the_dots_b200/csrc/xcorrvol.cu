// XCorrVol (zero-mean normalised cross-correlation cost volume) for sm_100a.
//
// Reference semantics: torchext/ext/ext.h:120-191 (XCorrVolFunctor), bound at ext_cuda.cpp:73-86.
// out[d,h,w] = sum_c dot / (sqrt(sigma0 * sigma1) + 1e-8) over a bs x bs window of in0 at (h,w) and
// of in1 at (h, w-d); rows replicate-clamped, in0 columns clamped, in1 columns clamped AFTER the
// disparity shift.  The reference has no batch dimension; here B images are one launch.
#include <algorithm>
#include <type_traits>

#include "ctd_common.cuh"
#include "ctd_tma.cuh"

namespace ctd {

extern int g_force_generic;
extern int g_xcorr_direct;
extern int g_xcorr_nofix;
extern int g_xcorr_hitcap;

// generic: any C, any block size, float or double; one output, reference operation order (built with -fmad=false), so it
// reproduces the reference's two-pass centred statistics exactly.  Shared by the volume and the disparity kernels.
template <typename T>
__device__ __forceinline__ T xcorr_generic_one(const T* __restrict__ in0, const T* __restrict__ in1, int64_t b, int C, int H,
                                               int W, int h, int w, int d, int bs) {
  const int half = bs / 2;
  const T bs2 = (T)(bs * bs);
  T val = 0;
  for (int c = 0; c < C; ++c) {
    const T* p0 = in0 + (b * C + c) * H * W;
    const T* p1 = in1 + (b * C + c) * H * W;
    T mu0 = 0, mu1 = 0;
    for (int bh = 0; bh < bs; ++bh) {
      const int64_t row = (int64_t)clampi(h + bh - half, 0, H - 1) * W;
      for (int bw = 0; bw < bs; ++bw) {
        const int w0 = w + bw - half;
        mu0 += __ldg(p0 + row + clampi(w0, 0, W - 1)) / bs2;
        mu1 += __ldg(p1 + row + clampi(w0 - d, 0, W - 1)) / bs2;
      }
    }
    T s0 = 0, s1 = 0, dot = 0;
    for (int bh = 0; bh < bs; ++bh) {
      const int64_t row = (int64_t)clampi(h + bh - half, 0, H - 1) * W;
      for (int bw = 0; bw < bs; ++bw) {
        const int w0 = w + bw - half;
        const T v0 = __ldg(p0 + row + clampi(w0, 0, W - 1)) - mu0;
        const T v1 = __ldg(p1 + row + clampi(w0 - d, 0, W - 1)) - mu1;
        dot += v0 * v1;
        s0 += v0 * v0;
        s1 += v1 * v1;
      }
    }
    const T norm = (T)((double)sqrt(s0 * s1) + 1e-8);
    val += dot / norm;
  }
  return val;
}

// one thread per output
template <typename T>
__global__ void __launch_bounds__(256)
xcorrvol_generic(const T* __restrict__ in0, const T* __restrict__ in1, T* __restrict__ out, int64_t B, int C,
                 int H, int W, int D, int bs) {
  const int64_t total = B * D * H * W;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int w = idx % W, h = (idx / W) % H, d = (idx / ((int64_t)W * H)) % D;
    const int64_t b = idx / ((int64_t)W * H * D);
    out[idx] = xcorr_generic_one<T>(in0, in1, b, C, H, W, h, w, d, bs);
  }
}

// ------------------------------------------------------------------------------------------
// Winner-take-all disparity (ctd_xcorr_disparity_*): d* = the first d with V[d] = max_d V[d], score = V[d*].
// Partial maxima merge through a 64-bit integer key: the order-preserving bits of the score above 0xFFFFFFFF - d, so
// the unsigned maximum is the largest score and, among equal scores, the smallest d.  -0.0 is keyed as +0.0 (they
// compare equal).  Key 0 is below every real key.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long wta_key(float v, int d) {
  unsigned u = __float_as_uint(v);
  if (u == 0x80000000u) u = 0u;
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((unsigned long long)u << 32) | (0xFFFFFFFFu - (unsigned)d);
}
__device__ __forceinline__ float wta_score(unsigned long long key) {
  const unsigned u = (unsigned)(key >> 32);
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u);
}
__device__ __forceinline__ int wta_disp(unsigned long long key, int D) {  // clamped: a key of 0 (no candidate) is never read out of range
  return (int)min(0xFFFFFFFFu - (unsigned)key, (unsigned)(D - 1));
}
// generic disparity: one thread per pixel sweeps d with xcorr_generic_one through a WtaRun, so d* and the score are the
// exact argmax and maximum of xcorrvol_generic's volume
template <typename T>
__global__ void __launch_bounds__(256)
xcorr_disparity_generic(const T* __restrict__ in0, const T* __restrict__ in1, T* __restrict__ disp, T* __restrict__ score,
                        int64_t B, int C, int H, int W, int D, int bs, int subpixel) {
  const int64_t total = B * H * W;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int w = idx % W, h = (idx / W) % H;
    const int64_t b = idx / ((int64_t)W * H);
    WtaRun<T> run;
    run.init();
    for (int d = 0; d < D; ++d) run.step(xcorr_generic_one<T>(in0, in1, b, C, H, W, h, w, d, bs), d);
    // disp is never null here (xcorr_disparity_impl requires it); without the hint the fp32 build reloads two more
    // spilled words per pixel
    __builtin_assume(disp != nullptr);
    wta_store<T>(disp, score, idx, run.bd, run.best, run.cm, run.cp, D, subpixel);
  }
}

// ------------------------------------------------------------------------------------------
// direct kernel: C = 1, odd block size BS <= 9, fp32.  Same centred two-pass arithmetic as the
// reference (so flat / low-texture windows, where normalised correlation is ill-conditioned, come out
// like ext_cpu's), but tiled: a CTA owns one image row, XD_TW pixels and XD_DC disparities.
//   * rows h-R..h+R of in0 (XD_TW + 2R columns) and of in1 (XD_TW + 2R + XD_DC - 1 columns, clamped
//     AFTER the disparity shift) are staged in shared memory once;
//   * mean and sigma of every in1 window the CTA touches depend only on x' = w - d: computed once per
//     x' in the prologue instead of once per (w, d);
//   * a thread owns one pixel, keeps its centred in0 window (BS*BS values) in registers, and sweeps
//     the disparities four at a time so each shared-memory row segment feeds 4 * BS taps.
// ------------------------------------------------------------------------------------------
constexpr int XD_TW = 128;  // pixels (threads) per CTA
constexpr int XD_DC = 32;   // disparities per CTA

template <int BS>
__global__ void __launch_bounds__(XD_TW)
xcorrvol_direct(const float* __restrict__ in0, const float* __restrict__ in1, float* __restrict__ out, int H, int W,
                int D, int nchunks) {
  constexpr int R = BS / 2, N = BS * BS;
  constexpr int AW = XD_TW + 2 * R;               // in0 tile width
  constexpr int BW = XD_TW + 2 * R + XD_DC - 1;   // in1 tile width
  constexpr int NP = XD_TW + XD_DC - 1;           // in1 window positions x' touched by this CTA
  __shared__ float As[BS][AW];
  __shared__ float Bs[BS][BW];
  __shared__ float Mu1[NP], S1[NP];
  const int tid = threadIdx.x;
  const int x0 = blockIdx.x * XD_TW, h = blockIdx.y;
  const int b = blockIdx.z / nchunks, d0 = (blockIdx.z % nchunks) * XD_DC;
  const int64_t plane = (int64_t)H * W;
  const float* a = in0 + b * plane;
  const float* bp = in1 + b * plane;
  // in1 tile column j <-> unclamped image column x0 - R - (d0 + XD_DC - 1) + j
  const int bcol0 = x0 - R - (d0 + XD_DC - 1);
  for (int i = tid; i < BS * AW; i += XD_TW) {
    const int r = i / AW, j = i % AW;
    As[r][j] = __ldg(a + (int64_t)clampi(h - R + r, 0, H - 1) * W + clampi(x0 - R + j, 0, W - 1));
  }
  for (int i = tid; i < BS * BW; i += XD_TW) {
    const int r = i / BW, j = i % BW;
    Bs[r][j] = __ldg(bp + (int64_t)clampi(h - R + r, 0, H - 1) * W + clampi(bcol0 + j, 0, W - 1));
  }
  __syncthreads();
  // statistics of the in1 windows: position p <-> window whose left tap is tile column p
  for (int p = tid; p < NP; p += XD_TW) {
    float mu = 0.f;
#pragma unroll
    for (int r = 0; r < BS; ++r)
#pragma unroll
      for (int c = 0; c < BS; ++c) mu += Bs[r][p + c] * (1.0f / float(N));
    float sg = 0.f;
#pragma unroll
    for (int r = 0; r < BS; ++r)
#pragma unroll
      for (int c = 0; c < BS; ++c) {
        const float v = Bs[r][p + c] - mu;
        sg += v * v;
      }
    Mu1[p] = mu;
    S1[p] = sg;
  }
  // this thread's centred in0 window
  float ac[N];
  float mu0 = 0.f;
#pragma unroll
  for (int r = 0; r < BS; ++r)
#pragma unroll
    for (int c = 0; c < BS; ++c) {
      ac[r * BS + c] = As[r][tid + c];
      mu0 += ac[r * BS + c] * (1.0f / float(N));
    }
  float s0 = 0.f;
#pragma unroll
  for (int k = 0; k < N; ++k) {
    ac[k] -= mu0;
    s0 += ac[k] * ac[k];
  }
  __syncthreads();
  const int w = x0 + tid;
  // disparity d = d0 + q: window left tap at tile column tid + (XD_DC - 1) - q
  for (int q = 0; q < XD_DC; q += 4) {
    const int base = tid + XD_DC - 4 - q;  // left tap of the window of disparity d0 + q + 3
    float dot[4] = {0.f, 0.f, 0.f, 0.f};
    float mu1[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) mu1[j] = Mu1[base + 3 - j];
#pragma unroll
    for (int r = 0; r < BS; ++r) {
      float v[BS + 3];
#pragma unroll
      for (int c = 0; c < BS + 3; ++c) v[c] = Bs[r][base + c];
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int c = 0; c < BS; ++c) dot[j] += ac[r * BS + c] * (v[3 - j + c] - mu1[j]);
    }
    if (w < W) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int d = d0 + q + j;
        if (d < D) {
          const float norm = (float)((double)sqrtf(s0 * S1[base + 3 - j]) + 1e-8);
          out[((int64_t)(b * D + d) * H + h) * W + w] = dot[j] / norm;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// separable kernel: C = 1, odd block size BS <= 9, fp32 -- the fast path.
//
//   dot(d,h,w) = sum_win (a - mu0)(b - mu1) = sum_win a*b  -  N * mu0(h,w) * mu1(h,w-d)
//
// so the only per-disparity work is a BS x BS box sum of the product plane a(h',x) * b(h',x-d): one
// multiply and ~7 adds per output instead of 2*BS*BS taps.  mu and sigma of every window depend on one
// image only and are computed once per pixel by xcorr_stats_kernel (fp64 box sums), for in1 over the
// replicate-padded column range u = w - d in [-(D-1), W-1].
//
// Main kernel: a CTA owns 128 columns x XH rows x 16 disparities.  Warp g owns four disparities, lane l
// four adjacent columns.  A thread walks down the tile rows: per row it reads 12 in0 and 16 in1 values
// from the staged tiles (seven 128-bit shared loads) and forms the 4 x 12 products and their horizontal
// BS-sums in registers.  The vertical BS-sum never subtracts (no sliding residue): rows are grouped in
// blocks of BS; F is the running sum of the current block, and when a block completes its rows are
// turned in place into suffix sums (rows j..BS-1), all in registers.  The window ending at row j of a
// block is then suffix(j+1) of the previous block + F -- every output is an exact subset sum of its own
// window's products.  Outputs leave as 128-bit stores of four adjacent columns, 512 B per warp and
// disparity.
//
// Conditioning: the expanded form cancels when a window's spread is small against its mean.
// xcorr_stats_kernel grades every window with L = floor(-4 log2(var / sum v^2)) (a byte per window, read
// only by the fix-up pass).  The fast path's error is about 1.5e-7 * sqrt(S2_0 S2_1) / (sd0 sd1) =
// 1.5e-7 * 2^((L0+L1)/8); outputs with L0 + L1 >= XS_LSUM (sd0 sd1 < 2^-5 sqrt(S2_0 S2_1), a few per
// thousand on LCN'd images) are recomputed by xcorr_fixup_kernel: it walks the listed windows
// (L >= XS_LLIST), compacts the affected outputs and evaluates them in the centred form, one fp32 pass with the
// window means of the statistics pass (xcorr_centred_one) -- or, for flat windows
// (var < 1e-6 sum v^2), where the reference's result is its own rounding noise, with the reference's
// centred two-pass fp32 arithmetic (ext.h:133-190).
// ------------------------------------------------------------------------------------------
constexpr int XS_W = 128;             // output columns per CTA (32 lanes x 4)
constexpr int XS_DT = 16;             // disparities per CTA
#ifndef CTD_XS_TD
#define CTD_XS_TD 4
#endif
constexpr int XS_TD = CTD_XS_TD;      // disparities per thread (4: 4 warps per CTA, 2: 8 warps per CTA)
constexpr int XS_AW = XS_W + 8;       // in0 tile: image columns x0-4 .. x0+131
constexpr int XS_BW = XS_W + 8 + 16;  // in1 tile: image columns x0-20-d0 .. x0+131-d0 (clamped)
constexpr int ST_W = 128, ST_H = 16;  // statistics tile
constexpr int XS_LSUM = 40;           // L0 + L1 >= 40 <=> (sd0 sd1)^2 <= 2^-10 S2_0 S2_1 (fast-path error ~5e-6): recompute centred
constexpr int XS_LLIST = 20;          // max(L0, L1) >= 20 whenever L0 + L1 >= 40
constexpr int XS_LEXACT = 76;         // var < 2^-19 sum v^2 (~2e-6): flat window, reference arithmetic
template <int TD>
struct XsNst {  // statistics rows in flight per warp (more warps per CTA -> shallower rings, same shared memory)
  static constexpr int value = 3;
};
template <int NST>
struct alignas(16) XsStatRing {
  float2 w[NST][XS_W];
  float2 u[NST][XS_W + 8];
  uint64_t full[NST];
};
template <int BS>
struct XsCfg {  // tile rows = a whole number of BS-row blocks
  static constexpr int R = BS / 2;
  static constexpr int NBLK = BS == 9 ? 5 : BS == 7 ? 6 : BS == 5 ? 8 : 13;
  static constexpr int TH = BS * NBLK;    // staged rows
  static constexpr int XH = TH - 2 * R;   // output rows per CTA (37, 36, 36, 37)
};

// reference arithmetic for one output (ext.h:133-190 with C = 1)
template <int BS>
__device__ __forceinline__ float xcorr_exact_one(const float* __restrict__ p0, const float* __restrict__ p1, int H, int W,
                                                 int h, int w, int d) {
  constexpr int R = BS / 2;
  const float bs2 = float(BS * BS);
  float mu0 = 0.f, mu1 = 0.f;
  for (int bh = 0; bh < BS; ++bh) {
    const int64_t row = (int64_t)clampi(h + bh - R, 0, H - 1) * W;
#pragma unroll
    for (int bw = 0; bw < BS; ++bw) {
      const int w0 = w + bw - R;
      mu0 += __ldg(p0 + row + clampi(w0, 0, W - 1)) / bs2;
      mu1 += __ldg(p1 + row + clampi(w0 - d, 0, W - 1)) / bs2;
    }
  }
  float s0 = 0.f, s1 = 0.f, dot = 0.f;
  for (int bh = 0; bh < BS; ++bh) {
    const int64_t row = (int64_t)clampi(h + bh - R, 0, H - 1) * W;
#pragma unroll
    for (int bw = 0; bw < BS; ++bw) {
      const int w0 = w + bw - R;
      const float v0 = __ldg(p0 + row + clampi(w0, 0, W - 1)) - mu0;
      const float v1 = __ldg(p1 + row + clampi(w0 - d, 0, W - 1)) - mu1;
      dot += v0 * v1;
      s0 += v0 * v0;
      s1 += v1 * v1;
    }
  }
  return dot / (float)((double)sqrtf(s0 * s1) + 1e-8);
}

// One output from the centred form with the window means and deviations the statistics pass already holds
// (fp64 box sums, rounded once): dot = sum (a - mu0)(b - mu1) in one fp32 pass.  a - mu is exact where it matters
// (Sterbenz), the rounding of the stored means enters only as N d0 d1, and the accumulation error is bounded by
// ~81 eps sd0 sd1 -- about 1e-6 of the normaliser however large the window means are.  Flat windows
// (grade >= XS_LEXACT), where the reference's result is its own rounding noise, go to xcorr_exact_one.
template <int BS>
__device__ __forceinline__ float xcorr_centred_one(const float* __restrict__ p0, const float* __restrict__ p1, int H, int W,
                                                   int h, int w, int d, float mu0, float mu1, float sd0, float sd1) {
  constexpr int R = BS / 2;
  unsigned ca[BS], cb[BS];  // byte offsets of the clamped columns of the two windows, once per output
#pragma unroll
  for (int bw = 0; bw < BS; ++bw) {
    ca[bw] = 4u * (unsigned)clampi(w + bw - R, 0, W - 1);
    cb[bw] = 4u * (unsigned)clampi(w + bw - R - d, 0, W - 1);
  }
  const char* q0 = reinterpret_cast<const char*>(p0);
  const char* q1 = reinterpret_cast<const char*>(p1);
  float dot[3] = {0.f, 0.f, 0.f};  // three rows in flight
#pragma unroll
  for (int bh = 0; bh < BS; ++bh) {
    const int64_t row = (int64_t)clampi(h + bh - R, 0, H - 1) * W * 4;
    const char* ra = q0 + row;
    const char* rb = q1 + row;
#pragma unroll
    for (int bw = 0; bw < BS; ++bw)
      dot[bh % 3] = fmaf(__ldg(reinterpret_cast<const float*>(ra + ca[bw])) - mu0,
                         __ldg(reinterpret_cast<const float*>(rb + cb[bw])) - mu1, dot[bh % 3]);
  }
  return ((dot[0] + dot[1]) + dot[2]) / (sd0 * sd1 + 1e-8f);
}

// xcorr_centred_one at disparities d - 1, d, d + 1 in one pass (c[k] at d - 1 + k, the same arithmetic, so the same
// values): the three in1 windows share BS - 1 of their BS + 1 columns, and the in0 window is common.
template <int BS>
__device__ __forceinline__ void xcorr_centred_three(const float* __restrict__ p0, const float* __restrict__ p1, int H, int W,
                                                    int h, int w, int d, float mu0, float sd0, const float (&mu1)[3],
                                                    const float (&sd1)[3], float (&c)[3]) {
  constexpr int R = BS / 2;
  unsigned ca[BS], cb[BS + 2];  // byte offsets of the clamped columns; tap bw of disparity d - 1 + k is in1 column cb[bw + 2 - k]
#pragma unroll
  for (int bw = 0; bw < BS; ++bw) ca[bw] = 4u * (unsigned)clampi(w + bw - R, 0, W - 1);
#pragma unroll
  for (int j = 0; j < BS + 2; ++j) cb[j] = 4u * (unsigned)clampi(w + j - R - d - 1, 0, W - 1);
  const char* q0 = reinterpret_cast<const char*>(p0);
  const char* q1 = reinterpret_cast<const char*>(p1);
  // rows accumulate into dot[k][bh % 3] as in xcorr_centred_one; the loop stays rolled (registers), so the row's slot is
  // always dot[k][0] and the slots rotate after each row
  float dot[3][3] = {};
#pragma unroll 1
  for (int bh = 0; bh < BS; ++bh) {
    const int64_t row = (int64_t)clampi(h + bh - R, 0, H - 1) * W * 4;
    float bv[BS + 2];
#pragma unroll
    for (int j = 0; j < BS + 2; ++j) bv[j] = __ldg(reinterpret_cast<const float*>(q1 + row + cb[j]));
#pragma unroll
    for (int bw = 0; bw < BS; ++bw) {
      const float av = __ldg(reinterpret_cast<const float*>(q0 + row + ca[bw])) - mu0;
#pragma unroll
      for (int k = 0; k < 3; ++k) dot[k][0] = fmaf(av, bv[bw + 2 - k] - mu1[k], dot[k][0]);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float t = dot[k][0];
      dot[k][0] = dot[k][1];
      dot[k][1] = dot[k][2];
      dot[k][2] = t;
    }
  }
  // slot j (rows bh = j mod 3) now sits at position (j - BS) mod 3
  constexpr int P0 = (0 + 3 - BS % 3) % 3, P1 = (1 + 3 - BS % 3) % 3, P2 = (2 + 3 - BS % 3) % 3;
#pragma unroll
  for (int k = 0; k < 3; ++k) c[k] = ((dot[k][P0] + dot[k][P1]) + dot[k][P2]) / (sd0 * sd1[k] + 1e-8f);
}

// Window statistics of one image over positions i = u + uoff, u = column of the window centre (may be
// negative: replicate padding).  st_out = {scale * mean, sqrt(sum (v - mean)^2)} interleaved, grade_out = L.
// Windows with L >= XS_LLIST are appended to `list` as (side | position).
template <int BS>
__global__ void __launch_bounds__(256)
xcorr_stats_kernel(const float* __restrict__ img, float2* __restrict__ st_out, uint8_t* __restrict__ grade_out, int H, int W, int ws, int uoff, float scale, unsigned side,
                   unsigned* __restrict__ list, unsigned* __restrict__ count) {
  constexpr int R = BS / 2, TH = ST_H + 2 * R, TW = ST_W + 2 * R;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  double(*H1)[ST_W] = reinterpret_cast<double(*)[ST_W]>(smem_raw);
  double(*H2)[ST_W] = H1 + TH;
  float(*T)[TW] = reinterpret_cast<float(*)[TW]>(H2 + TH);
  const int tid = threadIdx.x;
  const int i0 = blockIdx.x * ST_W, y0 = blockIdx.y * ST_H;
  const float* src = img + (int64_t)blockIdx.z * H * W;
  {  // every load of the tile in flight before the first shared-memory store (one round trip, not thirteen)
    constexpr int NLD = (TH * TW + 255) / 256;
    float v[NLD];
#pragma unroll
    for (int k = 0; k < NLD; ++k) {
      const int i = tid + 256 * k, r = i / TW, j = i % TW;
      if (i < TH * TW) v[k] = __ldg(src + (int64_t)clampi(y0 - R + r, 0, H - 1) * W + clampi(i0 - uoff - R + j, 0, W - 1));
    }
#pragma unroll
    for (int k = 0; k < NLD; ++k) {
      const int i = tid + 256 * k;
      if (i < TH * TW) T[i / TW][i % TW] = v[k];
    }
  }
  __syncthreads();
  for (int it = tid; it < TH * (ST_W / 4); it += 256) {
    const int r = it / (ST_W / 4), c = 4 * (it % (ST_W / 4));
    double v[BS + 3];
#pragma unroll
    for (int j = 0; j < BS + 3; ++j) v[j] = (double)T[r][c + j];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      double s1 = 0.0, s2 = 0.0;
#pragma unroll
      for (int j = 0; j < BS; ++j) {
        s1 += v[k + j];
        s2 = fma(v[k + j], v[k + j], s2);
      }
      H1[r][c + k] = s1;
      H2[r][c + k] = s2;
    }
  }
  __syncthreads();
  // thread (c, hh) produces output rows hh .. hh+7 of column c (exact subset sums, fp64)
  const int c = tid % ST_W, hh = (tid / ST_W) * (ST_H / 2);
  const double inv_n = 1.0 / double(BS * BS);
#pragma unroll 2
  for (int o = 0; o < ST_H / 2; ++o) {
    const int y = y0 + hh + o;
    if (y >= H || i0 + c >= ws) continue;
    double s1 = 0.0, s2 = 0.0;
#pragma unroll
    for (int j = 0; j < BS; ++j) {
      s1 += H1[hh + o + j][c];
      s2 += H2[hh + o + j][c];
    }
    const float var = (float)fmax(s2 - s1 * s1 * inv_n, 0.0), e2 = (float)s2;
    const float sd = sqrtf(var);
    // grade: L = floor(-4 log2(var / S2)); an all-zero window is exact (every product is 0): L = 0
    unsigned L = 0;
    if (e2 > 0.f) L = var > 0.f ? (unsigned)min(255, max(0, (int)floorf(-4.f * log2f(var / e2)))) : 255u;
    const int64_t off = ((int64_t)blockIdx.z * H + y) * ws + i0 + c;
    st_out[off] = make_float2((float)(s1 * inv_n) * scale, sd);
    grade_out[off] = (uint8_t)L;
    if (L >= (unsigned)XS_LLIST) list[atomicAdd(count, 1u)] = side | (unsigned)off;
  }
}

// o[k] = sum_{j=4-R+k}^{4+R+k} p[j], k = 0..3: the taps common to the four windows are summed once,
// every o[k] is an exact subset sum of its own window (nothing slides, so no residue from other taps)
template <int BS>
__device__ __forceinline__ void xs_hsum(const float* p, float* o) {
  constexpr int R = BS / 2;
  if (BS == 9) {
    const float mid = ((p[3] + p[4]) + (p[5] + p[6])) + (p[7] + p[8]);
    const float l12 = p[1] + p[2], r910 = p[9] + p[10];
    o[0] = mid + (p[0] + l12);
    o[1] = mid + (l12 + p[9]);
    o[2] = mid + (p[2] + r910);
    o[3] = mid + (r910 + p[11]);
  } else if (BS == 7) {
    const float mid = (p[4] + p[5]) + (p[6] + p[7]);
    o[0] = mid + ((p[1] + p[2]) + p[3]);
    o[1] = mid + ((p[2] + p[3]) + p[8]);
    o[2] = mid + (p[3] + (p[8] + p[9]));
    o[3] = mid + ((p[8] + p[9]) + p[10]);
  } else if (BS == 5) {
    const float mid = p[5] + p[6];
    o[0] = mid + ((p[2] + p[3]) + p[4]);
    o[1] = mid + ((p[3] + p[4]) + p[7]);
    o[2] = mid + (p[4] + (p[7] + p[8]));
    o[3] = mid + ((p[7] + p[8]) + p[9]);
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float s = p[4 - R + k];
#pragma unroll
      for (int j = 5 - R + k; j <= 4 + R + k; ++j) s += p[j];
      o[k] = s;
    }
  }
}

// The same four window sums straight from the factors (block 9): products and additions fused into FMA chains --
// 19 instructions instead of 12 multiplies + 15 additions, every o[k] still a sum of exactly its own window's
// products (nothing is subtracted), each product rounded at most once less than before.  b points at the factor of a[0].
__device__ __forceinline__ void xs_hsum9_fma(const float* a, const float* b, float* o) {
  const float m0 = fmaf(a[5], b[5], fmaf(a[4], b[4], a[3] * b[3]));
  const float m1 = fmaf(a[8], b[8], fmaf(a[7], b[7], a[6] * b[6]));
  const float mid = m0 + m1;
  const float l12 = fmaf(a[1], b[1], a[2] * b[2]), r910 = fmaf(a[9], b[9], a[10] * b[10]);
  o[0] = mid + fmaf(a[0], b[0], l12);
  o[1] = mid + fmaf(a[9], b[9], l12);
  o[2] = mid + fmaf(a[2], b[2], r910);
  o[3] = mid + fmaf(a[11], b[11], r910);
}

#ifndef CTD_XS_PACKED_VERTICAL
#define CTD_XS_PACKED_VERTICAL 1
#endif
// TD = disparities per thread.  TD = 4: 128 threads, 246 registers (suffix sums of 16 outputs), 8 warps/SM.
// TD = 2: 256 threads, half the suffix registers, 16 warps/SM -- the tile and the arithmetic per output are the
// same, the resident warps double (the kernel is latency-bound), the in1 row is read as seven 64-bit loads.
//
// Out = float: the volume.  Out = unsigned long long: the winner-take-all variant -- the same outputs, but instead of
// being stored each is a candidate for its pixel's maximum: a thread keeps the best of its TD disparities per column and
// merges it into the key plane `out` [B,H,W] with a 64-bit integer atomicMax (wta_key) per column and output row.  (A
// key tile in shared memory that merged the CTA's warps first cost 38 KB of shared memory per CTA and compiled to
// compare-and-swap loops: measured slower, 751 against 674 us at block 9, batch 8.)  Outputs the fix-up recomputes
// (L0 + L1 >= XS_LSUM, grades g0 / g1 of the statistics pass) take no part: their fast-path value can be far off.
template <int BS, int TD, bool VEC, typename Out>
__global__ void __launch_bounds__(512 / TD, 2)
xcorr_sep_kernel(const float* __restrict__ in0, const float* __restrict__ in1, Out* __restrict__ out,
                 const float2* __restrict__ st0, const float2* __restrict__ st1, const uint8_t* __restrict__ g0,
                 const uint8_t* __restrict__ g1, int H, int W, int D, int ws0, int ws1, int uoff, int ndchunks) {
  constexpr bool WTA = std::is_same<Out, unsigned long long>::value;
  constexpr int R = BS / 2, TH = XsCfg<BS>::TH, XH = XsCfg<BS>::XH, NBLK = XsCfg<BS>::NBLK;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float(*At)[XS_AW] = reinterpret_cast<float(*)[XS_AW]>(smem_raw);
  float(*Bt)[XS_BW] = reinterpret_cast<float(*)[XS_BW]>(smem_raw + sizeof(float) * TH * XS_AW);
  constexpr int NT = 512 / TD, NST = XsNst<TD>::value;
  typedef XsStatRing<NST> Ring;
  Ring* rings = reinterpret_cast<Ring*>(smem_raw + sizeof(float) * TH * (XS_AW + XS_BW));
  const int tid = threadIdx.x, lane = tid & 31;
  const int g = __shfl_sync(0xffffffffu, tid >> 5, 0);  // warp index, known to be warp-uniform (uniform datapath)
  const int x0 = blockIdx.x * XS_W, y0 = blockIdx.y * XH;
  const int b = blockIdx.z / ndchunks, d0 = (blockIdx.z % ndchunks) * XS_DT;
  const int64_t plane = (int64_t)H * W;
  const float* p0 = in0 + b * plane;
  const float* p1 = in1 + b * plane;
  // stage the tiles (replicate clamp; 128-bit loads where the four columns are inside the image), four
  // independent loads in flight per thread
  auto fetch4 = [&](const float* img, int r, int gx) -> float4 {
    const float* row = img + (int64_t)clampi(y0 - R + r, 0, H - 1) * W;
    if (VEC && gx >= 0 && gx + 3 < W) return ldg4(row + gx);
    return make_float4(__ldg(row + clampi(gx, 0, W - 1)), __ldg(row + clampi(gx + 1, 0, W - 1)),
                       __ldg(row + clampi(gx + 2, 0, W - 1)), __ldg(row + clampi(gx + 3, 0, W - 1)));
  };
  constexpr int NA = TH * (XS_AW / 4), NB = TH * (XS_BW / 4);
  for (int i0 = tid; i0 < NA; i0 += 4 * NT) {
    float4 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = i0 + k * NT;
      if (i < NA) v[k] = fetch4(p0, i / (XS_AW / 4), x0 - 4 + 4 * (i % (XS_AW / 4)));
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = i0 + k * NT;
      if (i < NA) *reinterpret_cast<float4*>(&At[i / (XS_AW / 4)][4 * (i % (XS_AW / 4))]) = v[k];
    }
  }
  for (int i0 = tid; i0 < NB; i0 += 4 * NT) {
    float4 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = i0 + k * NT;
      if (i < NB) v[k] = fetch4(p1, i / (XS_BW / 4), x0 - 20 - d0 + 4 * (i % (XS_BW / 4)));
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int i = i0 + k * NT;
      if (i < NB) *reinterpret_cast<float4*>(&Bt[i / (XS_BW / 4)][4 * (i % (XS_BW / 4))]) = v[k];
    }
  }
  __syncthreads();
  const int x = x0 + 4 * lane;
  const int dbase = d0 + TD * g;  // this warp's first disparity
  if (dbase >= D) return;  // warp-uniform: nothing to write, no CTA barrier follows
  // suf[j-1][dl][k], j = 1..BS-1: sum of rows j..BS-1 of the previous block; rows < j of the current block
  // overwrite it with their own horizontal sums as they are produced
  float suf[BS - 1][TD][4], F[TD][4];
#pragma unroll
  for (int dl = 0; dl < TD; ++dl)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      F[dl][k] = 0.f;
#pragma unroll
      for (int j = 0; j < BS - 1; ++j) suf[j][dl][k] = 0.f;
    }
  // tile column of image column (x - 4 - d) is 4*lane + 16 - (d - d0).  TD = 4: the 16 values from 4*lane + 12 - 4g
  // (128-bit aligned) cover the warp's four disparities, tap t of disparity dl is bv[4 - dl + t].  TD = 2: the 14 values
  // from 4*lane + 14 - 2g (64-bit aligned) cover two, tap t of disparity dl is bv[2 - dl + t].
  constexpr int BOFF = TD == 4 ? 4 : 2;
  const float* arow = &At[0][4 * lane];
  const float* brow = &Bt[0][4 * lane + 16 - BOFF - TD * g];
  // store pointer of the row being emitted (tile row r -> output row y0 + r - 2R), advanced by W per row: no
  // 64-bit index arithmetic inside the loop
  // (WTA: the key plane [B,H,W] -- this lane's four keys of the row)
  Out* orow = out + ((WTA ? (int64_t)b * H : ((int64_t)b * D + dbase) * H) + (y0 - 2 * R)) * W + x;
  const int64_t dstride = (int64_t)H * W;
  const int ndl = min(TD, D - dbase);  // disparities of this warp that exist
  const bool xin = VEC ? x < W : true;
  // WTA: grades of the lane's four w positions (gr[0], a byte each) and of its eight u positions (gr[1], gr[2]) in an
  // output row; a lane whose columns lie outside the image keeps 0xff grades (no candidates)
  const uint8_t* g0row = WTA ? g0 + ((int64_t)b * H + y0) * ws0 + x : nullptr;
  const uint8_t* g1row = WTA ? g1 + ((int64_t)b * H + y0) * ws1 + (x - dbase - 4 + uoff) : nullptr;
  unsigned grn[3] = {~0u, ~0u, ~0u};  // WTA: grades of the next output row, loaded one row ahead (the L2 round trip
                                     // overlaps a row of arithmetic)
  auto load_grades = [&](int e, unsigned (&gr)[3]) {
    const uint8_t* p0 = g0row + (int64_t)e * ws0;
    const uint8_t* p1 = g1row + (int64_t)e * ws1;
    gr[0] = __ldg(reinterpret_cast<const unsigned*>(p0));
    if (TD == 4) {  // 4-byte aligned: x, dbase, uoff and the row strides are multiples of 4
      gr[1] = __ldg(reinterpret_cast<const unsigned*>(p1));
      gr[2] = __ldg(reinterpret_cast<const unsigned*>(p1 + 4));
    } else {
      gr[1] = gr[2] = 0u;
#pragma unroll
      for (int j = 0; j < 8; ++j) gr[1 + j / 4] |= (unsigned)__ldg(p1 + j) << (8 * (j % 4));
    }
  };
  // Window statistics of the output rows stream through a per-warp shared-memory ring: one lane fetches a
  // row's w-side {N*mu0, sd0} (128 positions) and u-side {mu1, sd1} (136 positions u = x0-dbase-4 ..) with two
  // cp.async.bulk copies, NST rows ahead, completion on an mbarrier -- no registers are held across the
  // arithmetic and the L2 round trip is off the critical path.  Rows are fetched in order, so the source
  // pointers just advance; with NST | BS the stage of a row is a compile-time constant of the unrolled loop.
  Ring& ring = rings[g];
  const uint32_t ring_w = smem_u32(&ring.w[0][0]), ring_u = smem_u32(&ring.u[0][0]), ring_bar = smem_u32(&ring.full[0]);
  const char* wnext = reinterpret_cast<const char*>(st0 + ((int64_t)b * H + y0) * ws0 + x0);
  const char* unext = reinterpret_cast<const char*>(st1 + ((int64_t)b * H + y0) * ws1 + (x0 - dbase - 4 + uoff));
  const int64_t wstep = (int64_t)ws0 * 8, ustep = (int64_t)ws1 * 8;
  const uint32_t wbytes = (uint32_t)min(XS_W, ws0 - x0) * 8u;
  const uint32_t ubytes = (uint32_t)min(XS_W + 8, ws1 - (x0 - dbase - 4 + uoff)) * 8u;
  const int nrows = min(XH, H - y0);  // output rows of this tile
  int nissued = 0;                    // rows handed to the copy engine so far (every lane keeps the warp-uniform state)
  auto issue = [&](int st) {          // fetch the statistics of the next output row into stage st (lane 0 issues)
    if (lane == 0) {
      const uint32_t bar = ring_bar + 8u * st;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(wbytes + ubytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(ring_w + (uint32_t)(sizeof(float2) * XS_W) * st), "l"(wnext), "r"(wbytes), "r"(bar) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(ring_u + (uint32_t)(sizeof(float2) * (XS_W + 8)) * st), "l"(unext), "r"(ubytes), "r"(bar) : "memory");
    }
    wnext += wstep;
    unext += ustep;
    ++nissued;
  };
  if (lane == 0) {
#pragma unroll
    for (int st = 0; st < NST; ++st) mbar_init(&ring.full[st], 1);
    fence_barrier_init();
  }
  __syncwarp();
#pragma unroll
  for (int e = 0; e < NST; ++e)
    if (e < nrows) issue(e);
  __syncwarp();
  if (WTA && x < W) load_grades(0, grn);
  // the pieces of a row step shared by the two vertical-sum schemes below
  auto load_ab = [&](int r, float (&a)[12], float (&bv)[16]) {
    const float4* ap = reinterpret_cast<const float4*>(arow + r * XS_AW);
    const float4 a0 = ap[0], a1 = ap[1], a2 = ap[2];
    a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w;
    a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
    a[8] = a2.x; a[9] = a2.y; a[10] = a2.z; a[11] = a2.w;
    if (TD == 4) {
      const float4* bp = reinterpret_cast<const float4*>(brow + r * XS_BW);
      const float4 b0 = bp[0], b1 = bp[1], b2 = bp[2], b3 = bp[3];
      bv[0] = b0.x; bv[1] = b0.y; bv[2] = b0.z; bv[3] = b0.w;
      bv[4] = b1.x; bv[5] = b1.y; bv[6] = b1.z; bv[7] = b1.w;
      bv[8] = b2.x; bv[9] = b2.y; bv[10] = b2.z; bv[11] = b2.w;
      bv[12] = b3.x; bv[13] = b3.y; bv[14] = b3.z; bv[15] = b3.w;
    } else {
      const float2* bp = reinterpret_cast<const float2*>(brow + r * XS_BW);
#pragma unroll
      for (int q = 0; q < 7; ++q) {
        const float2 v2 = bp[q];
        bv[2 * q] = v2.x;
        bv[2 * q + 1] = v2.y;
      }
    }
  };
  auto hsum_row = [&](const float (&a)[12], const float (&bv)[16], int dl, float (&hs)[4]) {
    if (BS == 9) {
      xs_hsum9_fma(a, &bv[BOFF - dl], hs);
    } else {
      float p[12];
#pragma unroll
      for (int t = 4 - R; t <= 7 + R; ++t) p[t] = a[t] * bv[BOFF - dl + t];
      xs_hsum<BS>(p, hs);
    }
  };
  // conflict-free 128-bit reads of output row e's statistics (stage st), once per row
  auto load_stats = [&](int st, int e, float2 (&wst)[4], float2 (&ust)[8]) {
    mbar_wait(&ring.full[st], (uint32_t)(e / NST) & 1u);
    const float4* wp = reinterpret_cast<const float4*>(&ring.w[st][4 * lane]);
    const float4* up = reinterpret_cast<const float4*>(&ring.u[st][4 * lane]);
    const float4 w01 = wp[0], w23 = wp[1], u01 = up[0], u23 = up[1], u45 = up[2], u67 = up[3];
    wst[0] = make_float2(w01.x, w01.y); wst[1] = make_float2(w01.z, w01.w);
    wst[2] = make_float2(w23.x, w23.y); wst[3] = make_float2(w23.z, w23.w);
    ust[0] = make_float2(u01.x, u01.y); ust[1] = make_float2(u01.z, u01.w);
    ust[2] = make_float2(u23.x, u23.y); ust[3] = make_float2(u23.z, u23.w);
    ust[4] = make_float2(u45.x, u45.y); ust[5] = make_float2(u45.z, u45.w);
    ust[6] = make_float2(u67.x, u67.y); ust[7] = make_float2(u67.z, u67.w);
  };
  // lane's four columns: {N*mu0, sd0} pairs; its eight u positions (x - dbase - 4 ..): {mu1, sd1} pairs, of which
  // disparity dbase + dl uses positions 4 + k - dl
  // WTA: best[k] = the largest trusted output of column k so far in this row, byte k of bestdl = 1 + its dl (0: none yet);
  // ascending dl and a strict comparison keep the smallest d among equal scores
  auto emit_out = [&](int dl, const float (&S)[4], const float2 (&wst)[4], const float2 (&ust)[8], const unsigned (&gr)[3],
                      float (&best)[4], unsigned& bestdl) {
    float v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 ws_ = wst[k], us_ = ust[4 + k - dl];
      v[k] = fmaf(-ws_.x, us_.x, S[k]) * rcp_approx(fmaf(ws_.y, us_.y, 1e-8f));  // untrusted outputs: see fix-up
    }
    if constexpr (WTA) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int j = 4 + k - dl;  // u position of column k at this disparity
        const unsigned L0 = (gr[0] >> (8 * k)) & 255u, L1 = (gr[1 + j / 4] >> (8 * (j % 4))) & 255u;
        const bool ok = (VEC ? xin : x + k < W) && dl < ndl && L0 + L1 < (unsigned)XS_LSUM;
        if (ok && v[k] > best[k]) {
          best[k] = v[k];
          bestdl = (bestdl & ~(255u << (8 * k))) | ((unsigned)(dl + 1) << (8 * k));
        }
      }
    } else {
      float* dst = orow + dl * dstride;
      if (VEC) {
        if (xin && dl < ndl) __stcs(reinterpret_cast<float4*>(dst), make_float4(v[0], v[1], v[2], v[3]));
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (x + k < W && dl < ndl) dst[k] = v[k];
      }
    }
  };
  // One block of BS tile rows.  FIRST: the tile's first block only fills the vertical state (its last row
  // completes the first window); afterwards every row emits one output row.  Returns true when the tile's
  // last output row has been written.
  auto do_block = [&](auto first_tag, const int blk) -> bool {
    constexpr bool FIRST = decltype(first_tag)::value;
#pragma unroll
    for (int j = 0; j < BS; ++j) {
      const int r = blk * BS + j;
      const bool emit = !FIRST || j == BS - 1;  // compile-time after unrolling
      const int e = r - 2 * R;                  // output row of the tile completed by tile row r
      if (emit && e >= nrows) return true;      // warp-uniform
      unsigned gr[3] = {grn[0], grn[1], grn[2]};
      float best[4];
      unsigned bestdl = 0u;
      if (WTA && emit) {
        if (x < W && e + 1 < nrows) load_grades(e + 1, grn);
#pragma unroll
        for (int k = 0; k < 4; ++k) best[k] = -INFINITY;
      }
      float a[12], bv[16];
      load_ab(r, a, bv);
      // stage of this row's statistics: static when NST divides BS
      const int st = (BS % NST == 0) ? (j + NST * BS - 2 * R) % NST : e % NST;
      float2 wst[4], ust[8];
      if (emit) load_stats(st, e, wst, ust);
#pragma unroll
      for (int dl = 0; dl < TD; ++dl) {
        float hs[4], S[4];
        hsum_row(a, bv, dl, hs);
#if CTD_XS_PACKED_VERTICAL
        // the vertical bookkeeping two columns at a time (FADD2): same additions, half the instructions (520 -> 506 us)
#pragma unroll
        for (int k = 0; k < 4; k += 2) {
          const float2 h2 = make_float2(hs[k], hs[k + 1]);
          float2 f2 = make_float2(F[dl][k], F[dl][k + 1]);
          f2 = j == 0 ? h2 : __fadd2_rn(f2, h2);
          F[dl][k] = f2.x;
          F[dl][k + 1] = f2.y;
          const float2 s2 = j == BS - 1 ? f2 : __fadd2_rn(make_float2(suf[j < BS - 1 ? j : 0][dl][k], suf[j < BS - 1 ? j : 0][dl][k + 1]), f2);
          S[k] = s2.x;
          S[k + 1] = s2.y;
          if (j > 0) {
            suf[j - 1][dl][k] = hs[k];
            suf[j - 1][dl][k + 1] = hs[k + 1];
          }
        }
        if (j == BS - 1) {
#pragma unroll
          for (int k = 0; k < 4; k += 2) {
#pragma unroll
            for (int i = BS - 3; i >= 0; --i) {
              const float2 r2 = __fadd2_rn(make_float2(suf[i][dl][k], suf[i][dl][k + 1]), make_float2(suf[i + 1][dl][k], suf[i + 1][dl][k + 1]));
              suf[i][dl][k] = r2.x;
              suf[i][dl][k + 1] = r2.y;
            }
          }
        }
#else
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          F[dl][k] = j == 0 ? hs[k] : F[dl][k] + hs[k];  // a block starts with its first row (no 0 + x)
          S[k] = j == BS - 1 ? F[dl][k] : suf[j < BS - 1 ? j : 0][dl][k] + F[dl][k];  // suf[j] = rows j+1.. of the previous block
          if (j > 0) suf[j - 1][dl][k] = hs[k];
        }
        if (j == BS - 1) {  // the block is complete: rows -> suffix sums
#pragma unroll
          for (int k = 0; k < 4; ++k) {
#pragma unroll
            for (int i = BS - 3; i >= 0; --i) suf[i][dl][k] += suf[i + 1][dl][k];
          }
        }
#endif
        if (emit) emit_out(dl, S, wst, ust, gr, best, bestdl);
      }
      if (emit) {  // every lane has read this stage: hand it to the row NST further down
        if constexpr (WTA) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const unsigned dl1 = (bestdl >> (8 * k)) & 255u;
            if (dl1 != 0u) atomicMax(orow + k, wta_key(best[k], dbase + (int)dl1 - 1));
          }
        }
        __syncwarp();
        if (nissued < nrows) issue(st);
      }
      orow += W;
    }
    return false;
  };
  if (do_block(std::true_type{}, 0)) return;
#pragma unroll 1
  for (int blk = 1; blk < NBLK; ++blk)
    if (do_block(std::false_type{}, blk)) return;
}

// One output in the fix-up's arithmetic: centred form with the statistics pass's means, or the reference arithmetic
// where a window is flat.
template <int BS>
__device__ __forceinline__ float xcorr_fixed_value(const float* __restrict__ in0, const float* __restrict__ in1,
                                                   const float2* __restrict__ st0, const float2* __restrict__ st1,
                                                   const uint8_t* __restrict__ g0, const uint8_t* __restrict__ g1, int64_t b,
                                                   int h, int w, int d, int H, int W, int ws0, int ws1, int uoff) {
  const int64_t plane = (int64_t)H * W;
  const int64_t i0 = (b * H + h) * ws0 + w, i1 = (b * H + h) * ws1 + (w - d + uoff);
  if (g0[i0] >= XS_LEXACT || g1[i1] >= XS_LEXACT) return xcorr_exact_one<BS>(in0 + b * plane, in1 + b * plane, H, W, h, w, d);
  const float2 s0 = __ldg(st0 + i0), s1 = __ldg(st1 + i1);  // {N mu0, sd0}, {mu1, sd1}
  return xcorr_centred_one<BS>(in0 + b * plane, in1 + b * plane, H, W, h, w, d, s0.x * (1.0f / float(BS * BS)), s1.x, s0.y,
                               s1.y);
}

// where a recomputed output goes: the volume, or (winner-take-all) its pixel's key
__device__ __forceinline__ void xcorr_put(float* __restrict__ out, unsigned bd, int64_t b, int d, int64_t plane, unsigned hw,
                                          float v) {
  out[(int64_t)bd * plane + hw] = v;
}
__device__ __forceinline__ void xcorr_put(unsigned long long* __restrict__ keys, unsigned bd, int64_t b, int d, int64_t plane,
                                          unsigned hw, float v) {
  atomicMax(keys + b * plane + hw, wta_key(v, d));
}

// Recompute one untrusted output.
template <int BS, typename Out>
__device__ __forceinline__ void xcorr_fix_one(const float* __restrict__ in0, const float* __restrict__ in1, Out* __restrict__ out,
                                              const float2* __restrict__ st0, const float2* __restrict__ st1,
                                              const uint8_t* __restrict__ g0, const uint8_t* __restrict__ g1,
                                              unsigned long long e, int H, int W, int D, int ws0, int ws1, int uoff) {
  const int64_t plane = (int64_t)H * W;
  const unsigned hw = (unsigned)(e & 0xffffffffu), bd = (unsigned)(e >> 32);  // h*W + w, b*D + d
  const int w = (int)(hw % (unsigned)W), h = (int)(hw / (unsigned)W);
  const int d = (int)(bd % (unsigned)D);
  const int64_t b = bd / (unsigned)D;
  xcorr_put(out, bd, b, d, plane, hw, xcorr_fixed_value<BS>(in0, in1, st0, st1, g0, g1, b, h, w, d, H, W, ws0, ws1, uoff));
}

// Fix-up, step 1: which outputs are untrusted.  A listed window (side 0: window of in0 at (h, w) -> outputs
// (d, h, w); side 1: window of in1 at (h, u) -> outputs (d, h, u + d) inside the image) is checked against the
// grade of its partner window at every disparity; an output is owned by the side with the larger grade (side 0
// on ties) so it is listed once.  A warp takes SW_BATCH listed windows at a time: their list entries and grades are
// fetched by as many lanes in parallel, then the windows are visited one by one, lane l looking at disparities
// 32c + l, four chunks per step with the partner-grade loads issued together -- the only serial latency per window
// is one load; hits collect in a per-warp shared-memory queue that is flushed to `hits` with one atomic.  nhits
// keeps counting past `cap`, which hands the whole job to xcorr_fixup_kernel (below).
constexpr int SW_BATCH = 8;   // listed windows a warp takes at a time
constexpr int SW_QUEUE = 256;  // per-warp hit queue (flushed with one atomic when half full)
__global__ void __launch_bounds__(256)
xcorr_sweep_kernel(const uint8_t* __restrict__ g0, const uint8_t* __restrict__ g1, const unsigned* __restrict__ list,
                   const unsigned* __restrict__ count, unsigned long long* __restrict__ hits, unsigned* __restrict__ nhits,
                   unsigned cap, int H, int W, int D, int ws0, int ws1, int uoff) {
  __shared__ unsigned long long queue[8][SW_QUEUE];
  const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
  const unsigned nwarps = gridDim.x * (blockDim.x >> 5);
  const unsigned n = *count;
  const unsigned lt = (1u << lane) - 1u;
  unsigned nq = 0;  // warp-uniform queue length
  auto flush = [&]() {
    unsigned slot = 0;
    if (lane == 0) slot = atomicAdd(nhits, nq);
    slot = __shfl_sync(0xffffffffu, slot, 0);
    for (unsigned k = lane; k < nq; k += 32)
      if (slot + k < cap) hits[slot + k] = queue[wl][k];
    nq = 0;
    __syncwarp();
  };
  for (unsigned base = SW_BATCH * (blockIdx.x * (blockDim.x >> 5) + wl); base < n; base += SW_BATCH * nwarps) {
    // lane j < SW_BATCH: the facts of window base + j
    unsigned my_side = 0, my_row = 0, my_L = 0;
    int my_i = 0;
    if (lane < SW_BATCH && base + lane < n) {
      const unsigned e = list[base + lane];
      my_side = e >> 31;
      const unsigned pos = e & 0x7fffffffu, ws = my_side ? (unsigned)ws1 : (unsigned)ws0;
      my_row = pos / ws;  // b*H + h
      my_i = (int)(pos - my_row * ws);
      my_L = my_side ? g1[pos] : g0[pos];
    }
    const int nwin = (int)min((unsigned)SW_BATCH, n - base);
    for (int j = 0; j < nwin; ++j) {
      const unsigned side = __shfl_sync(0xffffffffu, my_side, j), row = __shfl_sync(0xffffffffu, my_row, j);
      const unsigned Ls = __shfl_sync(0xffffffffu, my_L, j);
      const int i = __shfl_sync(0xffffffffu, my_i, j);
      const uint8_t* other = side ? g0 + (size_t)row * ws0 : g1 + (size_t)row * ws1 + uoff;
      const unsigned bD = (row / (unsigned)H) * (unsigned)D, hW = (row % (unsigned)H) * (unsigned)W;
      for (int d0 = 0; d0 < D; d0 += 128) {
        unsigned Lo[4];
        int wv[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {  // the four partner grades of this lane, loads in flight together
          const int d = d0 + 32 * c + lane;
          wv[c] = side ? i - uoff + d : i;
          const bool valid = d < D && wv[c] >= 0 && wv[c] < W;
          Lo[c] = valid ? (unsigned)(side ? other[wv[c]] : other[wv[c] - d]) : 0xffffu;  // 0xffff: never a hit
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const bool hit = Lo[c] != 0xffffu && Ls + Lo[c] >= (unsigned)XS_LSUM && (side ? Ls > Lo[c] : Ls >= Lo[c]);
          const unsigned m = __ballot_sync(0xffffffffu, hit);
          if (hit)
            queue[wl][nq + __popc(m & lt)] =
                ((unsigned long long)(bD + (unsigned)(d0 + 32 * c + lane)) << 32) | (hW + (unsigned)wv[c]);
          nq += __popc(m);
        }
        __syncwarp();
        if (nq >= SW_QUEUE / 2) flush();  // at most 128 entries are added per step
      }
    }
  }
  if (nq > 0) flush();
}

// Fix-up, step 2: one thread per untrusted output (neighbouring hits are neighbouring disparities of one window, so
// the gathers of a warp stay within a few cache lines).
template <int BS, typename Out>
__global__ void __launch_bounds__(256)
xcorr_eval_kernel(const float* __restrict__ in0, const float* __restrict__ in1, Out* __restrict__ out,
                  const float2* __restrict__ st0, const float2* __restrict__ st1, const uint8_t* __restrict__ g0,
                  const uint8_t* __restrict__ g1, const unsigned long long* __restrict__ hits, const unsigned* __restrict__ nhits,
                  unsigned cap, int H, int W, int D, int ws0, int ws1, int uoff) {
  const unsigned n = *nhits;
  if (n > cap) return;  // the list overflowed: xcorr_fixup_kernel does the whole job
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    xcorr_fix_one<BS>(in0, in1, out, st0, st1, g0, g1, hits[i], H, W, D, ws0, ws1, uoff);
}

// Fallback when more outputs are untrusted than the hit list holds (pathological inputs: every window flat):
// the same sweep, but affected outputs are queued per warp and evaluated in place, 32 at a time, so the expensive
// path runs with full warps however sparse the hits are.  Exits at once when the list did not overflow.
// One warp per (listed window, 32 disparities): lane l looks at output d = 32*chunk + l.  side 0: window
// of in0 at (h, w) -> outputs (d, h, w); side 1: window of in1 at (h, u) -> outputs (d, h, u + d) inside the
// image.  An output is owned by the side with the larger grade (side 0 on ties) so it is done once.
// Affected outputs are queued per warp and evaluated 32 at a time, so the expensive path runs with full
// warps however sparse the hits are.
template <int BS, typename Out>
__global__ void __launch_bounds__(256)
xcorr_fixup_kernel(const float* __restrict__ in0, const float* __restrict__ in1, Out* __restrict__ out,
                   const float2* __restrict__ st0, const float2* __restrict__ st1, const uint8_t* __restrict__ g0,
                   const uint8_t* __restrict__ g1, const unsigned* __restrict__ list, const unsigned* __restrict__ count,
                   const unsigned* __restrict__ nhits, unsigned cap, int H, int W, int D, int ws0, int ws1, int uoff) {
  __shared__ unsigned long long queue[8][64];  // (b*D + d) << 32 | (h*W + w)
  if (*nhits <= cap) return;  // the hit list held everything: xcorr_eval_kernel has done the job
  const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
  const unsigned nwarps = gridDim.x * (blockDim.x >> 5);
  const unsigned dchunks = (unsigned)(D + 31) / 32u;
  const unsigned n = *count;
  const int64_t plane = (int64_t)H * W;
  int nq = 0;  // warp-uniform queue length
  auto drain = [&](int m) {  // evaluate the first m (<= 32) queued outputs, one per lane
    if (lane < m) xcorr_fix_one<BS>(in0, in1, out, st0, st1, g0, g1, queue[wl][lane], H, W, D, ws0, ws1, uoff);
    __syncwarp();
  };
  // listed windows are spread over the warps; a warp sweeps the disparities of its window 32 at a time
  for (unsigned it = blockIdx.x * (blockDim.x >> 5) + wl; it < n; it += nwarps) {
    const unsigned e = list[it];
    const unsigned side = e >> 31, pos = e & 0x7fffffffu;
    const unsigned ws = side ? (unsigned)ws1 : (unsigned)ws0;
    const unsigned row = pos / ws;                 // b*H + h
    const int i = (int)(pos - row * ws), h = (int)(row % (unsigned)H);
    const unsigned b = row / (unsigned)H;
    const unsigned Ls = side ? g1[pos] : g0[pos];
    const uint8_t* other = side ? g0 + (size_t)row * ws0 : g1 + (size_t)row * ws1;
    for (unsigned ch = 0; ch < dchunks; ++ch) {
      const int d = (int)(ch * 32u) + lane;
      const int w = side ? i - uoff + d : i;
      bool hit = false;
      if (d < D && w >= 0 && w < W) {
        const unsigned Lo = side ? other[w] : other[w - d + uoff];
        hit = Ls + Lo >= (unsigned)XS_LSUM && (side ? Ls > Lo : Ls >= Lo);
      }
      const unsigned m = __ballot_sync(0xffffffffu, hit);
      if (m == 0u) continue;
      if (hit) {
        const int slot = nq + __popc(m & ((1u << lane) - 1u));
        queue[wl][slot] = ((unsigned long long)(b * (unsigned)D + (unsigned)d) << 32) | (unsigned)(h * W + w);
      }
      nq += __popc(m);
      __syncwarp();
      if (nq >= 32) {
        drain(32);
        if (lane < nq - 32) queue[wl][lane] = queue[wl][lane + 32];
        nq -= 32;
        __syncwarp();
      }
    }
  }
  if (nq > 0) drain(nq);
}

// c[k] = xcorr_fixed_value at d - 1 + k: the rare case of a flat window among the three, kept out of line so that its
// registers do not count against the common path of xcorr_wta_finish_kernel
template <int BS>
__device__ __noinline__ void xcorr_fixed_three(const float* __restrict__ in0, const float* __restrict__ in1,
                                               const float2* __restrict__ st0, const float2* __restrict__ st1,
                                               const uint8_t* __restrict__ g0, const uint8_t* __restrict__ g1, int64_t b, int h,
                                               int w, int d, int H, int W, int ws0, int ws1, int uoff, float (&c)[3]) {
#pragma unroll 1
  for (int k = 0; k < 3; ++k) c[k] = xcorr_fixed_value<BS>(in0, in1, st0, st1, g0, g1, b, h, w, d - 1 + k, H, W, ws0, ws1, uoff);
}

// Winner-take-all, last pass: one thread per pixel decodes d* and the score from its key.  The sub-pixel parabola takes
// the scores at d* - 1, d*, d* + 1 in the fix-up's arithmetic (xcorr_fixed_value: centred form, reference arithmetic
// for flat windows; the three centred ones in one pass) instead of keeping neighbours of every candidate.
template <int BS>
__global__ void __launch_bounds__(256, 3)
xcorr_wta_finish_kernel(const float* __restrict__ in0, const float* __restrict__ in1, const float2* __restrict__ st0,
                        const float2* __restrict__ st1, const uint8_t* __restrict__ g0, const uint8_t* __restrict__ g1,
                        const unsigned long long* __restrict__ keys, float* __restrict__ disp, float* __restrict__ score,
                        int64_t npix, int H, int W, int D, int ws0, int ws1, int uoff, int subpixel) {
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < npix; idx += (int64_t)gridDim.x * blockDim.x) {
    const unsigned long long key = keys[idx];
    const int d = wta_disp(key, D);
    if (score) score[idx] = wta_score(key);
    double delta = 0.0;
    if (subpixel && d > 0 && d < D - 1) {
      const int w = (int)(idx % W), h = (int)((idx / W) % H);
      const int64_t b = idx / ((int64_t)W * H);
      const int64_t i0 = (b * H + h) * ws0 + w, i1 = (b * H + h) * ws1 + (w - d + uoff);  // in1 window of d - 1 + k: i1 + 1 - k
      float c[3];
      if (g0[i0] >= XS_LEXACT || g1[i1 - 1] >= XS_LEXACT || g1[i1] >= XS_LEXACT || g1[i1 + 1] >= XS_LEXACT) {
        xcorr_fixed_three<BS>(in0, in1, st0, st1, g0, g1, b, h, w, d, H, W, ws0, ws1, uoff, c);
      } else {
        const float2 s0 = __ldg(st0 + i0);
        float mu1[3], sd1[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const float2 s1 = __ldg(st1 + i1 + 1 - k);
          mu1[k] = s1.x;
          sd1[k] = s1.y;
        }
        const int64_t plane = (int64_t)H * W;
        xcorr_centred_three<BS>(in0 + b * plane, in1 + b * plane, H, W, h, w, d, s0.x * (1.0f / float(BS * BS)), s0.y, mu1, sd1, c);
      }
      delta = wta_subpixel(c[0], c[1], c[2]);
    }
    disp[idx] = (float)((double)d + delta);
  }
}

// a non-blocking side stream and four events per host thread and device, for the fork / join inside one call
struct SideStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[4] = {};
  int device = -1;
};
int g_xcorr_serial = 0;  // ctd_set_option("xcorr_serial", 1): every kernel of the call on the caller's stream (A/B runs)
static SideStream* side_stream() {
  static thread_local SideStream ss[8];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0) return nullptr;
  SideStream& s = ss[dev % 8];
  if (s.device != dev) {
    if (s.stream != nullptr) return nullptr;  // slot taken by another device (more than 8 devices per thread): serialise
    if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess) {
      cudaGetLastError();
      s.stream = nullptr;
      return nullptr;
    }
    for (int i = 0; i < 4; ++i)
      if (cudaEventCreateWithFlags(&s.ev[i], cudaEventDisableTiming) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
      }
    s.device = dev;
  }
  return &s;
}

// Winner-take-all outputs of one launch (ctd_xcorr_disparity_f32): [B,1,H,W] each; score may be null.
struct XcorrWta {
  float* disp;
  float* score;
  int subpixel;
};

// One launch of the separable path for B images: the volume into `out`, or with `wta` the winner-take-all disparity.
template <int BS>
static bool xcorr_sep_launch(const float* in0, const float* in1, float* out, int64_t B, int64_t H, int64_t W, int64_t D,
                             cudaStream_t st, const XcorrWta* wta = nullptr) {
  constexpr int R = BS / 2, XH = XsCfg<BS>::XH, TH = XsCfg<BS>::TH;
  const int64_t ndchunks = cdiv(D, XS_DT);
  const int64_t uoff = ndchunks * XS_DT, ws0 = cdiv(W, 4) * 4, ws1 = uoff + ws0;
  const int64_t n0 = B * H * ws0, n1 = B * H * ws1;
  if (B * ndchunks > 65535 || cdiv(H, XH) > 65535 || cdiv(H, ST_H) > 65535 || n1 >= ((int64_t)1 << 31)) return false;
  // hit list of the fix-up: room for 1/32 of the outputs, at most 16 M entries (128 MB of scratch).  Block 9 lists 0.2 % of
  // the outputs on the bench frames, block 5 2.5 % (flat 5x5 windows of a 10 % dot pattern): with the former ceiling of 4 M
  // entries block 5 overflowed at batch 8 and ran the fallback kernel, 986 instead of 752 us (xcorr_hitcap_bs5.py).
  // g_xcorr_hitcap >= 0 overrides (tests force the overflow path with 0)
  const int64_t cap = (g_xcorr_hitcap >= 0 ? g_xcorr_hitcap : std::min<int64_t>(B * D * H * W / 32 + 1024, (int64_t)1 << 24)) / 2 * 2;  // even: the statistics planes behind it stay 16-byte aligned
  // winner-take-all: one 64-bit key per pixel, an even count for the same reason
  const int64_t nkeys = wta ? (B * H * W + 1) / 2 * 2 : 0;
  const size_t words = (size_t)(2 * cap + 2 * nkeys) + (size_t)(3 * n0 + 3 * n1 + 4) + (size_t)(n0 + n1 + 3) / 4;
  float* scratch = static_cast<float*>(scratch_alloc(words * sizeof(float), st));
  if (!scratch) return false;
  unsigned long long* hits = reinterpret_cast<unsigned long long*>(scratch);  // 8-byte aligned: first
  unsigned long long* keys = hits + cap;
  float2* st0 = reinterpret_cast<float2*>(keys + nkeys);
  float2* st1 = st0 + n0;
  unsigned* list = reinterpret_cast<unsigned*>(st1 + n1);
  unsigned* count = list + n0 + n1;  // count[0]: listed windows, count[1]: untrusted outputs
  uint8_t* g0 = reinterpret_cast<uint8_t*>(count + 4);
  uint8_t* g1 = g0 + n0;
  const size_t st_smem = sizeof(double) * 2 * (ST_H + 2 * R) * ST_W + sizeof(float) * (ST_H + 2 * R) * (ST_W + 2 * R);
  constexpr int TD = XS_TD;
  // o: the volume (float) or the key plane (unsigned long long); the kernels are instantiated for its type
  auto run = [&](auto* o) -> bool {
    using Out = std::remove_pointer_t<decltype(o)>;
    constexpr bool WTA = std::is_same<Out, unsigned long long>::value;
    const bool fix = WTA || !g_xcorr_nofix;  // the disparity needs the fix-up: untrusted outputs are not in the main kernel's maximum
    const size_t smem = sizeof(float) * TH * (XS_AW + XS_BW) + (16 / TD) * sizeof(XsStatRing<XsNst<TD>::value>);
    // the attribute belongs to the device (context), not to the process: set it on every call (a process may use several GPUs)
    const bool attr_ok =
        cudaFuncSetAttribute(xcorr_stats_kernel<BS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)st_smem) == cudaSuccess &&
        cudaFuncSetAttribute(xcorr_sep_kernel<BS, TD, true, Out>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess &&
        cudaFuncSetAttribute(xcorr_sep_kernel<BS, TD, false, Out>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess;
    if (!attr_ok || cudaMemsetAsync(count, 0, 2 * sizeof(unsigned), st) != cudaSuccess ||
        (WTA && cudaMemsetAsync(keys, 0, sizeof(unsigned long long) * nkeys, st) != cudaSuccess)) {
      cudaGetLastError();
      return false;
    }
    // Fork / join inside the call (legal under stream capture: the side stream joins the capture through the events): the
    // statistics of the two images run side by side, and the sweep over the listed windows -- which needs only the grades
    // -- runs beside the main kernel instead of behind it.  The side stream and the events belong to the calling thread.
    SideStream* ss = side_stream();
    const bool fork = ss != nullptr && !g_xcorr_serial;
    cudaStream_t sd = fork ? ss->stream : st;
    if (fork) {
      cudaEventRecord(ss->ev[0], st);
      cudaStreamWaitEvent(sd, ss->ev[0], 0);
    }
    xcorr_stats_kernel<BS><<<dim3((unsigned)cdiv(ws1, ST_W), (unsigned)cdiv(H, ST_H), (unsigned)B), 256, st_smem, sd>>>(
        in1, st1, g1, (int)H, (int)W, (int)ws1, (int)uoff, 1.0f, 0x80000000u, list, count);
    xcorr_stats_kernel<BS><<<dim3((unsigned)cdiv(ws0, ST_W), (unsigned)cdiv(H, ST_H), (unsigned)B), 256, st_smem, st>>>(
        in0, st0, g0, (int)H, (int)W, (int)ws0, 0, float(BS * BS), 0u, list, count);
    if (fork) {
      cudaEventRecord(ss->ev[1], sd);
      cudaStreamWaitEvent(st, ss->ev[1], 0);   // the main kernel needs both statistics planes
      cudaEventRecord(ss->ev[2], st);
      cudaStreamWaitEvent(sd, ss->ev[2], 0);   // ... and so does the sweep
    }
    const int vec = (W % 4 == 0) && !((reinterpret_cast<uintptr_t>(in0) | reinterpret_cast<uintptr_t>(in1) |
                                       (WTA ? 0 : reinterpret_cast<uintptr_t>(o))) & 15);
    const dim3 sgrid((unsigned)cdiv(W, XS_W), (unsigned)cdiv(H, XH), (unsigned)(B * ndchunks));
    if (fix)
      xcorr_sweep_kernel<<<148 * 8, 256, 0, sd>>>(g0, g1, list, count, hits, count + 1, (unsigned)cap, (int)H, (int)W, (int)D,
                                                 (int)ws0, (int)ws1, (int)uoff);
    if (vec)
      xcorr_sep_kernel<BS, TD, true, Out><<<sgrid, 512 / TD, smem, st>>>(in0, in1, o, st0, st1, g0, g1, (int)H, (int)W, (int)D,
                                                                        (int)ws0, (int)ws1, (int)uoff, (int)ndchunks);
    else
      xcorr_sep_kernel<BS, TD, false, Out><<<sgrid, 512 / TD, smem, st>>>(in0, in1, o, st0, st1, g0, g1, (int)H, (int)W, (int)D,
                                                                         (int)ws0, (int)ws1, (int)uoff, (int)ndchunks);
    if (fork) {
      cudaEventRecord(ss->ev[3], sd);
      cudaStreamWaitEvent(st, ss->ev[3], 0);   // join: the evaluation of the hits overwrites outputs of the main kernel
    }
    if (fix) {
      xcorr_eval_kernel<BS, Out><<<148 * 8, 256, 0, st>>>(in0, in1, o, st0, st1, g0, g1, hits, count + 1, (unsigned)cap, (int)H,
                                                         (int)W, (int)D, (int)ws0, (int)ws1, (int)uoff);
      xcorr_fixup_kernel<BS, Out><<<148 * 3, 256, 0, st>>>(in0, in1, o, st0, st1, g0, g1, list, count, count + 1, (unsigned)cap,
                                                          (int)H, (int)W, (int)D, (int)ws0, (int)ws1, (int)uoff);
    }
    if constexpr (WTA) {
      const int64_t npix = B * H * W;
      xcorr_wta_finish_kernel<BS><<<(unsigned)std::min<int64_t>(cdiv(npix, 256), 148 * 16), 256, 0, st>>>(
          in0, in1, st0, st1, g0, g1, o, wta->disp, wta->score, npix, (int)H, (int)W, (int)D, (int)ws0, (int)ws1, (int)uoff,
          wta->subpixel);
    }
    count_launch(WTA ? 7 : fix ? 6 : 3);
    return true;
  };
  const bool ok = wta ? run(keys) : run(out);
  scratch_free(scratch, st);
  return ok;
}

// Images per separable launch (D, H, W >= 1): as many as keep the fix-up's hit list (1/32 of the outputs, 16 M entries at
// most) at its full relative size (see xcorrvol_impl), and no more than xcorr_sep_launch takes in one launch -- gridDim.z
// = images x disparity chunks <= 65535, statistics positions < 2^31.  A large batch is split into more launches instead
// of leaving the separable path; xcorr_sep_launch refuses only sizes that one image already exceeds.
static int64_t xcorr_images_per_launch(int64_t D, int64_t H, int64_t W) {
  const int64_t ndchunks = cdiv(D, XS_DT), ws1 = ndchunks * XS_DT + cdiv(W, 4) * 4;
  const int64_t hits = (((int64_t)1 << 24) - 1024) * 32 / (D * H * W);
  const int64_t grid = 65535 / ndchunks;
  const int64_t stats = (((int64_t)1 << 31) - 1) / (H * ws1);
  return std::max<int64_t>(1, std::min({hits, grid, stats}));
}

template <typename T>
static int xcorrvol_impl(const T* in0, const T* in1, T* out, int64_t B, int64_t C, int64_t H, int64_t W, int64_t D,
                         int bs, cudaStream_t st) {
  CTD_REQUIRE(B >= 0 && C >= 0 && H >= 0 && W >= 0 && D >= 0, "xcorrvol: negative size");
  CTD_REQUIRE(bs >= 1 && bs <= 255, "xcorrvol: block_size %d out of range [1,255]", bs);
  CTD_REQUIRE(H <= INT32_MAX && W <= INT32_MAX && D <= INT32_MAX && C <= INT32_MAX, "xcorrvol: dimension too large");
  const int64_t total = B * D * H * W;
  if (total == 0) return CTD_OK;
  CTD_REQUIRE(out && (C == 0 || (in0 && in1)), "xcorrvol: null pointer");
  if (sizeof(T) == 4 && C == 1 && !g_force_generic && !g_xcorr_direct && (bs == 3 || bs == 5 || bs == 7 || bs == 9)) {
    const float* f0 = reinterpret_cast<const float*>(in0);
    const float* f1 = reinterpret_cast<const float*>(in1);
    float* fo = reinterpret_cast<float*>(out);
    // Images per launch: as many as keep the fix-up's hit list (1/32 of the outputs, 16 M entries at most) at its full
    // relative size -- a large batch in one launch would overflow the list where many windows are flat (block 5) and fall
    // back to the slow fix-up kernel.  12 images at 480 x 640 x 128: launches that size lose nothing to tails.
    const int64_t per_image = D * H * W;
    const int64_t nb_max = xcorr_images_per_launch(D, H, W);
    bool done = true;
    for (int64_t b0 = 0; b0 < B && done; b0 += nb_max) {
      const int64_t nb = std::min(nb_max, B - b0);
      const float *q0 = f0 + b0 * H * W, *q1 = f1 + b0 * H * W;
      float* qo = fo + b0 * per_image;
      done = bs == 9   ? xcorr_sep_launch<9>(q0, q1, qo, nb, H, W, D, st)
             : bs == 7 ? xcorr_sep_launch<7>(q0, q1, qo, nb, H, W, D, st)
             : bs == 5 ? xcorr_sep_launch<5>(q0, q1, qo, nb, H, W, D, st)
                       : xcorr_sep_launch<3>(q0, q1, qo, nb, H, W, D, st);
      if (!done && b0 > 0) return fail(CTD_ERR_CUDA, "xcorrvol: launch of images %lld.. failed", (long long)b0);
    }
    if (done) return check_launch("xcorrvol(separable)");
  }
  if (sizeof(T) == 4 && C == 1 && !g_force_generic && (bs == 3 || bs == 5 || bs == 7 || bs == 9) && H <= 65535) {
    const int64_t nchunks = cdiv(D, XD_DC);
    for (int64_t b0 = 0; b0 < B; b0 += 1024) {  // keep gridDim.z under 65535
      const int64_t nb = std::min<int64_t>(1024, B - b0);
      if (nb * nchunks > 65535) break;
      const dim3 grid((unsigned)cdiv(W, XD_TW), (unsigned)H, (unsigned)(nb * nchunks));
      const float* p0 = reinterpret_cast<const float*>(in0) + b0 * H * W;
      const float* p1 = reinterpret_cast<const float*>(in1) + b0 * H * W;
      float* po = reinterpret_cast<float*>(out) + b0 * D * H * W;
      if (bs == 9) xcorrvol_direct<9><<<grid, XD_TW, 0, st>>>(p0, p1, po, (int)H, (int)W, (int)D, (int)nchunks);
      else if (bs == 7) xcorrvol_direct<7><<<grid, XD_TW, 0, st>>>(p0, p1, po, (int)H, (int)W, (int)D, (int)nchunks);
      else if (bs == 5) xcorrvol_direct<5><<<grid, XD_TW, 0, st>>>(p0, p1, po, (int)H, (int)W, (int)D, (int)nchunks);
      else xcorrvol_direct<3><<<grid, XD_TW, 0, st>>>(p0, p1, po, (int)H, (int)W, (int)D, (int)nchunks);
      count_launch();
      if (b0 + nb >= B) return check_launch("xcorrvol(direct)");
    }
  }
  const int grid = (int)std::min<int64_t>(cdiv(total, 256), 148 * 256);
  xcorrvol_generic<T><<<grid, 256, 0, st>>>(in0, in1, out, B, (int)C, (int)H, (int)W, (int)D, bs);
  count_launch();
  return check_launch("xcorrvol(generic)");
}

template <typename T>
static int xcorr_disparity_impl(const T* in0, const T* in1, T* disp, T* score, int64_t B, int64_t C, int64_t H, int64_t W,
                                int64_t D, int bs, int subpixel, cudaStream_t st) {
  CTD_REQUIRE(B >= 0 && C >= 0 && H >= 0 && W >= 0 && D >= 0, "xcorr_disparity: negative size");
  CTD_REQUIRE(bs >= 1 && bs <= 255, "xcorr_disparity: block_size %d out of range [1,255]", bs);
  CTD_REQUIRE(H <= INT32_MAX && W <= INT32_MAX && D <= INT32_MAX && C <= INT32_MAX, "xcorr_disparity: dimension too large");
  const int64_t npix = B * H * W;
  if (npix == 0) return CTD_OK;
  CTD_REQUIRE(D >= 1, "xcorr_disparity: n_disps must be >= 1");
  CTD_REQUIRE(disp && (C == 0 || (in0 && in1)), "xcorr_disparity: null pointer");
  if (sizeof(T) == 4 && C == 1 && !g_force_generic && (bs == 3 || bs == 5 || bs == 7 || bs == 9)) {
    const float* f0 = reinterpret_cast<const float*>(in0);
    const float* f1 = reinterpret_cast<const float*>(in1);
    const int64_t nb_max = xcorr_images_per_launch(D, H, W);
    bool done = true;
    for (int64_t b0 = 0; b0 < B && done; b0 += nb_max) {
      const int64_t nb = std::min(nb_max, B - b0), off = b0 * H * W;
      const XcorrWta wta{reinterpret_cast<float*>(disp) + off, score ? reinterpret_cast<float*>(score) + off : nullptr, subpixel};
      const float *q0 = f0 + off, *q1 = f1 + off;
      done = bs == 9   ? xcorr_sep_launch<9>(q0, q1, nullptr, nb, H, W, D, st, &wta)
             : bs == 7 ? xcorr_sep_launch<7>(q0, q1, nullptr, nb, H, W, D, st, &wta)
             : bs == 5 ? xcorr_sep_launch<5>(q0, q1, nullptr, nb, H, W, D, st, &wta)
                       : xcorr_sep_launch<3>(q0, q1, nullptr, nb, H, W, D, st, &wta);
      if (!done && b0 > 0) return fail(CTD_ERR_CUDA, "xcorr_disparity: launch of images %lld.. failed", (long long)b0);
    }
    if (done) return check_launch("xcorr_disparity(separable)");
  }
  const int grid = (int)std::min<int64_t>(cdiv(npix, 256), 148 * 64);
  xcorr_disparity_generic<T><<<grid, 256, 0, st>>>(in0, in1, disp, score, B, (int)C, (int)H, (int)W, (int)D, bs, subpixel);
  count_launch();
  return check_launch("xcorr_disparity(generic)");
}

}  // namespace ctd

CTD_API int ctd_xcorrvol_f32(const float* in0, const float* in1, float* out, int64_t B, int64_t C, int64_t H,
                                int64_t W, int64_t D, int bs, ctd_stream_t s) {
  return ctd::xcorrvol_impl<float>(in0, in1, out, B, C, H, W, D, bs, ctd::as_stream(s));
}
CTD_API int ctd_xcorrvol_f64(const double* in0, const double* in1, double* out, int64_t B, int64_t C, int64_t H,
                                int64_t W, int64_t D, int bs, ctd_stream_t s) {
  return ctd::xcorrvol_impl<double>(in0, in1, out, B, C, H, W, D, bs, ctd::as_stream(s));
}
CTD_API int ctd_xcorr_disparity_f32(const float* in0, const float* in1, float* disp, float* score, int64_t B, int64_t C,
                                    int64_t H, int64_t W, int64_t n_disps, int block_size, int subpixel, ctd_stream_t s) {
  return ctd::xcorr_disparity_impl<float>(in0, in1, disp, score, B, C, H, W, n_disps, block_size, subpixel, ctd::as_stream(s));
}
CTD_API int ctd_xcorr_disparity_f64(const double* in0, const double* in1, double* disp, double* score, int64_t B, int64_t C,
                                    int64_t H, int64_t W, int64_t n_disps, int block_size, int subpixel, ctd_stream_t s) {
  return ctd::xcorr_disparity_impl<double>(in0, in1, disp, score, B, C, H, W, n_disps, block_size, subpixel, ctd::as_stream(s));
}
