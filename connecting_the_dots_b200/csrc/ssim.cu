// SSIM photometric loss for sm_100a: forward, backward, and forward + backward + masked sums in one kernel.
//
// Definition (DESIGN.md section 4.11).  Per image n, channel c and pixel (h, w) the window is photometric_loss's:
// taps (clamp(h + i - bs/2, 0, H-1), clamp(w + j - bs/2, 0, W-1)), i, j in [0, bs), N = bs^2.  With x = es, y = ta
// and population statistics mx, my, vxx, vyy, vxy over the window
//   A1 = 2 mx my + c1   A2 = 2 vxy + c2   B1 = mx^2 + my^2 + c1   B2 = vxx + vyy + c2   S = A1 A2 / (B1 B2)
//   out[n,0,h,w] = sum_c (1 - S_c) / 2.
// The gradient is taken w.r.t. es only.  With m(w,p) = how many of window w's clamped taps land on p,
//   grad_es[p] = -1/2 sum_w m(w,p) go[w] (a_w + beta_w (x_p - mx_w) + gamma_w (y_p - my_w)),
//   a = 2 (my A2/B2 - mx S) / (N B1),   beta = -2 S / (N B2),   gamma = 2 A1 / (N B1 B2).
//
// Numerics.  Flat windows have vxx ~ 0, and in fp32 E[x^2] - mx^2 rounds to ~1e-8 -- not small against c2 = 9e-4.  So
// the means come from fp32 window sums but the second moments are CENTRED: a second pass over the staged tile forms
// sum (x - mx)^2 etc.  Where es ~ ta, S is close to 1 and both 1 - S and a are differences of nearly equal terms; they
// are evaluated without that cancellation (ssim_eval): with D1 = (mx - my)^2 = B1 - A1 and D2 = var(x - y) = B2 - A2,
// each formed directly (D2 from the centred pass),
//   1 - S = D1/B1 + (A1/B1) (D2/B2),   S = (A1/B1)(1 - D2/B2),   a = -2 (1 - D2/B2)(mx - my)(my (mx + my) + c1) / (N B1^2).  The backward cannot use a per-window shift inside a box adjoint, so it uses one shift (cx, cy)
// per CTA and channel (the (x, y) at the tile's centre):
//   grad = -1/2 [ S^T(go (a - beta (mx - cx) - gamma (my - cy))) + (x - cx) S^T(go beta) + (y - cy) S^T(go gamma) ]
// where S^T is the adjoint of the replicate-clamped box (photo_bwd_box9's, generalised from radius 4 to R): three
// coefficient planes per channel, then a zero-padded box gather whose first / last image row and column collect the
// clamp multiplicity.  A CTA recomputes every window touching its tile (tile + R), so the shift is consistent.
//
// Kernels
//   * ssim_fwd_tile<R>    odd bs = 2R+1 in {3..11}, fp32: (x, y) staged with an R halo as float2 pairs, four windows
//                         per thread (sliding row sums for the means, packed FADD2 / FFMA2 for the centred moments);
//   * ssim_bwd_tile<R, FWD, MASK>   the same window pass on tile + R with a 2R halo, the three go-weighted planes in
//                         shared memory, the separable adjoint gather, grad_in stored; FWD also writes the loss map and
//                         MASK the deterministic masked sums (finish_masked_sums).  No atomics on floating-point data;
//   * generic kernels for everything else (even or large bs, fp64, images smaller than the window, C = 0): a direct
//     per-pixel forward, and a backward as a coefficient pass into scratch planes followed by a gather pass.
// Every output element is overwritten; nothing is allocated with cudaMalloc; all launches are legal under capture.
#include <algorithm>

#include "ctd_common.cuh"

namespace ctd {

extern int g_force_generic;
int masked_sums_launch(const float* diff, const float* mask, int64_t n, float* out2, cudaStream_t st);

namespace {

// ------------------------------------------------------------------------------------------
// generic kernels (any block size, channel count and size; float or double)
// ------------------------------------------------------------------------------------------

// S, the loss (1 - S) / 2 and the gradient coefficients a, beta, gamma (already / N) of one window from its means and
// centred variances vxx, vyy and vee = var(x - y), in the cancellation-free form of the header comment
template <typename T>
struct SsimTerms {
  T S, loss, a, beta, gamma;
};

template <typename T, bool GRAD>
__device__ __forceinline__ SsimTerms<T> ssim_eval(T mx, T my, T vxx, T vyy, T vee, T inv_n, T c1, T c2) {
  const T dm = mx - my;
  const T B1 = mx * mx + my * my + c1, B2 = vxx + vyy + c2;
  const T i1 = T(1) / B1, i2 = T(1) / B2;
  const T r1 = (T(2) * mx * my + c1) * i1, d1 = dm * dm * i1, d2 = vee * i2;  // A1/B1, D1/B1, D2/B2
  SsimTerms<T> t;
  t.S = r1 * (T(1) - d2);
  t.loss = (d1 + r1 * d2) / T(2);
  if (GRAD) {
    t.a = T(-2) * inv_n * (T(1) - d2) * dm * (my * (mx + my) + c1) * (i1 * i1);
    t.beta = T(-2) * inv_n * t.S * i2;
    t.gamma = T(2) * inv_n * r1 * i2;
  }
  return t;
}

// window statistics of pixel (h, w) of one channel plane: means, then centred second moments (all / N).  The generic
// kernels evaluate in fp64 whatever the storage type: they are the slow path, and the accurate side of the tile-kernel
// comparison (force_generic).
template <typename T>
__device__ __forceinline__ void window_stats(const T* __restrict__ x, const T* __restrict__ y, int h, int w, int H, int W,
                                             int bs, double& mx, double& my, double& vxx, double& vyy, double& vee) {
  const int lo = bs / 2;
  const double inv_n = 1.0 / (double)(bs * bs);
  double sx = 0, sy = 0;
  for (int i = 0; i < bs; ++i) {
    const int64_t row = (int64_t)clampi(h + i - lo, 0, H - 1) * W;
    for (int j = 0; j < bs; ++j) {
      const int64_t o = row + clampi(w + j - lo, 0, W - 1);
      sx += (double)x[o];
      sy += (double)y[o];
    }
  }
  mx = sx * inv_n;
  my = sy * inv_n;
  double qxx = 0, qyy = 0, qee = 0;
  for (int i = 0; i < bs; ++i) {
    const int64_t row = (int64_t)clampi(h + i - lo, 0, H - 1) * W;
    for (int j = 0; j < bs; ++j) {
      const int64_t o = row + clampi(w + j - lo, 0, W - 1);
      const double dx = (double)x[o] - mx, dy = (double)y[o] - my;
      qxx += dx * dx;
      qyy += dy * dy;
      qee += (dx - dy) * (dx - dy);
    }
  }
  vxx = qxx * inv_n;
  vyy = qyy * inv_n;
  vee = qee * inv_n;
}

template <typename T>
__global__ void __launch_bounds__(256)
ssim_fwd_generic(const T* __restrict__ es, const T* __restrict__ ta, T* __restrict__ out, int64_t B, int C, int H, int W,
                 int bs, T c1, T c2) {
  const int64_t total = B * H * W, plane = (int64_t)H * W;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int w = idx % W, h = (idx / W) % H;
    const int64_t n = idx / plane;
    double acc = 0;
    for (int c = 0; c < C; ++c) {
      double mx, my, vxx, vyy, vee;
      window_stats<T>(es + (n * C + c) * plane, ta + (n * C + c) * plane, h, w, H, W, bs, mx, my, vxx, vyy, vee);
      acc += ssim_eval<double, false>(mx, my, vxx, vyy, vee, 1.0 / (double)(bs * bs), (double)c1, (double)c2).loss;
    }
    out[idx] = (T)acc;
  }
}

// planes[k * total + (n, c, h, w)] for window (h, w): go*a, go*beta, go*gamma, mx, my
template <typename T>
__global__ void __launch_bounds__(256)
ssim_coef_generic(const T* __restrict__ es, const T* __restrict__ ta, const T* __restrict__ go, T* __restrict__ planes,
                  int64_t B, int C, int H, int W, int bs, T c1, T c2) {
  const int64_t plane = (int64_t)H * W, total = B * C * plane;
  const double inv_n = 1.0 / (double)(bs * bs);
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int w = idx % W, h = (idx / W) % H;
    const int64_t nc = idx / plane, n = nc / C;
    double mx, my, vxx, vyy, vee;
    window_stats<T>(es + nc * plane, ta + nc * plane, h, w, H, W, bs, mx, my, vxx, vyy, vee);
    const SsimTerms<double> t = ssim_eval<double, true>(mx, my, vxx, vyy, vee, inv_n, (double)c1, (double)c2);
    const double g = (double)go[n * plane + (int64_t)h * W + w];
    planes[idx] = (T)(g * t.a);
    planes[total + idx] = (T)(g * t.beta);
    planes[2 * total + idx] = (T)(g * t.gamma);
    planes[3 * total + idx] = (T)mx;
    planes[4 * total + idx] = (T)my;
  }
}

// number of window offsets d in [-lo, hi] with clamp(p + d, 0, n-1) == i
__device__ __forceinline__ int ssim_mult(int p, int i, int n, int lo, int hi) {
  int m = 0;
  for (int d = -lo; d <= hi; ++d) m += (clampi(p + d, 0, n - 1) == i);
  return m;
}

template <typename T>
__global__ void __launch_bounds__(256)
ssim_gather_generic(const T* __restrict__ es, const T* __restrict__ ta, const T* __restrict__ planes, T* __restrict__ gi,
                    int64_t B, int C, int H, int W, int bs) {
  const int64_t plane = (int64_t)H * W, total = B * C * plane;
  const int lo = bs / 2, hi = bs - 1 - lo;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int x = idx % W, y = (idx / W) % H;
    const int64_t base = idx - ((int64_t)y * W + x);
    const double xp = es[idx], yp = ta[idx];
    double acc = 0;
    for (int py = max(0, y - hi); py <= min(H - 1, y + lo); ++py) {
      const int my = ssim_mult(py, y, H, lo, hi);
      if (!my) continue;
      for (int px = max(0, x - hi); px <= min(W - 1, x + lo); ++px) {
        const int mx = ssim_mult(px, x, W, lo, hi);
        if (!mx) continue;
        const int64_t o = base + (int64_t)py * W + px;
        acc += (double)(my * mx) * ((double)planes[o] + (double)planes[total + o] * (xp - (double)planes[3 * total + o]) +
                                    (double)planes[2 * total + o] * (yp - (double)planes[4 * total + o]));
      }
    }
    gi[idx] = (T)(acc / -2.0);
  }
}

// ------------------------------------------------------------------------------------------
// tile kernels, fp32, odd block size 2R+1 <= 11
// ------------------------------------------------------------------------------------------
constexpr int ST_W = 32, ST_H = 32;  // output tile; 256 threads = 32 rows x 8 groups of four columns

__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }

// XY[r * stride + c] = (es, ta) at image (clamp(oy + r), clamp(ox + c)) for r < rows, c < cols; global reads in 16-byte
// chunks aligned in the image row (128-bit loads when vec), scalar clamped reads at the borders
__device__ __forceinline__ void stage_xy(float2* XY, int stride, const float* __restrict__ x, const float* __restrict__ y,
                                         int ox, int oy, int rows, int cols, int H, int W, int vec, int tid) {
  const int xa = ox - (((ox % 4) + 4) % 4);
  const int nch = (ox + cols - xa + 3) / 4;
  for (int it = tid; it < rows * nch; it += 256) {
    const int r = it / nch, k = it % nch;
    const int64_t row = (int64_t)clampi(oy + r, 0, H - 1) * W;
    const int gx = xa + 4 * k;
    float a[4], b[4];
    if (vec && gx >= 0 && gx + 3 < W) {
      const float4 a4 = ldg4(x + row + gx), b4 = ldg4(y + row + gx);
      a[0] = a4.x; a[1] = a4.y; a[2] = a4.z; a[3] = a4.w;
      b[0] = b4.x; b[1] = b4.y; b[2] = b4.z; b[3] = b4.w;
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t o = row + clampi(gx + j, 0, W - 1);
        a[j] = __ldg(x + o);
        b[j] = __ldg(y + o);
      }
    }
    const int c0 = gx - ox;
    float2* dst = XY + r * stride;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (c0 + j >= 0 && c0 + j < cols) dst[c0 + j] = make_float2(a[j], b[j]);
  }
}

// NV consecutive float2 of a staged row (16-byte aligned, NV even)
template <int NV>
__device__ __forceinline__ void load_row2(float2 (&v)[NV], const float2* p) {
  const float4* q = reinterpret_cast<const float4*>(p);
#pragma unroll
  for (int i = 0; i < NV / 2; ++i) {
    const float4 t = q[i];
    v[2 * i] = make_float2(t.x, t.y);
    v[2 * i + 1] = make_float2(t.z, t.w);
  }
}

// Statistics of four horizontally adjacent windows whose top-left taps are p[0..3] (staged (x, y) pairs, row stride
// `stride`): mu = (mx, my), q = (sum (x-mx)^2, sum (y-my)^2), qee = sum ((x-mx) - (y-my))^2, all over the window.
template <int R>
__device__ __forceinline__ void window_stats4(const float2* p, int stride, float2 (&mu)[4], float2 (&q)[4], float (&qee)[4]) {
  constexpr int K = 2 * R + 1, NV = 4 + 2 * R;
  constexpr float INV_N = 1.0f / (float)(K * K);
  float2 s[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) s[k] = make_float2(0.f, 0.f);
#pragma unroll 1
  for (int i = 0; i < K; ++i) {
    float2 v[NV];
    load_row2<NV>(v, p + i * stride);
    float2 r = v[0];
#pragma unroll
    for (int j = 1; j < K; ++j) r = add2(r, v[j]);
    s[0] = add2(s[0], r);
#pragma unroll
    for (int k = 1; k < 4; ++k) {  // slide the row sum one column
      r = add2(r, sub2(v[k + K - 1], v[k - 1]));
      s[k] = add2(s[k], r);
    }
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    mu[k] = __fmul2_rn(s[k], make_float2(INV_N, INV_N));
    q[k] = make_float2(0.f, 0.f);
    qee[k] = 0.f;
  }
#pragma unroll 1
  for (int i = 0; i < K; ++i) {  // per-row partial sums, then added: rounding grows with 2K terms, not K^2
    float2 v[NV];
    load_row2<NV>(v, p + i * stride);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float2 qr = make_float2(0.f, 0.f);
      float qe = 0.f;
#pragma unroll
      for (int j = 0; j < K; ++j) {
        const float2 d = sub2(v[k + j], mu[k]);
        qr = __ffma2_rn(d, d, qr);
        const float e = d.x - d.y;
        qe = fmaf(e, e, qe);
      }
      q[k] = add2(q[k], qr);
      qee[k] += qe;
    }
  }
}

template <int R, bool GRAD>
__device__ __forceinline__ SsimTerms<float> ssim_terms(float2 mu, float2 q, float qee, float c1, float c2) {
  constexpr float INV_N = 1.0f / (float)((2 * R + 1) * (2 * R + 1));
  return ssim_eval<float, GRAD>(mu.x, mu.y, q.x * INV_N, q.y * INV_N, qee * INV_N, INV_N, c1, c2);
}

template <int R>
__global__ void __launch_bounds__(256)
ssim_fwd_tile(const float* __restrict__ es, const float* __restrict__ ta, float* __restrict__ out, int C, int H, int W,
              float c1, float c2, int vec) {
  constexpr int SR = ST_H + 2 * R, SC = ST_W + 2 * R;  // staged rows / columns (SC is even: rows stay 16-byte aligned)
  __shared__ __align__(16) float2 XY[SR * SC];
  const int x0 = blockIdx.x * ST_W, y0 = blockIdx.y * ST_H;
  const int64_t n = blockIdx.z, plane = (int64_t)H * W;
  const int tid = threadIdx.x, q = tid % 8, r = tid / 8;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int c = 0; c < C; ++c) {
    if (c) __syncthreads();
    stage_xy(XY, SC, es + (n * C + c) * plane, ta + (n * C + c) * plane, x0 - R, y0 - R, SR, SC, H, W, vec, tid);
    __syncthreads();
    float2 mu[4], qq[4];
    float qee[4];
    window_stats4<R>(XY + r * SC + 4 * q, SC, mu, qq, qee);
#pragma unroll
    for (int k = 0; k < 4; ++k) acc[k] += ssim_terms<R, false>(mu[k], qq[k], qee[k], c1, c2).loss;
  }
  const int gy = y0 + r, gx = x0 + 4 * q;
  if (gy >= H) return;
  float* dst = out + n * plane + (int64_t)gy * W + gx;
  if (vec) {
    if (gx < W) *reinterpret_cast<float4*>(dst) = make_float4(acc[0], acc[1], acc[2], acc[3]);
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (gx + k < W) dst[k] = acc[k];
  }
}

// shared-memory layout of ssim_bwd_tile
template <int R>
struct BwdGeom {
  static constexpr int RH = ST_H + 2 * R, RW = ST_W + 2 * R;  // windows whose taps reach the tile
  static constexpr int RWP = (RW + 3) & ~3;                    // ... in whole groups of four
  static constexpr int SR = RH + 2 * R, SC = RWP + 2 * R;     // staged (x, y): tile + 2R
  static constexpr size_t XY_FLOATS = 2 * (size_t)SR * SC;
  static constexpr size_t P_FLOATS = 3 * (size_t)RH * RWP;     // go-weighted coefficient planes
  static constexpr size_t H_FLOATS = 3 * (size_t)RH * ST_W;    // their horizontal adjoint sums
  static constexpr size_t L_FLOATS = (size_t)ST_H * ST_W;      // loss map of the tile (summed over channels)
  static constexpr size_t BYTES = 4 * (XY_FLOATS + P_FLOATS + H_FLOATS + L_FLOATS);
};

// One CTA: ST_H x ST_W pixels of one image, every channel.  Per channel: stage (x, y) with a 2R halo, form the windows of
// tile + R and their planes P0 = go (a - beta (mx - cx) - gamma (my - cy)), P1 = go beta, P2 = go gamma (zero for windows
// outside the image), then grad = -1/2 (S^T P0 + (x - cx) S^T P1 + (y - cy) S^T P2) with S^T separable: horizontal sums
// over the window columns plus the clamp multiplicity of the first / last image column, then the same vertically.
// FWD: the loss map from the same windows; MASK: also sums2 = (sum(mask * out), sum(mask)).
template <int R, bool FWD, bool MASK>
__global__ void __launch_bounds__(256)
ssim_bwd_tile(const float* __restrict__ es, const float* __restrict__ ta, const float* __restrict__ go, float* __restrict__ gi,
              float* __restrict__ out, const float* __restrict__ mask, double* __restrict__ partials, unsigned* __restrict__ ticket,
              float* __restrict__ sums2, int C, int H, int W, float c1, float c2, int vec) {
  using G = BwdGeom<R>;
  constexpr int K = 2 * R + 1, NH = 4 + 2 * R;
  extern __shared__ __align__(16) float smem[];
  float2* XY = reinterpret_cast<float2*>(smem);
  float* P = smem + G::XY_FLOATS;
  float* Hs = P + G::P_FLOATS;
  float* L = Hs + G::H_FLOATS;
  const int x0 = blockIdx.x * ST_W, y0 = blockIdx.y * ST_H;
  const int64_t n = blockIdx.z, plane = (int64_t)H * W;
  const int tid = threadIdx.x;
  const float* gon = go + n * plane;
  for (int c = 0; c < C; ++c) {
    if (c) __syncthreads();
    stage_xy(XY, G::SC, es + (n * C + c) * plane, ta + (n * C + c) * plane, x0 - 2 * R, y0 - 2 * R, G::SR, G::SC, H, W, vec, tid);
    __syncthreads();
    const float2 cc = XY[(ST_H / 2 + 2 * R) * G::SC + ST_W / 2 + 2 * R];  // the shift (cx, cy) of this CTA and channel
    // 1. windows of tile + R -> coefficient planes (and the loss map)
    for (int it = tid; it < G::RH * (G::RWP / 4); it += 256) {
      const int r = it / (G::RWP / 4), q4 = 4 * (it % (G::RWP / 4));
      float2 mu[4], qq[4];
      float qee[4];
      window_stats4<R>(XY + r * G::SC + q4, G::SC, mu, qq, qee);
      const int wy = y0 - R + r;
      float p0[4], p1[4], p2[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const SsimTerms<float> t = ssim_terms<R, true>(mu[k], qq[k], qee[k], c1, c2);
        const int wx = x0 - R + q4 + k;
        const float g = (wy >= 0 && wy < H && wx >= 0 && wx < W) ? __ldg(gon + (int64_t)wy * W + wx) : 0.f;
        const float gb = g * t.beta, gg = g * t.gamma;
        p0[k] = fmaf(g, t.a, -fmaf(gb, mu[k].x - cc.x, gg * (mu[k].y - cc.y)));
        p1[k] = gb;
        p2[k] = gg;
        if (FWD) {
          const int tr = r - R, tc = q4 + k - R;
          if (tr >= 0 && tr < ST_H && tc >= 0 && tc < ST_W) {
            const float l = t.loss;
            L[tr * ST_W + tc] = c ? L[tr * ST_W + tc] + l : l;
          }
        }
      }
      const int o = r * G::RWP + q4;
      *reinterpret_cast<float4*>(P + o) = make_float4(p0[0], p0[1], p0[2], p0[3]);
      *reinterpret_cast<float4*>(P + G::RH * G::RWP + o) = make_float4(p1[0], p1[1], p1[2], p1[3]);
      *reinterpret_cast<float4*>(P + 2 * G::RH * G::RWP + o) = make_float4(p2[0], p2[1], p2[2], p2[3]);
    }
    __syncthreads();
    // 2. horizontal adjoint: rows of tile + R, columns of the tile
    for (int it = tid; it < G::RH * (ST_W / 4); it += 256) {
      const int r = it / (ST_W / 4), q4 = 4 * (it % (ST_W / 4));
#pragma unroll
      for (int pl = 0; pl < 3; ++pl) {
        const float* row = P + pl * G::RH * G::RWP + r * G::RWP + q4;  // window columns q4 .. q4 + 3 + 2R
        float v[(NH + 3) & ~3];
#pragma unroll
        for (int i = 0; i < (NH + 3) / 4; ++i) {
          const float4 t = reinterpret_cast<const float4*>(row)[i];
          v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
        }
        float h[4];  // direct sums (the planes have mixed signs: a sliding sum would carry their rounding along)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float s = v[k];
#pragma unroll
          for (int j = 1; j < K; ++j) s += v[k + j];
          h[k] = s;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int gx = x0 + q4 + k;
          if (gx == 0) {  // windows at x = t < R reach column 0 with R - t extra taps
#pragma unroll
            for (int t = 0; t < R; ++t) h[k] = fmaf((float)(R - t), v[k + R + t], h[k]);
          }
          if (gx == W - 1) {  // windows at x = W-1-t likewise
#pragma unroll
            for (int t = 0; t < R; ++t) h[k] = fmaf((float)(R - t), v[k + R - t], h[k]);
          }
        }
        *reinterpret_cast<float4*>(Hs + pl * G::RH * ST_W + r * ST_W + q4) = make_float4(h[0], h[1], h[2], h[3]);
      }
    }
    __syncthreads();
    // 3. vertical adjoint and the gradient of this channel
    {
      const int r = tid / 8, q4 = 4 * (tid % 8);
      const int gy = y0 + r, gx = x0 + q4;
      if (gy < H) {
        float4 V[3];
#pragma unroll
        for (int pl = 0; pl < 3; ++pl) {
          const float* col = Hs + pl * G::RH * ST_W + q4;
          float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int i = 0; i < K; ++i) {
            const float4 t = *reinterpret_cast<const float4*>(col + (r + i) * ST_W);
            acc = make_float4(acc.x + t.x, acc.y + t.y, acc.z + t.z, acc.w + t.w);
          }
          if (gy == 0) {
#pragma unroll
            for (int t = 0; t < R; ++t) {
              const float4 u = *reinterpret_cast<const float4*>(col + (r + R + t) * ST_W);
              const float m = (float)(R - t);
              acc = make_float4(fmaf(m, u.x, acc.x), fmaf(m, u.y, acc.y), fmaf(m, u.z, acc.z), fmaf(m, u.w, acc.w));
            }
          }
          if (gy == H - 1) {
#pragma unroll
            for (int t = 0; t < R; ++t) {
              const float4 u = *reinterpret_cast<const float4*>(col + (r + R - t) * ST_W);
              const float m = (float)(R - t);
              acc = make_float4(fmaf(m, u.x, acc.x), fmaf(m, u.y, acc.y), fmaf(m, u.z, acc.z), fmaf(m, u.w, acc.w));
            }
          }
          V[pl] = acc;
        }
        const float2* xy = XY + (r + 2 * R) * G::SC + q4 + 2 * R;
        const float v0[4] = {V[0].x, V[0].y, V[0].z, V[0].w}, v1[4] = {V[1].x, V[1].y, V[1].z, V[1].w};
        const float v2[4] = {V[2].x, V[2].y, V[2].z, V[2].w};
        float g[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 p = xy[k];
          g[k] = -0.5f * fmaf(p.x - cc.x, v1[k], fmaf(p.y - cc.y, v2[k], v0[k]));
        }
        float* dst = gi + (n * C + c) * plane + (int64_t)gy * W + gx;
        if (vec) {
          if (gx < W) *reinterpret_cast<float4*>(dst) = make_float4(g[0], g[1], g[2], g[3]);
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (gx + k < W) dst[k] = g[k];
        }
      }
    }
  }
  if (FWD) {
    __syncthreads();
    const int r = tid / 8, q4 = 4 * (tid % 8);
    const int gy = y0 + r, gx = x0 + q4;
    float mnum = 0.f, mden = 0.f;
    if (gy < H) {
      const float4 l = *reinterpret_cast<const float4*>(L + r * ST_W + q4);
      const float lv[4] = {l.x, l.y, l.z, l.w};
      const int64_t off = n * plane + (int64_t)gy * W + gx;
      if (MASK) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (gx + k < W) {
            const float m = __ldg(mask + off + k);
            mnum = fmaf(m, lv[k], mnum);
            mden += m;
          }
      }
      if (vec) {
        if (gx < W) *reinterpret_cast<float4*>(out + off) = l;
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (gx + k < W) out[off + k] = lv[k];
      }
    }
    if (MASK) finish_masked_sums((double)mnum, (double)mden, partials, ticket, sums2);
  }
}

// ------------------------------------------------------------------------------------------
// dispatch
// ------------------------------------------------------------------------------------------
int check_args(const void* a, const void* b, const void* c, int64_t B, int64_t C, int64_t H, int64_t W, int bs, double c1,
               double c2) {
  CTD_REQUIRE(B >= 0 && C >= 0 && H >= 0 && W >= 0, "ssim: negative size");
  CTD_REQUIRE(bs >= 1 && bs <= 255, "ssim: block_size %d out of range [1,255]", bs);
  CTD_REQUIRE(c1 > 0 && c2 > 0 && c1 < INFINITY && c2 < INFINITY, "ssim: c1 and c2 must be positive and finite (c1=%g, c2=%g)", c1, c2);
  CTD_REQUIRE(H <= INT32_MAX && W <= INT32_MAX && C <= INT32_MAX, "ssim: dimension too large");
  if (B * C * H * W > 0) CTD_REQUIRE(a && b && c, "ssim: null pointer");
  return CTD_OK;
}

// the tile kernels: odd block sizes 3..11, the image at least one window wide, grid.z = B
bool tile_ok(int bs, int64_t B, int64_t C, int64_t H, int64_t W) {
  return !g_force_generic && bs % 2 == 1 && bs >= 3 && bs <= 11 && H >= bs && W >= bs && C >= 1 && B >= 1 && B <= 65535 &&
         H * W < ((int64_t)1 << 31);
}

int grid_of(int64_t total) { return (int)std::max<int64_t>(1, std::min<int64_t>(cdiv(total, 256), 148 * 64)); }

template <typename T>
int fwd_generic(const T* es, const T* ta, T* out, int64_t B, int64_t C, int64_t H, int64_t W, int bs, double c1, double c2,
                cudaStream_t st) {
  if (B * H * W == 0) return CTD_OK;
  ssim_fwd_generic<T><<<grid_of(B * H * W), 256, 0, st>>>(es, ta, out, B, (int)C, (int)H, (int)W, bs, (T)c1, (T)c2);
  count_launch();
  return check_launch("ssim_fwd(generic)");
}

template <typename T>
int bwd_generic(const T* es, const T* ta, const T* go, T* gi, int64_t B, int64_t C, int64_t H, int64_t W, int bs, double c1,
                double c2, cudaStream_t st) {
  const int64_t total = B * C * H * W;
  if (total == 0) return CTD_OK;
  T* planes = static_cast<T*>(scratch_alloc(5 * (size_t)total * sizeof(T), st));
  if (!planes) return fail(CTD_ERR_NOMEM, "ssim_bwd(generic): no scratch memory for the coefficient planes");
  ssim_coef_generic<T><<<grid_of(total), 256, 0, st>>>(es, ta, go, planes, B, (int)C, (int)H, (int)W, bs, (T)c1, (T)c2);
  ssim_gather_generic<T><<<grid_of(total), 256, 0, st>>>(es, ta, planes, gi, B, (int)C, (int)H, (int)W, bs);
  count_launch(2);
  scratch_free(planes, st);
  return check_launch("ssim_bwd(generic)");
}

bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int vec_of(int64_t W, const void* a, const void* b, const void* c, const void* d) {
  return W % 4 == 0 && al16(a) && al16(b) && al16(c) && al16(d);
}

template <int R>
void fwd_tile_launch(const float* es, const float* ta, float* out, int64_t B, int64_t C, int64_t H, int64_t W, float c1,
                     float c2, cudaStream_t st) {
  const dim3 grid((unsigned)cdiv(W, ST_W), (unsigned)cdiv(H, ST_H), (unsigned)B);
  ssim_fwd_tile<R><<<grid, 256, 0, st>>>(es, ta, out, (int)C, (int)H, (int)W, c1, c2, vec_of(W, es, ta, out, out));
  count_launch();
}

// backward tile kernel; out != nullptr: also the loss map; mask != nullptr: also sums2 (false = no reduction workspace)
template <int R>
bool bwd_tile_launch(const float* es, const float* ta, const float* go, float* gi, float* out, const float* mask, float* sums2,
                     int64_t B, int64_t C, int64_t H, int64_t W, float c1, float c2, cudaStream_t st) {
  const dim3 grid((unsigned)cdiv(W, ST_W), (unsigned)cdiv(H, ST_H), (unsigned)B);
  const size_t smem = BwdGeom<R>::BYTES;
  auto kernel = mask ? ssim_bwd_tile<R, true, true> : (out ? ssim_bwd_tile<R, true, false> : ssim_bwd_tile<R, false, false>);
  // the attribute belongs to the device: set on every call (a process may use several GPUs)
  if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  const int vec = vec_of(W, es, ta, go, gi) && al16(out) && al16(mask);
  MsSlot ms = {nullptr, nullptr, nullptr};
  if (mask && !ms_acquire((size_t)grid.x * grid.y * grid.z, st, &ms)) return false;
  kernel<<<grid, 256, smem, st>>>(es, ta, go, gi, out, mask, ms.partials, ms.ticket, sums2, (int)C, (int)H, (int)W, c1, c2, vec);
  count_launch();
  ms_release(&ms, st);
  return true;
}

#define CTD_SSIM_BY_RADIUS(bs, CALL) \
  switch (bs) {                      \
    case 3: CALL(1); break;          \
    case 5: CALL(2); break;          \
    case 7: CALL(3); break;          \
    case 9: CALL(4); break;          \
    default: CALL(5); break;         \
  }

}  // namespace
}  // namespace ctd

using namespace ctd;

CTD_API int ctd_ssim_fwd_f32(const float* es, const float* ta, float* out, int64_t B, int64_t C, int64_t H, int64_t W,
                             int block_size, double c1, double c2, ctd_stream_t stream) {
  if (int rc = check_args(es, ta, out, B, C, H, W, block_size, c1, c2)) return rc;
  cudaStream_t st = as_stream(stream);
  if (!tile_ok(block_size, B, C, H, W)) return fwd_generic<float>(es, ta, out, B, C, H, W, block_size, c1, c2, st);
#define CALL(R) fwd_tile_launch<R>(es, ta, out, B, C, H, W, (float)c1, (float)c2, st)
  CTD_SSIM_BY_RADIUS(block_size, CALL)
#undef CALL
  return check_launch("ssim_fwd(tile)");
}

CTD_API int ctd_ssim_fwd_f64(const double* es, const double* ta, double* out, int64_t B, int64_t C, int64_t H, int64_t W,
                             int block_size, double c1, double c2, ctd_stream_t stream) {
  if (int rc = check_args(es, ta, out, B, C, H, W, block_size, c1, c2)) return rc;
  return fwd_generic<double>(es, ta, out, B, C, H, W, block_size, c1, c2, as_stream(stream));
}

CTD_API int ctd_ssim_bwd_f32(const float* es, const float* ta, const float* grad_out, float* grad_in, int64_t B, int64_t C,
                             int64_t H, int64_t W, int block_size, double c1, double c2, ctd_stream_t stream) {
  if (int rc = check_args(es, ta, grad_in, B, C, H, W, block_size, c1, c2)) return rc;
  if (B * C * H * W == 0) return CTD_OK;
  CTD_REQUIRE(grad_out, "ssim_bwd: null grad_out");
  cudaStream_t st = as_stream(stream);
  if (tile_ok(block_size, B, C, H, W)) {
    bool ok = false;
#define CALL(R) ok = bwd_tile_launch<R>(es, ta, grad_out, grad_in, nullptr, nullptr, nullptr, B, C, H, W, (float)c1, (float)c2, st)
    CTD_SSIM_BY_RADIUS(block_size, CALL)
#undef CALL
    if (ok) return check_launch("ssim_bwd(tile)");
  }
  return bwd_generic<float>(es, ta, grad_out, grad_in, B, C, H, W, block_size, c1, c2, st);
}

CTD_API int ctd_ssim_bwd_f64(const double* es, const double* ta, const double* grad_out, double* grad_in, int64_t B,
                             int64_t C, int64_t H, int64_t W, int block_size, double c1, double c2, ctd_stream_t stream) {
  if (int rc = check_args(es, ta, grad_in, B, C, H, W, block_size, c1, c2)) return rc;
  if (B * C * H * W == 0) return CTD_OK;
  CTD_REQUIRE(grad_out, "ssim_bwd: null grad_out");
  return bwd_generic<double>(es, ta, grad_out, grad_in, B, C, H, W, block_size, c1, c2, as_stream(stream));
}

// forward + backward + sums2 = (sum(mask * out), sum(mask)) in one kernel (tile path), else the three generic steps
CTD_API int ctd_ssim_fwd_bwd_masked_f32(const float* es, const float* ta, const float* grad_out, const float* mask, float* out,
                                        float* grad_in, float* sums2, int64_t B, int64_t C, int64_t H, int64_t W,
                                        int block_size, double c1, double c2, ctd_stream_t stream) {
  if (int rc = check_args(es, ta, grad_in, B, C, H, W, block_size, c1, c2)) return rc;
  CTD_REQUIRE(sums2 && (B * H * W == 0 || (grad_out && mask && out)), "ssim_fwd_bwd_masked: null pointer");
  cudaStream_t st = as_stream(stream);
  if (B * H * W == 0) {
    CTD_CUDA(cudaMemsetAsync(sums2, 0, 2 * sizeof(float), st));
    return CTD_OK;
  }
  if (tile_ok(block_size, B, C, H, W)) {
    bool ok = false;
#define CALL(R) ok = bwd_tile_launch<R>(es, ta, grad_out, grad_in, out, mask, sums2, B, C, H, W, (float)c1, (float)c2, st)
    CTD_SSIM_BY_RADIUS(block_size, CALL)
#undef CALL
    if (ok) return check_launch("ssim_fwd_bwd_masked(tile)");
  }
  if (int rc = fwd_generic<float>(es, ta, out, B, C, H, W, block_size, c1, c2, st)) return rc;
  if (int rc = bwd_generic<float>(es, ta, grad_out, grad_in, B, C, H, W, block_size, c1, c2, st)) return rc;
  if (int rc = masked_sums_launch(out, mask, B * H * W, sums2, st)) return rc;
  return check_launch("ssim_fwd_bwd_masked(generic)");
}
