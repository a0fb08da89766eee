// The rest of the LCN row of SURVEY.md section 8f-4:
//   * ctd_lcn_bwd_f32: the gradient of networks.LCN (model/networks.py:523-533) w.r.t. its input, i.e. what autograd
//     produces for `(data - avgs) / stds, stds` when upstream gradients arrive for both outputs;
//   * ctd_lcn_cython_f32: the OFFLINE local contrast normalisation of the data generator (data/lcn/lcn.pyx:36-55, called at
//     data/create_syn_data.py:182): no padding (a border of `kernel_size` pixels stays 0), centred two-pass variance,
//     std = sqrt(var) without the 1e-6 floor, out = (x - mean) / (std + eps) -- a different formula from networks.LCN.
#include <algorithm>

#include "ctd_common.cuh"

namespace ctd {
namespace {

__device__ __forceinline__ int reflect_idx(int i, int n) {  // torch ReflectionPad2d: no edge repeat
  i = i < 0 ? -i : i;
  return i >= n ? 2 * (n - 1) - i : i;
}

// ---- LCN backward ---------------------------------------------------------------------------------------------------
// Forward: B = box sum over the reflection-padded image, n = (2r+1)^2, avg = B(x)/n, v = B(x^2)/n - avg^2 + 1e-6,
// s = sqrt(v) + eps, l = (x - avg)/s.  With upstream g_l, g_s:
//   dL/ds = g_s - g_l * l / s,   dL/dv = dL/ds / (2 (s - eps)),   dL/davg = -g_l / s - 2 avg dL/dv,
//   dL/dx = g_l / s + B^T(dL/davg)/n + 2 x B^T(dL/dv)/n,
// B^T = adjoint of the padded box sum: zero-padded box sums evaluated also at the mirror images of the pixel (positions -p
// and 2(W-1) - p of each axis, where they exist), because reflected copies of a pixel feed the windows near the border.
// Kernel 1 (elementwise) writes the two coefficient planes, kernel 2 does the adjoint box sums from shared-memory tiles.
__global__ void __launch_bounds__(256)
lcn_bwd_coeff_kernel(const float* __restrict__ x, const float* __restrict__ l, const float* __restrict__ s, const float* __restrict__ gl,
                     const float* __restrict__ gs, float* __restrict__ ca, float* __restrict__ cv, int64_t n, float eps, float inv_n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float sv = s[i], lv = l[i], g1 = gl ? gl[i] : 0.f, g2 = gs ? gs[i] : 0.f;
    const float inv_s = 1.f / sv;
    const float dls = g2 - g1 * lv * inv_s;
    const float dlv = dls / (2.f * (sv - eps));
    const float avg = x[i] - lv * sv;
    ca[i] = (-g1 * inv_s - 2.f * avg * dlv) * inv_n;
    cv[i] = dlv * inv_n;
  }
}

constexpr int LB_TW = 32, LB_TH = 16, LB_RMAX = 8;  // 37 KB of static shared memory
constexpr int LB_SW = LB_TW + 4 * LB_RMAX, LB_SH = LB_TH + 4 * LB_RMAX;

// tile of LB_TW x LB_TH pixels; shared planes cover the tile plus 2r on every side (zero outside the image): first the
// horizontal pass folds the mirrored centres of each column, then the vertical pass does the same for the rows.
__global__ void __launch_bounds__(256)
lcn_bwd_box_kernel(const float* __restrict__ x, const float* __restrict__ s, const float* __restrict__ gl, const float* __restrict__ ca,
                   const float* __restrict__ cv, float* __restrict__ gx, int H, int W, int r) {
  __shared__ float A[LB_SH][LB_SW + 1], V[LB_SH][LB_SW + 1];
  __shared__ float HA[LB_SH][LB_TW + 1], HV[LB_SH][LB_TW + 1];
  const int x0 = blockIdx.x * LB_TW, y0 = blockIdx.y * LB_TH;
  const int64_t plane = (int64_t)H * W, base = blockIdx.z * plane;
  const int sw = LB_TW + 4 * r, sh = LB_TH + 4 * r;
  for (int i = threadIdx.x; i < sw * sh; i += 256) {
    const int rr = i / sw, cc = i % sw, gy = y0 - 2 * r + rr, gxx = x0 - 2 * r + cc;
    const bool in = gy >= 0 && gy < H && gxx >= 0 && gxx < W;
    A[rr][cc] = in ? ca[base + (int64_t)gy * W + gxx] : 0.f;
    V[rr][cc] = in ? cv[base + (int64_t)gy * W + gxx] : 0.f;
  }
  __syncthreads();
  // horizontal: zero-padded box sum centred at column t of the extended axis = columns t-r..t+r; fold t in {p, -p, 2(W-1)-p}
  for (int i = threadIdx.x; i < sh * LB_TW; i += 256) {
    const int rr = i / LB_TW, c = i % LB_TW, p = x0 + c;
    float sa = 0.f, sv = 0.f;
    if (p < W) {
      const int cen[3] = {p, -p, 2 * (W - 1) - p};
      const bool ok[3] = {true, p >= 1 && p <= r, p <= W - 2 && p >= W - 1 - r};
#pragma unroll
      for (int m = 0; m < 3; ++m) {
        if (!ok[m]) continue;
        const int tc = cen[m] - (x0 - 2 * r);  // tile column of the centre; its window tc-r..tc+r lies inside the staged span
        for (int d = -r; d <= r; ++d) {
          const int col = tc + d;  // columns beyond the staged span lie outside the image (zero)
          if (col >= 0 && col < sw) {
            sa += A[rr][col];
            sv += V[rr][col];
          }
        }
      }
    }
    HA[rr][c] = sa;
    HV[rr][c] = sv;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < LB_TH * LB_TW; i += 256) {
    const int rr = i / LB_TW, c = i % LB_TW, px = x0 + c, py = y0 + rr;
    if (px >= W || py >= H) continue;
    const int cen[3] = {py, -py, 2 * (H - 1) - py};
    const bool ok[3] = {true, py >= 1 && py <= r, py <= H - 2 && py >= H - 1 - r};
    float sa = 0.f, sv = 0.f;
#pragma unroll
    for (int m = 0; m < 3; ++m) {
      if (!ok[m]) continue;
      const int tr = cen[m] - (y0 - 2 * r);
      for (int d = -r; d <= r; ++d) {
        const int row = tr + d;
        if (row >= 0 && row < sh) {
          sa += HA[row][c];
          sv += HV[row][c];
        }
      }
    }
    const int64_t o = base + (int64_t)py * W + px;
    const float g1 = gl ? gl[o] : 0.f;
    gx[o] = g1 / s[o] + sa + 2.f * x[o] * sv;
  }
}

// ---- data/lcn/lcn.pyx ------------------------------------------------------------------------------------------------
// one thread per pixel; the two window passes add in the reference's order (rows outer, columns inner, fp32), so the
// result is the reference's bit for bit (IEEE division and square root)
__global__ void __launch_bounds__(256)
lcn_cython_kernel(const float* __restrict__ img, float* __restrict__ lcn, float* __restrict__ sd, int64_t B, int M, int N, int ks, float eps) {
  const int64_t total = B * M * N;
  const float num = (float)((ks * 2 + 1) * (ks * 2 + 1));
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(idx % N), m = (int)((idx / N) % M);
    float o = 0.f, so = 0.f;
    if (m >= ks && m < M - ks && n >= ks && n < N - ks) {
      const float* p = img + (idx - (int64_t)m * N - n);
      float mean = 0.f;
      for (int i = -ks; i <= ks; ++i)
        for (int j = -ks; j <= ks; ++j) mean = __fadd_rn(mean, __ldg(p + (int64_t)(m + i) * N + n + j));
      mean = __fdiv_rn(mean, num);
      float sdv = 0.f;
      for (int i = -ks; i <= ks; ++i)
        for (int j = -ks; j <= ks; ++j) {
          const float dv = __fsub_rn(__ldg(p + (int64_t)(m + i) * N + n + j), mean);
          sdv = __fadd_rn(sdv, __fmul_rn(dv, dv));
        }
      sdv = __fsqrt_rn(__fdiv_rn(sdv, num));
      o = __fdiv_rn(__fsub_rn(__ldg(p + (int64_t)m * N + n), mean), __fadd_rn(sdv, eps));
      so = sdv;
    }
    lcn[idx] = o;
    sd[idx] = so;
  }
}

}  // namespace
}  // namespace ctd

using namespace ctd;

// d loss / d x of networks.LCN (model/networks.py:523-533) given the forward's input x and outputs (lcn, std) and the
// upstream gradients g_lcn, g_std (either may be NULL = zero).  All [N,1,H,W] fp32; grad_x is overwritten.
CTD_API int ctd_lcn_bwd_f32(const float* x, const float* lcn, const float* std_, const float* g_lcn, const float* g_std, float* grad_x,
                            int64_t N, int64_t H, int64_t W, int radius, float epsilon, ctd_stream_t stream) {
  cudaStream_t st = as_stream(stream);
  CTD_REQUIRE(N >= 0 && H >= 0 && W >= 0, "lcn_bwd: negative size");
  CTD_REQUIRE(radius >= 0 && radius <= LB_RMAX, "lcn_bwd: radius %d out of range [0,%d]", radius, LB_RMAX);
  if (N * H * W == 0) return CTD_OK;
  CTD_REQUIRE(x && lcn && std_ && grad_x, "lcn_bwd: null pointer");
  CTD_REQUIRE(radius < H && radius < W, "lcn_bwd: radius %d needs an image larger than %d x %d (ReflectionPad2d)", radius, (int)H, (int)W);
  CTD_REQUIRE(H <= INT32_MAX && W <= INT32_MAX, "lcn_bwd: dimension too large");
  const int64_t n = N * H * W, plane = H * W;
  float* scratch = static_cast<float*>(scratch_alloc(sizeof(float) * 2 * (size_t)n, st));
  if (!scratch) return fail(CTD_ERR_NOMEM, "lcn_bwd: no scratch memory for the coefficient planes");
  const float inv_n = 1.f / float((2 * radius + 1) * (2 * radius + 1));
  const int g1 = (int)std::min<int64_t>(cdiv(n, 256), 148 * 16);
  lcn_bwd_coeff_kernel<<<g1, 256, 0, st>>>(x, lcn, std_, g_lcn, g_std, scratch, scratch + n, n, epsilon, inv_n);
  count_launch();
  // the box kernel takes the image index from gridDim.z (at most 65535): chunks of images
  for (int64_t b0 = 0; b0 < N; b0 += 65535) {
    const int64_t nb = std::min<int64_t>(65535, N - b0), o = b0 * plane;
    const dim3 grid((unsigned)cdiv(W, LB_TW), (unsigned)cdiv(H, LB_TH), (unsigned)nb);
    lcn_bwd_box_kernel<<<grid, 256, 0, st>>>(x + o, std_ + o, g_lcn ? g_lcn + o : nullptr, scratch + o, scratch + n + o, grad_x + o,
                                             (int)H, (int)W, radius);
    count_launch();
  }
  scratch_free(scratch, st);
  return check_launch("lcn_bwd");
}

// data/lcn/lcn.pyx:16-58 `normalize(img, kernel_size, epsilon)` for a batch of B images [M,N]: (lcn, std), zeros in the
// border of width kernel_size.
CTD_API int ctd_lcn_cython_f32(const float* img, float* lcn, float* std_, int64_t B, int64_t M, int64_t N, int kernel_size, float epsilon,
                               ctd_stream_t stream) {
  CTD_REQUIRE(B >= 0 && M >= 0 && N >= 0 && kernel_size >= 0, "lcn_cython: negative size");
  if (B * M * N == 0) return CTD_OK;
  CTD_REQUIRE(img && lcn && std_, "lcn_cython: null pointer");
  CTD_REQUIRE(M <= INT32_MAX && N <= INT32_MAX && kernel_size <= 64, "lcn_cython: dimension too large");
  const int grid = (int)std::min<int64_t>(cdiv(B * M * N, 256), 148 * 32);
  lcn_cython_kernel<<<grid, 256, 0, as_stream(stream)>>>(img, lcn, std_, B, (int)M, (int)N, kernel_size, epsilon);
  count_launch();
  return check_launch("lcn_cython");
}
