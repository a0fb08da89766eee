// Census-transform stereo matching (ctd_census_transform_*, ctd_census_vol_*, ctd_census_disparity_*) for sm_100a.
//
// Definition (include/ctd_b200.h states it in full): T = the census transform of each channel over a (wh, ww) window
// (bit k set when the k-th tap, row-major without the centre, is < the centre; coordinates clamped), Hm[d] =
// sum_c popcount(T0 ^ T1 shifted by -d, column clamped), S = the replicate-padded bs x bs box sum of Hm, V = -S.  Every
// value is an integer of magnitude <= 2^24 (the ABI enforces it), so the kernels reproduce the definition bit for bit in
// either dtype and the fused winner-take-all equals disparity_from_volume(V) including its fp64 sub-pixel offset.
//
// Kernels (one code path per entry point; ctd_set_option("force_generic") does not apply):
//   * census_transform: a CTA stages a tile of CT_ROWS rows x 128 columns plus the window's halo (clamped) in shared
//     memory and writes one uint64 per pixel and channel, two adjacent pixels per thread (128-bit stores where aligned).
//   * census_match<T, R, WTA>: a CTA owns CM_ROWS rows x 128 columns of one image, a warp a row, a lane 4 adjacent
//     pixels.  For each d in order it forms the Hamming plane of the tile plus its R = bs/2 halo (POPC of the XOR of the
//     two descriptors per channel, read through L1), sums it by columns then by rows in shared memory (exact integer
//     sums), and either stores the tile's row of V[d] (128-bit where aligned) or steps the winner-take-all run
//     (WtaRun, ctd_common.cuh) of each of the lane's pixels over -S as int.  R = 0 (bs = 1, the volume SGM consumes) is a
//     compile-time case with no shared memory: the lane's own four pixels are the plane.
// No atomics, no cudaMalloc (descriptor scratch comes from the library pool, stream-ordered), no host synchronisation:
// every call is capture-safe.
#include <algorithm>

#include "ctd_common.cuh"

namespace ctd {

namespace {

constexpr int CT_ROWS = 8;     // census_transform tile rows (a warp per row)
constexpr int CM_ROWS = 8;     // census_match tile rows (a warp per row)
constexpr int TILE_W = 128;    // tile columns: 32 lanes x 4 pixels

__device__ __forceinline__ int popc64(uint64_t x) { return __popcll(x); }

// T[b,c,h,w] of one (b, c) image; a thread makes the words of the pixel pairs (2*lane, 2*lane + 1) and (64 + 2*lane, ...)
template <typename T>
__global__ void __launch_bounds__(32 * CT_ROWS)
census_transform_kernel(const T* __restrict__ in, uint64_t* __restrict__ out, int64_t nimg, int H, int W, int wh, int ww) {
  extern __shared__ __align__(16) unsigned char ct_smem[];
  T* tile = reinterpret_cast<T*>(ct_smem);
  const int rh = wh / 2, rw = ww / 2, tw = TILE_W + 2 * rw, th = CT_ROWS + 2 * rh;
  const int ntx = (W + TILE_W - 1) / TILE_W, nty = (H + CT_ROWS - 1) / CT_ROWS;
  const int64_t ntiles = nimg * ntx * nty;
  const int lane = threadIdx.x & 31, row = threadIdx.x >> 5;
  const int64_t plane = (int64_t)H * W;
  const int centre = rh * ww + rw;
  for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    const int64_t img = t / ((int64_t)ntx * nty);
    const int rem = (int)(t - img * ntx * nty), h0 = (rem / ntx) * CT_ROWS, w0 = (rem % ntx) * TILE_W;
    const T* src = in + img * plane;
    __syncthreads();  // the previous tile's readers are done
    for (int i = threadIdx.x; i < th * tw; i += blockDim.x) {
      const int r = i / tw, c = i - r * tw;
      tile[i] = __ldg(src + (int64_t)clampi(h0 - rh + r, 0, H - 1) * W + clampi(w0 - rw + c, 0, W - 1));
    }
    __syncthreads();
    const int h = h0 + row;
    if (h >= H) continue;
    uint64_t* dst = out + img * plane + (int64_t)h * W;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int c0 = half * 64 + 2 * lane, w = w0 + c0;  // tile column of the pair's left pixel
      if (w >= W) break;
      const T x0 = tile[(row + rh) * tw + c0 + rw], x1 = tile[(row + rh) * tw + c0 + 1 + rw];
      uint64_t b0 = 0, b1 = 0;
      int k = 0;  // tap index of (i, j) with the centre left out
      for (int i = 0; i < wh; ++i) {
        const T* trow = tile + (row + i) * tw + c0;
        T prev = trow[0];
        for (int j = 0; j < ww; ++j) {
          const T next = trow[j + 1];
          if (i * ww + j != centre) {
            b0 |= (uint64_t)(prev < x0) << k;
            b1 |= (uint64_t)(next < x1) << k;
            ++k;
          }
          prev = next;
        }
      }
      if (w + 1 < W && aligned16(dst + w)) {
        *reinterpret_cast<ulonglong2*>(dst + w) = make_ulonglong2(b0, b1);
      } else {
        dst[w] = b0;
        if (w + 1 < W) dst[w + 1] = b1;
      }
    }
  }
}

// store the four scores -S of pixels w .. w + 3 of one row (those inside the image)
template <typename T>
__device__ __forceinline__ void store4(T* p, int w, int W, const int (&s)[4]) {
  if (w + 3 < W && aligned16(p)) {
    if (sizeof(T) == 4) {
      *reinterpret_cast<float4*>(p) = make_float4(-(float)s[0], -(float)s[1], -(float)s[2], -(float)s[3]);
    } else {
      reinterpret_cast<double2*>(p)[0] = make_double2(-(double)s[0], -(double)s[1]);
      reinterpret_cast<double2*>(p)[1] = make_double2(-(double)s[2], -(double)s[3]);
    }
  } else {
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (w + k < W) p[k] = -(T)s[k];
  }
}

template <typename T, int R, bool WTA>
__global__ void __launch_bounds__(32 * CM_ROWS)
census_match(const uint64_t* __restrict__ t0, const uint64_t* __restrict__ t1, T* __restrict__ vol, T* __restrict__ disp,
             T* __restrict__ score, int64_t B, int C, int H, int W, int D, int subpixel) {
  constexpr int HW_ = TILE_W + 2 * R;                   // halo tile width
  constexpr int PITCH = 4 * ((TILE_W + 2 * R + 3) / 4);  // row pitch: int4 reads of a lane's 4 + 2R window stay inside
  constexpr int HROWS = CM_ROWS + 2 * R;
  __shared__ __align__(16) int hm[R > 0 ? HROWS * PITCH : 1];
  __shared__ __align__(16) int cs[R > 0 ? CM_ROWS * PITCH : 1];
  const int lane = threadIdx.x & 31, row = threadIdx.x >> 5;
  const int ntx = (W + TILE_W - 1) / TILE_W, nty = (H + CM_ROWS - 1) / CM_ROWS;
  const int64_t plane = (int64_t)H * W, ntiles = B * ntx * nty;
  const int64_t cstride = plane;  // channel stride of T
  for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    const int64_t b = t / ((int64_t)ntx * nty);
    const int rem = (int)(t - b * ntx * nty), h0 = (rem / ntx) * CM_ROWS, w0 = (rem % ntx) * TILE_W;
    const int h = h0 + row, w = w0 + 4 * lane;
    const uint64_t* a0 = t0 + b * C * plane;
    const uint64_t* a1 = t1 + b * C * plane;
    WtaRun<int> run[4];  // over -S: its first maximum is the first minimum of S
#pragma unroll
    for (int k = 0; k < 4; ++k) run[k].init();
    for (int d = 0; d < D; ++d) {
      int s[4];
      if constexpr (R == 0) {
        // the lane's own pixels (clamped reads past the right edge are computed and not stored)
        const int hc = min(h, H - 1);
#pragma unroll
        for (int k = 0; k < 4; ++k) s[k] = 0;
        for (int c = 0; c < C; ++c) {
          const uint64_t* r0 = a0 + c * cstride + (int64_t)hc * W;
          const uint64_t* r1 = a1 + c * cstride + (int64_t)hc * W;
          uint64_t x[4];
          if (w + 3 < W && aligned16(r0 + w)) {
            const ulonglong2 p = __ldg(reinterpret_cast<const ulonglong2*>(r0 + w));
            const ulonglong2 q = __ldg(reinterpret_cast<const ulonglong2*>(r0 + w + 2));
            x[0] = p.x, x[1] = p.y, x[2] = q.x, x[3] = q.y;
          } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) x[k] = __ldg(r0 + min(w + k, W - 1));
          }
#pragma unroll
          for (int k = 0; k < 4; ++k) s[k] += popc64(x[k] ^ __ldg(r1 + max(min(w + k, W - 1) - d, 0)));
        }
      } else {
        __syncthreads();  // the previous d's readers of hm and cs are done
        // Hamming plane of the tile plus its halo, at clamped coordinates
        for (int i = threadIdx.x; i < HROWS * HW_; i += blockDim.x) {
          const int r = i / HW_, c = i - r * HW_;
          const int hc = clampi(h0 - R + r, 0, H - 1), wc = clampi(w0 - R + c, 0, W - 1), ws = max(wc - d, 0);
          const uint64_t* r0 = a0 + (int64_t)hc * W;
          const uint64_t* r1 = a1 + (int64_t)hc * W;
          int acc = 0;
          for (int ch = 0; ch < C; ++ch) acc += popc64(__ldg(r0 + ch * cstride + wc) ^ __ldg(r1 + ch * cstride + ws));
          hm[r * PITCH + c] = acc;
        }
        __syncthreads();
        // column sums over 2R + 1 rows, a running sum down each column
        for (int c = threadIdx.x; c < HW_; c += blockDim.x) {
          int acc = 0;
#pragma unroll
          for (int r = 0; r < 2 * R; ++r) acc += hm[r * PITCH + c];
#pragma unroll
          for (int r = 0; r < CM_ROWS; ++r) {
            acc += hm[(r + 2 * R) * PITCH + c];
            cs[r * PITCH + c] = acc;
            acc -= hm[r * PITCH + c];
          }
        }
        __syncthreads();
        // row sums over 2R + 1 columns for the lane's 4 pixels, from (4 + 2R) column sums read as int4
        constexpr int NV = (4 + 2 * R + 3) / 4;
        int v[4 * NV];
#pragma unroll
        for (int q = 0; q < NV; ++q) {
          const int4 x = *reinterpret_cast<const int4*>(cs + row * PITCH + 4 * lane + 4 * q);
          v[4 * q] = x.x, v[4 * q + 1] = x.y, v[4 * q + 2] = x.z, v[4 * q + 3] = x.w;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          int acc = 0;
#pragma unroll
          for (int j = 0; j <= 2 * R; ++j) acc += v[k + j];
          s[k] = acc;
        }
      }
      if (h < H) {
        if (!WTA) {
          store4<T>(vol + (b * D + d) * plane + (int64_t)h * W + w, w, W, s);
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k) run[k].step(-s[k], d);
        }
      }
    }
    if (WTA && h < H) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (w + k >= W) break;
        // the score is -(T)S like the volume's (S = 0 is -0.0); the sign of a zero cm or cp does not change the offset
        const WtaRun<int>& r = run[k];
        wta_store<T>(disp, score, b * plane + (int64_t)h * W + w + k, r.bd, -(T)(-r.best), (T)r.cm, (T)r.cp, D, subpixel);
      }
    }
  }
}

template <typename T>
int transform_launch(const T* in, uint64_t* out, int64_t nimg, int H, int W, int wh, int ww, cudaStream_t st) {
  const size_t smem = (size_t)(CT_ROWS + 2 * (wh / 2)) * (TILE_W + 2 * (ww / 2)) * sizeof(T);
  auto kernel = census_transform_kernel<T>;
  const int rs = raise_smem_limit(kernel, smem, "census_transform");
  if (rs != CTD_OK) return rs;
  const int64_t ntiles = nimg * cdiv(W, TILE_W) * cdiv(H, CT_ROWS);
  kernel<<<(unsigned)std::min<int64_t>(ntiles, INT32_MAX), 32 * CT_ROWS, smem, st>>>(in, out, nimg, H, W, wh, ww);
  count_launch();
  return check_launch("census_transform");
}

template <typename T, int R>
int match_launch_r(const uint64_t* t0, const uint64_t* t1, T* vol, T* disp, T* score, int64_t B, int C, int H, int W, int D,
                   int subpixel, cudaStream_t st) {
  const int64_t ntiles = B * cdiv(W, TILE_W) * cdiv(H, CM_ROWS);
  const unsigned grid = (unsigned)std::min<int64_t>(ntiles, INT32_MAX);
  if (vol)
    census_match<T, R, false><<<grid, 32 * CM_ROWS, 0, st>>>(t0, t1, vol, nullptr, nullptr, B, C, H, W, D, 0);
  else
    census_match<T, R, true><<<grid, 32 * CM_ROWS, 0, st>>>(t0, t1, nullptr, disp, score, B, C, H, W, D, subpixel);
  count_launch();
  return check_launch(vol ? "census_vol" : "census_disparity");
}

template <typename T>
int match_launch(const uint64_t* t0, const uint64_t* t1, T* vol, T* disp, T* score, int64_t B, int C, int H, int W, int D, int bs,
                 int subpixel, cudaStream_t st) {
  switch (bs / 2) {
#define CTD_CENSUS_R(R) \
  case R: return match_launch_r<T, R>(t0, t1, vol, disp, score, B, C, H, W, D, subpixel, st);
    CTD_CENSUS_R(0) CTD_CENSUS_R(1) CTD_CENSUS_R(2) CTD_CENSUS_R(3) CTD_CENSUS_R(4) CTD_CENSUS_R(5) CTD_CENSUS_R(6)
    CTD_CENSUS_R(7)
#undef CTD_CENSUS_R
  }
  return fail(CTD_ERR_INVALID, "census: block_size %d out of range", bs);
}

// the checks every entry point shares, in the order the header lists them (before any device work)
int check_window(const char* op, int64_t B, int64_t C, int64_t H, int64_t W, int wh, int ww, int bs) {
  CTD_REQUIRE(wh >= 1 && ww >= 1 && (wh & 1) && (ww & 1), "%s: window sides must be odd and positive, got %dx%d", op, wh, ww);
  CTD_REQUIRE((int64_t)wh * ww >= 2 && (int64_t)wh * ww <= 65, "%s: window %dx%d must have 2 to 65 taps", op, wh, ww);
  CTD_REQUIRE(bs >= 1 && bs <= 15 && (bs & 1), "%s: block_size must be odd in [1,15], got %d", op, bs);
  CTD_REQUIRE(B >= 0 && C >= 0 && H >= 0 && W >= 0, "%s: negative size", op);
  CTD_REQUIRE(H <= INT32_MAX && W <= INT32_MAX && C <= INT32_MAX, "%s: dimension too large", op);
  CTD_REQUIRE(C * (wh * ww - 1) * bs * bs <= (1 << 24),
              "%s: C*(wh*ww-1)*block_size^2 = %lld exceeds 2^24 (scores would not be exact in float32)", op,
              (long long)(C * (wh * ww - 1) * bs * bs));
  return CTD_OK;
}

}  // namespace

template <typename T>
static int census_transform_impl(const T* in, uint64_t* out, int64_t B, int64_t C, int64_t H, int64_t W, int wh, int ww,
                                 cudaStream_t st) {
  const int rc = check_window("census_transform", B, C, H, W, wh, ww, 1);
  if (rc != CTD_OK) return rc;
  const int64_t n = B * C * H * W;
  if (n == 0) return CTD_OK;
  CTD_REQUIRE(in && out, "census_transform: null pointer");
  CTD_REQUIRE(ranges_disjoint(in, n * sizeof(T), out, n * sizeof(uint64_t)), "census_transform: out overlaps in");
  return transform_launch<T>(in, out, B * C, (int)H, (int)W, wh, ww, st);
}

// census_vol (vol != null) or census_disparity (vol == null)
template <typename T>
static int census_match_impl(bool is_vol, const T* in0, const T* in1, T* vol, T* disp, T* score, int64_t B, int64_t C,
                             int64_t H, int64_t W, int64_t D, int wh, int ww, int bs, int subpixel, cudaStream_t st) {
  const char* op = is_vol ? "census_vol" : "census_disparity";
  const int rc = check_window(op, B, C, H, W, wh, ww, bs);
  if (rc != CTD_OK) return rc;
  CTD_REQUIRE(D >= 0 && D <= INT32_MAX, "%s: n_disps %lld out of range", op, (long long)D);
  const int64_t npix = B * H * W;
  if (npix == 0) return CTD_OK;
  CTD_REQUIRE(D >= 1, "%s: n_disps must be >= 1 (D = 0)", op);
  CTD_REQUIRE((C == 0 || (in0 && in1)) && (is_vol ? vol != nullptr : disp != nullptr), "%s: null pointer", op);
  const size_t nin = (size_t)(npix * C) * sizeof(T), nvol = is_vol ? (size_t)(npix * D) * sizeof(T) : 0;
  const size_t nmap = is_vol ? 0 : (size_t)npix * sizeof(T);
  const void* outs[3] = {vol, disp, score};
  const size_t nout[3] = {nvol, nmap, nmap};
  for (int i = 0; i < 3; ++i)
    CTD_REQUIRE(ranges_disjoint(outs[i], nout[i], in0, nin) && ranges_disjoint(outs[i], nout[i], in1, nin),
                "%s: an output overlaps an input", op);
  CTD_REQUIRE(ranges_disjoint(disp, nmap, score, nmap), "%s: disp overlaps score", op);
  const size_t words = (size_t)(npix * C);
  uint64_t* t = words ? static_cast<uint64_t*>(scratch_alloc(2 * words * sizeof(uint64_t), st)) : nullptr;
  CTD_REQUIRE(!words || t, "%s: no scratch memory for the descriptors (%zu bytes)", op, 2 * words * sizeof(uint64_t));
  int r = CTD_OK;
  if (words) r = transform_launch<T>(in0, t, B * C, (int)H, (int)W, wh, ww, st);
  if (r == CTD_OK && words) r = transform_launch<T>(in1, t + words, B * C, (int)H, (int)W, wh, ww, st);
  if (r == CTD_OK) r = match_launch<T>(t, t + words, vol, disp, score, B, (int)C, (int)H, (int)W, (int)D, bs, subpixel, st);
  if (t) scratch_free(t, st);
  return r;
}

}  // namespace ctd

CTD_API int ctd_census_transform_f32(const float* in, uint64_t* out, int64_t B, int64_t C, int64_t H, int64_t W, int wh, int ww,
                                     ctd_stream_t s) {
  return ctd::census_transform_impl<float>(in, out, B, C, H, W, wh, ww, ctd::as_stream(s));
}
CTD_API int ctd_census_transform_f64(const double* in, uint64_t* out, int64_t B, int64_t C, int64_t H, int64_t W, int wh, int ww,
                                     ctd_stream_t s) {
  return ctd::census_transform_impl<double>(in, out, B, C, H, W, wh, ww, ctd::as_stream(s));
}
CTD_API int ctd_census_vol_f32(const float* in0, const float* in1, float* out, int64_t B, int64_t C, int64_t H, int64_t W,
                               int64_t n_disps, int wh, int ww, int block_size, ctd_stream_t s) {
  return ctd::census_match_impl<float>(true, in0, in1, out, nullptr, nullptr, B, C, H, W, n_disps, wh, ww, block_size, 0,
                                       ctd::as_stream(s));
}
CTD_API int ctd_census_vol_f64(const double* in0, const double* in1, double* out, int64_t B, int64_t C, int64_t H, int64_t W,
                               int64_t n_disps, int wh, int ww, int block_size, ctd_stream_t s) {
  return ctd::census_match_impl<double>(true, in0, in1, out, nullptr, nullptr, B, C, H, W, n_disps, wh, ww, block_size, 0,
                                        ctd::as_stream(s));
}
CTD_API int ctd_census_disparity_f32(const float* in0, const float* in1, float* disp, float* score, int64_t B, int64_t C, int64_t H,
                                     int64_t W, int64_t n_disps, int wh, int ww, int block_size, int subpixel, ctd_stream_t s) {
  return ctd::census_match_impl<float>(false, in0, in1, nullptr, disp, score, B, C, H, W, n_disps, wh, ww, block_size,
                                       subpixel, ctd::as_stream(s));
}
CTD_API int ctd_census_disparity_f64(const double* in0, const double* in1, double* disp, double* score, int64_t B, int64_t C,
                                     int64_t H, int64_t W, int64_t n_disps, int wh, int ww, int block_size, int subpixel,
                                     ctd_stream_t s) {
  return ctd::census_match_impl<double>(false, in0, in1, nullptr, disp, score, B, C, H, W, n_disps, wh, ww,
                                        block_size, subpixel, ctd::as_stream(s));
}
