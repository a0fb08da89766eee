// Left-right consistency and uniqueness checks over a [B,D,H,W] score volume (ctd_disparity_check_*) for sm_100a.
//
// Definition (include/ctd_b200.h states it in full): the left view is disparity_from_volume(V) (first maximum over d,
// fp64 three-point sub-pixel offset); the right view of right pixel x is the same winner-take-all over VR[d] = V[d,x+d],
// d < Dx = min(D, W - x); valid = LR (x = w - d*L >= 0 and |d*L - dR*(x)| <= max_diff, or max_diff < 0) and uniqueness
// (V[d*L] - max{V[d] : |d - d*L| >= 2} >= uniqueness in fp64, or uniqueness = 0, or that set empty).  Only maxima, compares
// and the stated fp64 operations are involved, so every output is bit-equal to the definition.
//
// Kernel (one code path for every W and D): a CTA owns an image row (b, h) and walks it in chunks of seg = 4 * blockDim.x
// columns (one chunk when W <= seg, the common case); a thread owns pixels w0 + tid + k * blockDim.x, k < 4, as a left
// pixel w and as a right pixel x at once.  The rows V[d,h,w0 .. w0+seg) of DC_DS = 4 consecutive d (and, for a chunk that
// is not the last, the columns [w0+seg, w0+seg+d) the right pixels reach past it) fill one slot of a 4-slot shared ring
// through coalesced cp.async copies (16 bytes where aligned), three slots ahead; one barrier per slot.  For each d the
// thread then steps two winner-take-all runs (WtaRun, ctd_common.cuh), the left one over buf[w] and the right one over
// buf[x + d], and, for the left pixel, the uniqueness maxima: the prefix maximum of V lagged by two steps (the maximum
// below d*-1, taken at each new best) and the maximum over d >= d*+2 (reset at each new best).
// After the chunk's last d the right pixels store dR* in a per-CTA row of pool scratch; after one barrier each left pixel
// reads dR*(w - d*L), which lies in this chunk or an earlier one of the same row.  Every element of V is read from global
// memory once (twice for columns a wide row's right pixels reach across a chunk boundary).  No atomics, no host
// synchronisation, scratch from the library's stream-ordered pool: every call is capture-safe.
#include <cuda_pipeline.h>

#include <algorithm>
#include <cmath>

#include "ctd_common.cuh"

namespace ctd {

namespace {

constexpr int DC_PPT = 4;       // pixels per thread
constexpr int DC_MAXT = 256;    // threads per CTA at most: a chunk is at most 1024 columns
constexpr int DC_DS = 4;        // disparities staged per ring slot (one barrier per DC_DS rows of V)
constexpr int DC_STAGES = 4;    // ring slots; the copies of DC_STAGES - 1 groups are in flight

// columns [0, n) of a row starting at src into dst (16-byte aligned): 16-byte copies when src is aligned, then the tail
template <typename T>
__device__ __forceinline__ void stage_columns(T* dst, const T* src, int n) {
  constexpr int V = 16 / sizeof(T);
  int done = 0;
  if (aligned16(src)) {
    const int nv = n / V;
    for (int i = threadIdx.x; i < nv; i += blockDim.x) __pipeline_memcpy_async(dst + i * V, src + i * V, 16);
    done = nv * V;
  }
  for (int i = done + threadIdx.x; i < n; i += blockDim.x) __pipeline_memcpy_async(dst + i, src + i, sizeof(T));
}

// position of one CTA's walk: image row `row` (b * H + h, whose V[b,0,h,0] is at element `off`), chunk `ch` of the row,
// group `g` of DC_DS disparities
struct DcCursor {
  int64_t row, off;
  int ch, g;
  __device__ __forceinline__ void seek(int64_t r, int D, int H, int W) {
    const int64_t b = r / H;
    row = r, off = (b * D * H + (r - b * H)) * W, ch = 0, g = 0;
  }
  __device__ __forceinline__ void next(int ngroups, int nch, int D, int H, int W) {
    if (++g == ngroups) {
      g = 0;
      if (++ch == nch) seek(row + gridDim.x, D, H, W);
    }
  }
};

template <typename T>
__global__ void __launch_bounds__(DC_MAXT)
disparity_check_kernel(const T* __restrict__ vol, T* __restrict__ disp, T* __restrict__ score, T* __restrict__ disp_r,
                       T* __restrict__ score_r, uint8_t* __restrict__ valid, int* dr_rows, int64_t B, int D, int H, int W,
                       int stage_elems, int max_diff, double uniqueness, int subpixel) {
  extern __shared__ __align__(16) unsigned char dc_smem[];
  T* ring = reinterpret_cast<T*>(dc_smem);
  const T ninf = lowest<T>();
  const int seg = DC_PPT * blockDim.x, nch = (W + seg - 1) / seg, ngroups = (D + DC_DS - 1) / DC_DS;
  const int64_t nrows = B * H, plane = (int64_t)H * W;
  const bool lr_check = valid && max_diff >= 0;
  int* dr = lr_check ? dr_rows + (int64_t)blockIdx.x * W : nullptr;  // dR* of this CTA's current row

  // issue the copies of group f into ring slot `slot`: per d, the chunk's columns and those its right pixels reach past it
  auto fetch = [&](const DcCursor& f, int slot) {
    const int w0 = f.ch * seg, aend = min(W, w0 + seg);
#pragma unroll
    for (int j = 0; j < DC_DS; ++j) {
      const int d = f.g * DC_DS + j;
      if (d >= D) break;
      const T* src = vol + f.off + d * plane;
      T* dst = ring + (size_t)(slot * DC_DS + j) * stage_elems;
      stage_columns<T>(dst, src + w0, aend - w0);
      const int bstart = max(aend, w0 + d), bend = (int)min((long long)W, (long long)aend + d);
      if (bstart < bend) stage_columns<T>(dst + seg, src + bstart, bend - bstart);
    }
  };

  DcCursor f, c;
  f.seek(blockIdx.x, D, H, W);
  c = f;
  int fslot = 0, cslot = 0;
  for (int s = 0; s < DC_STAGES - 1; ++s) {
    if (f.row < nrows) fetch(f, fslot);
    __pipeline_commit();
    f.next(ngroups, nch, D, H, W);
    fslot = fslot + 1 == DC_STAGES ? 0 : fslot + 1;
  }

  // the runs of the thread's left and right pixels and the left pixels' uniqueness maxima (see the file comment)
  WtaRun<T> L[DC_PPT], R[DC_PPT];
  T lpm[DC_PPT], lsec[DC_PPT], lfar[DC_PPT];
  while (c.row < nrows) {
    __pipeline_wait_prior(DC_STAGES - 2);
    __syncthreads();  // group c's rows are in; every thread is done with the slot the next fetch overwrites
    if (f.row < nrows) fetch(f, fslot);
    __pipeline_commit();
    f.next(ngroups, nch, D, H, W);
    fslot = fslot + 1 == DC_STAGES ? 0 : fslot + 1;

    const T* slot = ring + (size_t)cslot * DC_DS * stage_elems;
    cslot = cslot + 1 == DC_STAGES ? 0 : cslot + 1;
    const int w0 = c.ch * seg, aend = min(W, w0 + seg);
    if (c.g == 0) {
#pragma unroll
      for (int k = 0; k < DC_PPT; ++k) {
        L[k].init();
        R[k].init();
        lpm[k] = lsec[k] = lfar[k] = ninf;
      }
    }
#pragma unroll
    for (int j = 0; j < DC_DS; ++j) {
      const int d = c.g * DC_DS + j;
      if (d >= D) break;
      const T* buf = slot + (size_t)j * stage_elems;
      const int bshift = max(aend, w0 + d) - aend;  // columns >= aend sit at buf[col - w0 - bshift]
#pragma unroll
      for (int k = 0; k < DC_PPT; ++k) {
        const int p = threadIdx.x + k * blockDim.x, w = w0 + p;
        if (w < aend) {
          // d >= d* + 2 feeds the uniqueness maximum above d*, with the d* and the V at d - 1 of before the step
          const T v = buf[p];
          const int bd = L[k].bd;
          const T vm = L[k].prev;
          const bool nb = L[k].step(v, d);
          lfar[k] = nb ? ninf : (d - 2 >= bd ? fmax(lfar[k], v) : lfar[k]);
          lsec[k] = nb ? lpm[k] : lsec[k];
          lpm[k] = fmax(lpm[k], vm);
          const int col = w + d;  // right pixel x = w reads VR[d] = V[d, x + d]
          if (col < W) R[k].step(buf[col >= aend ? p + d - bshift : p + d], d);
        }
      }
    }

    if (c.g == ngroups - 1) {  // the chunk's walk is complete (CTA-uniform)
      const int64_t base = c.row * W;
#pragma unroll
      for (int k = 0; k < DC_PPT; ++k) {
        const int x = w0 + threadIdx.x + k * blockDim.x;
        if (x >= aend) break;
        if (lr_check) dr[x] = R[k].bd;
        wta_store<T>(disp_r, score_r, base + x, R[k].bd, R[k].best, R[k].cm, R[k].cp, min(D, W - x), subpixel);
      }
      if (lr_check) __syncthreads();  // dR* of every x < aend of this row is in dr
#pragma unroll
      for (int k = 0; k < DC_PPT; ++k) {
        const int w = w0 + threadIdx.x + k * blockDim.x;
        if (w >= aend) break;
        const int bd = L[k].bd;
        wta_store<T>(disp, score, base + w, bd, L[k].best, L[k].cm, L[k].cp, D, subpixel);
        if (valid) {
          const int x = w - bd;
          const bool lr = max_diff < 0 || (x >= 0 && abs(bd - dr[x]) <= max_diff);
          const bool far_empty = bd < 2 && bd + 2 > D - 1;
          const bool uq = uniqueness == 0.0 || far_empty ||
                          (double)L[k].best - (double)fmax(lsec[k], lfar[k]) >= uniqueness;
          valid[base + w] = lr && uq;
        }
      }
    }
    c.next(ngroups, nch, D, H, W);
  }
  __pipeline_wait_prior(0);
}

}  // namespace

template <typename T>
static int disparity_check_impl(const T* vol, T* disp, T* score, T* disp_r, T* score_r, uint8_t* valid, int64_t B, int64_t D,
                                int64_t H, int64_t W, int max_diff, double uniqueness, int subpixel, cudaStream_t st) {
  const char* op = "disparity_check";
  CTD_REQUIRE(B >= 0 && D >= 0 && H >= 0 && W >= 0, "%s: negative size", op);
  CTD_REQUIRE(D <= INT32_MAX && H <= INT32_MAX && W <= INT32_MAX, "%s: dimension too large", op);
  CTD_REQUIRE(std::isfinite(uniqueness) && uniqueness >= 0.0, "%s: uniqueness must be finite and >= 0, got %g", op,
              uniqueness);
  const int64_t npix = B * H * W;
  if (npix == 0) return CTD_OK;
  CTD_REQUIRE(D >= 1, "%s: the volume has no disparities (D = 0)", op);
  CTD_REQUIRE(vol, "%s: null pointer (vol)", op);
  const size_t nvol = (size_t)(npix * D) * sizeof(T), nmap = (size_t)npix * sizeof(T);
  const void* outs[5] = {disp, score, disp_r, score_r, valid};
  const size_t nout[5] = {nmap, nmap, nmap, nmap, (size_t)npix};
  for (int i = 0; i < 5; ++i) {
    CTD_REQUIRE(ranges_disjoint(outs[i], nout[i], vol, nvol), "%s: an output overlaps vol", op);
    for (int j = 0; j < i; ++j) CTD_REQUIRE(ranges_disjoint(outs[i], nout[i], outs[j], nout[j]), "%s: two outputs overlap", op);
  }
  if (!disp && !score && !disp_r && !score_r && !valid) return CTD_OK;

  // chunks of at most 1024 (fp32) or 512 (fp64) columns keep the ring within 128 KB of shared memory
  const int threads = (int)std::min<int64_t>(DC_MAXT * 4 / sizeof(T), std::max<int64_t>(32, 32 * cdiv(cdiv(W, DC_PPT), 32)));
  const int seg = DC_PPT * threads;
  const int stage_elems = (W > seg ? 2 : 1) * seg;
  const size_t smem = (size_t)DC_STAGES * DC_DS * stage_elems * sizeof(T);
  auto kernel = disparity_check_kernel<T>;
  const int rs = raise_smem_limit(kernel, smem, op);
  if (rs != CTD_OK) return rs;
  int dev = 0, sms = 0, per_sm = 0;
  CTD_CUDA(cudaGetDevice(&dev));
  CTD_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  CTD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
  if (per_sm < 1) return fail(CTD_ERR_CUDA, "%s: a %d-thread CTA with %zu bytes of shared memory does not fit", op, threads, smem);
  const int64_t grid = std::min<int64_t>(B * H, (int64_t)per_sm * sms);
  const bool lr_check = valid && max_diff >= 0;
  int* dr_rows = nullptr;
  if (lr_check) {
    dr_rows = static_cast<int*>(scratch_alloc((size_t)grid * W * sizeof(int), st));
    CTD_REQUIRE(dr_rows, "%s: no scratch memory for the right disparities (%zu bytes)", op, (size_t)grid * W * sizeof(int));
  }
  kernel<<<(unsigned)grid, threads, smem, st>>>(vol, disp, score, disp_r, score_r, valid, dr_rows, B, (int)D, (int)H, (int)W,
                                                stage_elems, max_diff, uniqueness, subpixel);
  count_launch();
  const int r = check_launch(op);
  if (dr_rows) scratch_free(dr_rows, st);
  return r;
}

}  // namespace ctd

CTD_API int ctd_disparity_check_f32(const float* vol, float* disp, float* score, float* disp_right, float* score_right,
                                    uint8_t* valid, int64_t B, int64_t D, int64_t H, int64_t W, int max_diff, double uniqueness,
                                    int subpixel, ctd_stream_t s) {
  return ctd::disparity_check_impl<float>(vol, disp, score, disp_right, score_right, valid, B, D, H, W, max_diff, uniqueness,
                                          subpixel, ctd::as_stream(s));
}
CTD_API int ctd_disparity_check_f64(const double* vol, double* disp, double* score, double* disp_right, double* score_right,
                                    uint8_t* valid, int64_t B, int64_t D, int64_t H, int64_t W, int max_diff, double uniqueness,
                                    int subpixel, ctd_stream_t s) {
  return ctd::disparity_check_impl<double>(vol, disp, score, disp_right, score_right, valid, B, D, H, W, max_diff,
                                           uniqueness, subpixel, ctd::as_stream(s));
}
