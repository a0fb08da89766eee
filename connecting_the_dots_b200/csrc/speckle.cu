// Speckle filter of a disparity map (ctd_speckle_filter_*) for sm_100a: union-find connected-component labelling under a
// disparity-difference rule (Playne & Hawick 2018; the block-based union-find of Allegretti et al.).
//
// Definition (include/ctd_b200.h states it in full): two 4-neighbours of one image are adjacent when both are valid and
// |(double)disp[p] - (double)disp[q]| <= max_diff; valid_out = valid && the size of the pixel's connected component under
// that adjacency > max_size.  Components and their sizes do not depend on how they are found, so every output is bit-equal
// to the definition.
//
// Labels are image-local int32 pixel indices, -1 for an invalid pixel.  A parent is always below its child, so the root of
// a tree is the smallest index of its component.  Four launches, whatever the sizes:
//   1. speckle_tiles: a CTA stages a 32x32 tile of disp and valid in shared memory and evaluates each pixel's right and
//      down adjacency once.  Row runs come from a warp ballot of the right bits; down pairs are united in shared memory
//      (atomicMin), one union per stretch of pairs the previous pair does not already cover.  Every pixel's tile root
//      goes to scratch as its label and, at each tile root, the tile-local size (0 elsewhere).
//   2. speckle_merge: a warp per tile border re-evaluates its pixel pairs and unites the two trees of each pair the previous
//      lane's pair does not cover, in global memory (atomicMin on the larger root, retried until it links a root; finds
//      halve their paths).
//   3. speckle_sizes: each tile root finds its global root, adds its tile-local size there (integer atomicAdd) and stores
//      the global root as its label.  Only global roots are written then, so walks that pass a tile root finish at once.
//   4. speckle_mark: valid_out[p] = labels[p] >= 0 && sizes[labels[labels[p]]] > max_size (two hops: pixel -> tile root
//      -> global root).
// Labels and sizes (8 B/px) come from the library's stream-ordered scratch pool; no host synchronisation, integer atomics
// only, 64-bit indexing over the batch: every call is capture-safe and deterministic.
#include <algorithm>
#include <cmath>

#include "ctd_common.cuh"

namespace ctd {

namespace {

constexpr int SP_T = 32;                     // tile edge: a tile row is one warp
constexpr int SP_THREADS = 256;              // 8 warps; a thread owns SP_T * SP_T / SP_THREADS = 4 pixels of a tile
constexpr int SP_ROWS = SP_THREADS / SP_T;   // rows between a thread's pixels

template <typename T>
__device__ __forceinline__ bool sp_adjacent(T a, T b, double max_diff) {
  return fabs((double)a - (double)b) <= max_diff;  // false for NaN
}

// Root of x.  Path halving: each visited node is pointed at its grandparent, an ancestor of it below its parent.
__device__ __forceinline__ int sp_find(volatile int* L, int x) {
  for (;;) {
    const int p = L[x];
    if (p == x) return x;
    const int g = L[p];
    if (g == p) return p;
    L[x] = g;
    x = g;
  }
}

// Join the trees of a and b: link the larger root under the smaller one.  The atomicMin succeeds only while its target
// is still a root; otherwise the value it met is an ancestor of that target and the loop continues from there.
__device__ __forceinline__ void sp_unite(int* L, int a, int b) {
  for (;;) {
    a = sp_find(L, a);
    b = sp_find(L, b);
    if (a == b) return;
    if (a > b) {
      const int t = a;
      a = b;
      b = t;
    }
    const int old = atomicMin(L + b, a);
    if (old == b) return;
    b = old;
  }
}

// Grids are 2-D: blockIdx.y strides over the images, blockIdx.x over the tiles or pixels of one image, so indices inside
// an image are int32 and the image offset b * H * W is the only 64-bit product.
#define SP_FOR_IMAGES(b) for (int64_t b = blockIdx.y; b < B; b += gridDim.y)

template <typename T>
__global__ void __launch_bounds__(SP_THREADS)
speckle_tiles(const T* __restrict__ disp, const uint8_t* __restrict__ valid, int* __restrict__ labels,
              int* __restrict__ sizes, int64_t B, int H, int W, int ntx, int nty, double max_diff) {
  __shared__ T sd[SP_T * SP_T];
  __shared__ bool sv[SP_T * SP_T];
  __shared__ int lab[SP_T * SP_T], cnt[SP_T * SP_T];
  __shared__ unsigned rjoin[SP_T];  // bit l of row r: pixel (r, l) is adjacent to (r, l + 1)
  const int tx = threadIdx.x % SP_T, ty0 = threadIdx.x / SP_T;
  const int64_t plane = (int64_t)H * W;
  SP_FOR_IMAGES(b) {
    for (int t = blockIdx.x; t < ntx * nty; t += gridDim.x) {
      const int h0 = t / ntx * SP_T, w0 = t % ntx * SP_T, w = w0 + tx;
#pragma unroll
      for (int k = 0; k < SP_T / SP_ROWS; ++k) {
        const int ty = ty0 + k * SP_ROWS, i = ty * SP_T + tx, h = h0 + ty;
        const bool in = h < H && w < W;
        const int64_t g = b * plane + (int64_t)h * W + w;
        sd[i] = in ? disp[g] : T(0);
        sv[i] = in && (!valid || valid[g]);
        cnt[i] = 0;
      }
      __syncthreads();
      // row runs: a warp holds one tile row, and each pixel's label starts as the first pixel of its run of right-joined
      // pixels (no atomics)
#pragma unroll
      for (int k = 0; k < SP_T / SP_ROWS; ++k) {
        const int ty = ty0 + k * SP_ROWS, i = ty * SP_T + tx;
        const bool right = tx + 1 < SP_T && sv[i] && sv[i + 1] && sp_adjacent(sd[i], sd[i + 1], max_diff);
        const unsigned joins = __ballot_sync(0xffffffffu, right);
        const unsigned breaks = ~joins & ((1u << tx) - 1);  // pixels left of tx that do not join their right neighbour
        lab[i] = ty * SP_T + (breaks ? 32 - __clz(breaks) : 0);
        if (tx == 0) rjoin[ty] = joins;
      }
      __syncthreads();
      // down pairs: one union per stretch of down-joined pairs whose upper and lower pixels are both right-joined to the
      // previous pair's (the previous pair's union already covers them)
#pragma unroll
      for (int k = 0; k < SP_T / SP_ROWS; ++k) {
        const int ty = ty0 + k * SP_ROWS, i = ty * SP_T + tx;
        const bool down = ty + 1 < SP_T && sv[i] && sv[i + SP_T] && sp_adjacent(sd[i], sd[i + SP_T], max_diff);
        const unsigned downs = __ballot_sync(0xffffffffu, down);
        const bool covered = tx > 0 && (downs >> (tx - 1) & rjoin[ty] >> (tx - 1) & rjoin[ty + 1 < SP_T ? ty + 1 : ty] >> (tx - 1) & 1u);
        if (down && !covered) sp_unite(lab, i, i + SP_T);
      }
      __syncthreads();
      int root[SP_T / SP_ROWS];
#pragma unroll
      for (int k = 0; k < SP_T / SP_ROWS; ++k) {
        const int i = (ty0 + k * SP_ROWS) * SP_T + tx;
        root[k] = sp_find(lab, i);
        if (sv[i]) atomicAdd(cnt + root[k], 1);
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < SP_T / SP_ROWS; ++k) {
        const int ty = ty0 + k * SP_ROWS, i = ty * SP_T + tx, h = h0 + ty;
        if (h >= H || w >= W) continue;
        const int64_t g = b * plane + (int64_t)h * W + w;
        const int r = root[k];
        labels[g] = sv[i] ? (h0 + r / SP_T) * W + w0 + r % SP_T : -1;
        sizes[g] = sv[i] && r == i ? cnt[i] : 0;
      }
      __syncthreads();  // shared memory is restaged for the next tile
    }
  }
}

// A warp takes one border of a tile: lanes e % 64 < 32 the pairs across its right border (rows h0 + lane), the others the
// pairs across its bottom border (columns w0 + lane).  A pair is united unless the previous lane's pair is adjacent and
// both of its pixels are adjacent to this pair's (then that union already joins them).
template <typename T>
__global__ void __launch_bounds__(SP_THREADS)
speckle_merge(const T* __restrict__ disp, const uint8_t* __restrict__ valid, int* labels, int64_t B, int H, int W,
              int ntx, int nty, double max_diff) {
  const int64_t plane = (int64_t)H * W;
  const int64_t n = (int64_t)ntx * nty * 2 * SP_T;
  const int lane = threadIdx.x % SP_T;
  SP_FOR_IMAGES(b) {
    const T* dimg = disp + b * plane;
    const uint8_t* vimg = valid ? valid + b * plane : nullptr;
    for (int64_t e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {  // warp-uniform trips
      const int t = (int)(e / (2 * SP_T));
      const bool across = e % (2 * SP_T) < SP_T;
      const int h0 = t / ntx * SP_T, w0 = t % ntx * SP_T;
      const int h = across ? h0 + lane : h0 + SP_T - 1, w = across ? w0 + SP_T - 1 : w0 + lane;
      const bool in = h < H && w < W && (across ? w + 1 < W : h + 1 < H);
      const int p = h * W + w, q = across ? p + 1 : p + W;
      const bool vp = in && (!vimg || vimg[p]), vq = in && (!vimg || vimg[q]);
      const T dp = vp ? dimg[p] : T(0), dq = vq ? dimg[q] : T(0);
      const bool pair = vp && vq && sp_adjacent(dp, dq, max_diff);
      const bool prev_pair = __shfl_up_sync(0xffffffffu, pair, 1);
      const bool prev_vp = __shfl_up_sync(0xffffffffu, vp, 1), prev_vq = __shfl_up_sync(0xffffffffu, vq, 1);
      const T prev_dp = __shfl_up_sync(0xffffffffu, dp, 1), prev_dq = __shfl_up_sync(0xffffffffu, dq, 1);
      const bool covered = lane > 0 && prev_pair && prev_vp && prev_vq && sp_adjacent(prev_dp, dp, max_diff) &&
                           sp_adjacent(prev_dq, dq, max_diff);
      if (pair && !covered) sp_unite(labels + b * plane, p, q);
    }
  }
}

__global__ void __launch_bounds__(SP_THREADS)
speckle_sizes(int* labels, int* sizes, int64_t B, int plane) {
  SP_FOR_IMAGES(b) {
    volatile int* L = labels + b * plane;
    int* S = sizes + b * plane;
    for (int64_t i = blockIdx.x * blockDim.x + threadIdx.x; i < plane; i += gridDim.x * blockDim.x) {
      const int s = S[i];
      if (s == 0) continue;  // not a tile root
      int r = (int)i;
      for (int up = L[r]; up != r; up = L[r]) r = up;
      if (r != i) {
        atomicAdd(S + r, s);
        L[i] = r;
      }
    }
  }
}

__global__ void __launch_bounds__(SP_THREADS)
speckle_mark(const int* __restrict__ labels, const int* __restrict__ sizes, uint8_t* __restrict__ valid_out, int64_t B,
             int plane, int64_t max_size) {
  SP_FOR_IMAGES(b) {
    const int* L = labels + b * plane;
    for (int64_t i = blockIdx.x * blockDim.x + threadIdx.x; i < plane; i += gridDim.x * blockDim.x) {
      const int q = L[i];
      valid_out[b * plane + i] = q >= 0 && sizes[b * plane + L[q]] > max_size;
    }
  }
}

}  // namespace

template <typename T>
static int speckle_impl(const T* disp, const uint8_t* valid, uint8_t* valid_out, int64_t B, int64_t H, int64_t W,
                        int64_t max_size, double max_diff, cudaStream_t st) {
  const char* op = "speckle_filter";
  CTD_REQUIRE(B >= 0 && H >= 0 && W >= 0, "%s: negative size", op);
  CTD_REQUIRE(W == 0 || H <= INT32_MAX / W, "%s: an image has more than INT32_MAX pixels (H = %lld, W = %lld)", op,
              (long long)H, (long long)W);
  const int64_t plane = H * W;
  CTD_REQUIRE(plane == 0 || B <= INT64_MAX / 8 / plane, "%s: batch too large", op);
  CTD_REQUIRE(max_size >= 0, "%s: max_size must be >= 0, got %lld", op, (long long)max_size);
  CTD_REQUIRE(std::isfinite(max_diff) && max_diff >= 0.0, "%s: max_diff must be finite and >= 0, got %g", op, max_diff);
  const int64_t npix = B * plane;
  if (npix == 0) return CTD_OK;
  CTD_REQUIRE(disp, "%s: null pointer (disp)", op);
  CTD_REQUIRE(ranges_disjoint(valid_out, (size_t)npix, disp, (size_t)npix * sizeof(T)), "%s: valid_out overlaps disp", op);
  CTD_REQUIRE(ranges_disjoint(valid_out, (size_t)npix, valid, (size_t)npix), "%s: valid_out overlaps valid", op);
  if (!valid_out) return CTD_OK;

  int dev = 0, sms = 0;
  CTD_CUDA(cudaGetDevice(&dev));
  CTD_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int ntx = (int)cdiv(W, SP_T), nty = (int)cdiv(H, SP_T);
  // one wave of full occupancy (8 CTAs of 256 threads per SM), images across y; the kernels stride past it
  const int64_t cap = (int64_t)sms * (2048 / SP_THREADS);
  const unsigned gy = (unsigned)std::min<int64_t>(B, 65535);
  auto grid = [&](int64_t blocks_per_image) {
    return dim3((unsigned)std::max<int64_t>(1, std::min(blocks_per_image, cap / gy)), gy);
  };

  int* labels = static_cast<int*>(scratch_alloc((size_t)npix * 2 * sizeof(int), st));
  CTD_REQUIRE(labels, "%s: no scratch memory for labels and sizes (%zu bytes)", op, (size_t)npix * 2 * sizeof(int));
  int* sizes = labels + npix;
  speckle_tiles<T><<<grid((int64_t)ntx * nty), SP_THREADS, 0, st>>>(disp, valid, labels, sizes, B, (int)H, (int)W, ntx, nty,
                                                                     max_diff);
  speckle_merge<T><<<grid(cdiv((int64_t)ntx * nty * 2 * SP_T, SP_THREADS)), SP_THREADS, 0, st>>>(
      disp, valid, labels, B, (int)H, (int)W, ntx, nty, max_diff);
  speckle_sizes<<<grid(cdiv(plane, SP_THREADS)), SP_THREADS, 0, st>>>(labels, sizes, B, (int)plane);
  speckle_mark<<<grid(cdiv(plane, SP_THREADS)), SP_THREADS, 0, st>>>(labels, sizes, valid_out, B, (int)plane, max_size);
  count_launch(4);
  const int r = check_launch(op);
  scratch_free(labels, st);
  return r;
}

}  // namespace ctd

CTD_API int ctd_speckle_filter_f32(const float* disp, const uint8_t* valid, uint8_t* valid_out, int64_t B, int64_t H,
                                   int64_t W, int64_t max_size, double max_diff, ctd_stream_t s) {
  return ctd::speckle_impl<float>(disp, valid, valid_out, B, H, W, max_size, max_diff, ctd::as_stream(s));
}
CTD_API int ctd_speckle_filter_f64(const double* disp, const uint8_t* valid, uint8_t* valid_out, int64_t B, int64_t H,
                                   int64_t W, int64_t max_size, double max_diff, ctd_stream_t s) {
  return ctd::speckle_impl<double>(disp, valid, valid_out, B, H, W, max_size, max_diff, ctd::as_stream(s));
}
