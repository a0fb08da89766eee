// PhotometricLoss census_mse / census_sad, block size 9, C = 1, fp32: pair-symmetric forward, backward and fused
// forward+backward(+masked sums) kernel for sm_100a.
//
// Reference semantics: torchext/ext/ext.h:201-266 (forward), :268-344 (backward); caller model/networks.py:376-377.
//
// With des = es[i] - es[q], dta = ta[i] - ta[q] and dd = des * rsqrt(des^2 + eps) - dta * rsqrt(dta^2 + eps)
// (= 2 (h(des) - h(dta)), h the soft step of ext.h:245) the soft census term of a pixel pair is antisymmetric,
// dd(q, i) = -dd(i, q).  For a pixel at least four pixels away from the image border every window tap is a distinct
// real pixel, so
//     out[i]     = s_f * sum_q psi(dd(i,q))                          psi = |.| (census_sad) or square (census_mse)
//     grad_in[i] = K   * sum_q phi(dd(i,q)) r1^3 (go[q] + go[i])     phi = sign or identity, K = eps / (2 * 81)
// over the 80 neighbours q of i, and the summand of (i,q) is the same number (forward) or the negated number
// (backward) as that of (q,i).  The gather kernels of photometric.cu evaluate every pair from both ends: 162
// MUFU.RSQ per pixel, which is what bounds them (XU pipe, 16 lanes/clk/SM).  Here every unordered pair is evaluated
// ONCE -- 80 reciprocal square roots per pixel -- and credited to both ends in registers:
//
//   * a warp owns a strip of 128 image rows, lane l rows 4l .. 4l+3, and walks along the columns.  At column c it
//     evaluates the pairs (i, q) with i = its four pixels of column c and q in columns c .. c+4 (offsets (0, 1..4) and
//     (1..4, -4..4): 40 per pixel).  The credit to i stays in the thread; so does the credit to a q in the thread's own
//     rows (a four-column ring of accumulators that shifts by one per step); credits to the four rows above / below
//     are summed per q and handed to the neighbouring lane with one shuffle per value and column.  Lanes 0 and 31 are
//     halo lanes (their pixels belong to the neighbouring strips, 120 useful rows per strip; for the first strip the
//     halo lane is the image's own border band).
//   * a CTA = 10 such warps on one (strip, column tile of up to 36 columns): the es / ta / grad_out tiles are staged
//     TRANSPOSED in shared memory (column-major, so a lane's 12 rows of a column are three conflict-free 128-bit
//     loads); warp w >= 1 walks the tile's columns 4(w-1) .. 4w-1, warp 0 the four columns in front of the tile (with
//     the offsets that reach into it: 2.25 columns' worth of pairs).  A warp's ring still holds the credits for the
//     four columns after its last one, which are exactly the next warp's: they are added to that warp's staged results
//     after a barrier ("carry").
//   * results are staged column-major in shared memory and written out row-major with 128-bit stores; the masked-mean
//     terms of the caller (networks.py:377) are accumulated on the way out.
//   * census_sad takes sign(dd).  A pair with |dd| < 3e-6 (the error bound of the MUFU path) flags both of its pixels
//     in a bitmap; after the walk the CTA recomputes those pixels' gradients from the staged tiles with the
//     reference's IEEE operation sequence (one warp per pixel), so every sign decision matches ext_cpu.
//   * the 4-pixel band along the image border, whose windows are replicate-clamped (a tap can hit the same pixel
//     several times), is computed by extra CTAs of the same launch with the direct gather from small shared-memory
//     tiles (3 % of a 480x640 image); they come first in the grid and share the SMs with the first tiles.
#include <algorithm>

#include "ctd_common.cuh"

namespace ctd {

extern int g_force_generic;
// ctd_set_option("census_sym", v): 0 = never (gather kernels of photometric.cu), 1 = every census entry point (tests, A/B
// runs), 2 (default) = where it is the faster kernel.  Measured on B200 (tools/experiments/census_sym_ab.py,
// profiles/r02_census_sym_ab.json), us per launch, this kernel / gather kernel:
//                            batch 2      batch 8       batch 64
//   forward                  40 / 33      82 / 103      585 / 680
//   census_mse backward      50 / 36     103 / 113      743 / 827
//   census_mse fused + sums  61 / 43     127 / 133      922 / 973
//   census_sad backward      55 / 40     119 / 128      816 / 931
//   census_sad fused + sums  69 / 48     152 / 146     1030 / 1066
// A tile holds an SM slot for ~50 us, so a call needs about two waves of tiles (2 x 296) before the halved MUFU count
// pays; the fused census_sad call (one more ALU instruction per pair and the near-tie pass) only wins on large batches.
int g_census_sym = 2;
int g_census_sym_noguard = 0;  // experiments only: never take the near-tie path (wrong signs at near-ties)
int g_census_sym_dbg = 0;  // experiments only (wrong results): 1 = no global loads in the staging, 2 = no stores in the write-out, 4 = no band CTAs, 8 = no masked sums
long long* g_census_sym_timeline = nullptr;  // experiments only: 16 x 8 int64 per CTA: per warp the globaltimer at start / staged / walked / exact done / end / walk end / carry end, smid

namespace {

constexpr int R9 = 4;
constexpr float INV81 = 1.0f / 81.0f;
constexpr int64_t CS_MIN_PIXELS = 1800000;             // automatic dispatch: about six 480x640 images (two waves of tiles)
// |error| of dd on the MUFU path: two rsqrt.approx (2^-22 relative each on a product of magnitude <= 1) and three
// roundings -- below 8e-7; 2e-6 leaves a factor of two
constexpr float SIGN_GUARD = 2e-6f;
#ifndef CTD_CS_NW
#define CTD_CS_NW 10
#endif
constexpr int CS_NW = CTD_CS_NW;         // warps per CTA: one for the run-in in front of the tile, the others for four columns each
constexpr int CS_ROWS = 128;             // tile rows: 32 lanes x 4
constexpr int CS_USE = 120;              // useful rows per strip (lanes 1..30)
constexpr int CS_PT = CS_ROWS + 8;       // tile pitch (floats): 4 zero rows, 128 rows, 4 zero rows
constexpr int CS_XC = 4 * (CS_NW - 1);   // output columns per tile (at most)
constexpr int CS_MINB = CS_NW >= 8 ? 2 : (CS_NW >= 6 ? 3 : 4);  // resident CTAs per SM the kernel is compiled for
constexpr int CS_TC = CS_XC + 8;         // tile columns: 4 in front (first warp's run-in), 4 behind
constexpr int CS_FLAGW = CS_ROWS / 32;   // bitmap words per tile column
constexpr size_t CS_SMEM = sizeof(float) * (3 * CS_TC * CS_PT + 2 * CS_XC * CS_ROWS) + sizeof(unsigned) * CS_TC * CS_FLAGW;

struct SymGeom {
  int H, W;
  int nstrips, nct;     // strips per image, column tiles per strip
  int ncol;             // interior columns (W - 8)
  int vec;              // 128-bit global accesses (W % 4 == 0, 16-byte aligned pointers): tiles start on a quad
  int ntiles;           // B * nstrips * nct
  int nbandcta;         // CTAs of the border band (they come first in the grid)
  int pf_stride;        // tiles resident at a time (2 per SM): tile t prefetches tile t + pf_stride into L2
};

__device__ __forceinline__ float or_sign(float mag, float s) {  // mag > 0 with the sign bit of s
  return __uint_as_float(__float_as_uint(mag) | (__float_as_uint(s) & 0x80000000u));
}
__device__ __forceinline__ float sgnf(float d) { return d < 0.f ? -1.f : (d > 0.f ? 1.f : 0.f); }

// one unordered pair: i = "centre" end, q = the other end.  fi/fq: forward sums, ai/aq: backward sums, nm: smallest |dd|
template <int TYPE, bool FWD, bool BWD>
__device__ __forceinline__ void pair_eval(float ei, float ti, float gi, float eq, float tq, float gq, float eps, float& fi,
                                          float& fq, float& ai, float& aq, float& nm) {
  const float des = ei - eq, dta = ti - tq;
  const float r1 = rsqrt_approx(fmaf(des, des, eps));
  const float r2 = rsqrt_approx(fmaf(dta, dta, eps));
  const float dd = fmaf(des, r1, -(dta * r2));
  if (FWD) {
    if (TYPE == 2) {
      fi = fmaf(dd, dd, fi);
      fq = fmaf(dd, dd, fq);
    } else {
      fi += fabsf(dd);
      fq += fabsf(dd);
    }
  }
  if (BWD) {
    const float r3 = r1 * r1 * r1;
    const float gs = gi + gq;
    if (TYPE == 2) {
      const float w = dd * r3;
      ai = fmaf(w, gs, ai);
      aq = fmaf(-w, gs, aq);
    } else {
      const float sr3 = or_sign(r3, dd);  // sign(dd) * r3; dd = +-0 and near-ties are redone by the exact pass
      ai = fmaf(sr3, gs, ai);
      aq = fmaf(-sr3, gs, aq);
      nm = fminf(nm, fabsf(dd));
    }
  }
}

__device__ __forceinline__ void ld4(float* d, const float* p) {
  const float4 v = *reinterpret_cast<const float4*>(p);
  d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
}

// Rare path: this lane saw |dd| < SIGN_GUARD among the pairs of (tile column x, offset column dx).  Find them again
// (same arithmetic), evaluate the two sign decisions of each with the reference's IEEE operation sequence (ext.h:321-330;
// the pair enters both pixels' sums in two roles, "tap" and "centre") and flag both pixels ONLY when a decision differs
// from the fast path's sign(dd) -- most near-ties agree, and an exact +-0 (sign 0 in the reference) never does.
// Tile rows live at index row + 4 of a column.
// The WHOLE warp works on the pairs of one lane (`owner`): 36 pairs (16 for dx = 0), at most two per lane, so the rescan
// is two short iterations instead of a serial chain of 36 that the other warps of the CTA wait for at the next barrier.
__device__ __forceinline__ void flag_near_ties(const float* __restrict__ E, const float* __restrict__ T, unsigned* flags, int x, int dx,
                                            int owner, int lane, float eps) {
  for (int p = lane; p < 36; p += 32) {
    const int k = p / 9, dy = p % 9 - R9;
    if (dx == 0 && dy < 1) continue;
    const int ri = 4 * owner + k, rq = ri + dy;
    if (rq < 0 || rq >= CS_ROWS) continue;
    const float des = E[x * CS_PT + 4 + ri] - E[(x + dx) * CS_PT + 4 + rq], dta = T[x * CS_PT + 4 + ri] - T[(x + dx) * CS_PT + 4 + rq];
    const float r1 = rsqrt_approx(fmaf(des, des, eps));
    const float r2 = rsqrt_approx(fmaf(dta, dta, eps));
    const float dd = fmaf(des, r1, -(dta * r2));
    if (fabsf(dd) < SIGN_GUARD) {
      const float q1 = __fdiv_rn(des, __fsqrt_rn(__fadd_rn(__fmul_rn(des, des), eps)));
      const float q2 = __fdiv_rn(dta, __fsqrt_rn(__fadd_rn(__fmul_rn(dta, dta), eps)));
      const float d_tap = __fsub_rn(0.5f * __fadd_rn(1.f, q1), 0.5f * __fadd_rn(1.f, q2));    // h(es_i - es_q) - h(ta_i - ta_q)
      const float d_ctr = __fsub_rn(0.5f * __fadd_rn(1.f, -q1), 0.5f * __fadd_rn(1.f, -q2));  // h(es_q - es_i) - h(ta_q - ta_i)
      const float sf = (__float_as_uint(dd) & 0x80000000u) ? -1.f : 1.f;                       // what or_sign() applied
      if (sgnf(d_tap) != sf || sgnf(d_ctr) != -sf) {
        atomicOr(&flags[x * CS_FLAGW + (ri >> 5)], 1u << (ri & 31));
        atomicOr(&flags[(x + dx) * CS_FLAGW + (rq >> 5)], 1u << (rq & 31));
      }
    }
  }
}

// census_sad gradient sum of the interior pixel at tile column tc, tile row r, with the reference's own IEEE operation
// sequence for the sign decisions (ext.h:321-330), both roles of the pixel; lane l takes taps l, l+32, l+64.
// Returns the un-scaled sum (grad_in = K * sum), like the walk's accumulators.
__device__ __forceinline__ float exact_sad_sum(const float* __restrict__ E, const float* __restrict__ T, const float* __restrict__ G,
                                               int tc, int r, float eps, int lane) {
  const float ei = E[tc * CS_PT + 4 + r], ti = T[tc * CS_PT + 4 + r], gc = G[tc * CS_PT + 4 + r];
  float acc = 0.f;
  for (int t = lane; t < 81; t += 32) {
    const int dy = t / 9 - R9, dx = t % 9 - R9;
    const int o = (tc + dx) * CS_PT + 4 + r + dy;
    const float des = ei - E[o], dta = ti - T[o], gq = G[o];
    const float s = __fadd_rn(__fmul_rn(des, des), eps);
    const float q1 = __fdiv_rn(des, __fsqrt_rn(s));
    const float q2 = __fdiv_rn(dta, __fsqrt_rn(__fadd_rn(__fmul_rn(dta, dta), eps)));
    // role "pixel is a tap of centre q": h(es[i] - es[q]) - h(ta[i] - ta[q])
    const float d_tap = __fsub_rn(0.5f * __fadd_rn(1.f, q1), 0.5f * __fadd_rn(1.f, q2));
    // role "pixel is the centre, q its tap": the differences flip sign exactly, so do the quotients
    const float d_ctr = __fsub_rn(0.5f * __fadd_rn(1.f, -q1), 0.5f * __fadd_rn(1.f, -q2));
    const float r1 = rsqrt_approx(s);
    acc = fmaf(r1 * r1 * r1, sgnf(d_tap) * gq - sgnf(d_ctr) * gc, acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  return acc;
}

// ---- the border band: direct gather with clamp multiplicities, from shared-memory tiles ---------------------------
// grad_in[i] = K * sum over the 81 window offsets of phi(dd(i,t)) r1^3 (go[i] + [p real] M(i,p) go[p]), t the clamped tap,
// p = i + offset unclamped, M(i,p) = how many offsets of p clamp onto i (1 unless i lies on the image border).
// A band CTA owns 256 band pixels -- 64 columns of the first / last four rows, or 64 rows of the first / last four columns
// -- and stages their halo (replicate-clamped es / ta, grad_out zero outside the image) in shared memory first: with one
// thread per pixel reading global memory the band was a chain of dependent loads that held an SM slot for 17-22 us.
constexpr int BD_LONG = 64, BD_SHORT = 4;

struct BandTile {
  int64_t n;
  int ox0, oy0, ow, oh;  // output region (may stick out of the image / the band at its far end)
  int ymin, ymax;        // rows of the region that belong to this part of the band: [ymin, ymax)
};

__device__ __forceinline__ BandTile band_tile(const SymGeom& g, int cta) {
  BandTile b;
  const int ntx = (g.W + BD_LONG - 1) / BD_LONG, nty = (g.H - 8 + BD_LONG - 1) / BD_LONG, per = 2 * ntx + 2 * nty;
  b.n = cta / per;
  int k = cta % per;
  if (k < 2 * ntx) {  // rows 0..3 and H-4..H-1
    b.ow = BD_LONG; b.oh = BD_SHORT;
    b.ox0 = (k % ntx) * BD_LONG;
    b.oy0 = k < ntx ? 0 : g.H - 4;
    b.ymin = b.oy0; b.ymax = b.oy0 + 4;
  } else {            // columns 0..3 and W-4..W-1 of the rows between
    k -= 2 * ntx;
    b.ow = BD_SHORT; b.oh = BD_LONG;
    b.ox0 = k < nty ? 0 : g.W - 4;
    b.oy0 = 4 + (k % nty) * BD_LONG;
    b.ymin = b.oy0; b.ymax = min(b.oy0 + BD_LONG, g.H - 4);
  }
  return b;
}

template <int TYPE, bool FWD, bool BWD, bool EXACT>
__device__ __forceinline__ void band_pixel_sums(const float* __restrict__ Eb, const float* __restrict__ Tb, const float* __restrict__ Gb, int pitch,
                                                int lx, int ly, int x, int y, int H, int W, float eps, float& facc, float& acc, float& near0) {
  const float ei = Eb[(ly + 4) * pitch + lx + 4], ti = Tb[(ly + 4) * pitch + lx + 4];
  const float gc = BWD ? Gb[(ly + 4) * pitch + lx + 4] : 0.f;
  facc = 0.f;
  acc = 0.f;
  near0 = 1.f;
  for (int dy = -R9; dy <= R9; ++dy) {
    const int py = y + dy, ty = clampi(py, 0, H - 1);
    const float my = y == 0 ? float(R9 + 1 - dy) : (y == H - 1 ? float(R9 + 1 + dy) : 1.f);
    const int ro = (ly + 4 + dy) * pitch + lx + 4;
#pragma unroll
    for (int dx = -R9; dx <= R9; ++dx) {
      const int px = x + dx, tx = clampi(px, 0, W - 1);
      const float des = ei - Eb[ro + dx], dta = ti - Tb[ro + dx];
      const bool self = ty == y && tx == x;
      float gq = 0.f;  // grad_out of p = i + offset (zero in the tile when p is not a real pixel) times M(i,p)
      if (BWD) {
        const float mx = x == 0 ? float(R9 + 1 - dx) : (x == W - 1 ? float(R9 + 1 + dx) : 1.f);
        gq = (mx * my) * Gb[ro + dx];
      }
      if (!EXACT) {
        const float r1 = rsqrt_approx(fmaf(des, des, eps));
        const float r2 = rsqrt_approx(fmaf(dta, dta, eps));
        const float dd = fmaf(des, r1, -(dta * r2));
        if (FWD) facc = TYPE == 2 ? fmaf(dd, dd, facc) : facc + fabsf(dd);
        if (BWD) {
          const float r3 = r1 * r1 * r1;
          acc = fmaf((TYPE == 2 ? dd : sgnf(dd)) * r3, gq + gc, acc);
          if (TYPE == 3 && !self) near0 = fminf(near0, fabsf(dd));
        }
      } else {  // census_sad backward with the reference's IEEE sequence; the two roles are evaluated separately
        const float s = __fadd_rn(__fmul_rn(des, des), eps);
        const float q1 = __fdiv_rn(des, __fsqrt_rn(s));
        const float q2 = __fdiv_rn(dta, __fsqrt_rn(__fadd_rn(__fmul_rn(dta, dta), eps)));
        const float d_tap = __fsub_rn(0.5f * __fadd_rn(1.f, q1), 0.5f * __fadd_rn(1.f, q2));
        const float d_ctr = __fsub_rn(0.5f * __fadd_rn(1.f, -q1), 0.5f * __fadd_rn(1.f, -q2));
        const float r1 = rsqrt_approx(s);
        acc = fmaf(r1 * r1 * r1, sgnf(d_tap) * gq - sgnf(d_ctr) * gc, acc);
      }
    }
  }
}

template <int TYPE, bool FWD, bool BWD>
__device__ __forceinline__ void band_block(float* __restrict__ sm, const float* __restrict__ es, const float* __restrict__ ta,
                                           const float* __restrict__ go, float* __restrict__ out, float* __restrict__ gi,
                                           const float* __restrict__ mask, const SymGeom& g, float eps, int cta, int tid, float& mnum,
                                           float& mden) {
  const BandTile b = band_tile(g, cta);
  const int H = g.H, W = g.W;
  const int64_t plane = (int64_t)H * W;
  const float* ep = es + b.n * plane;
  const float* tp = ta + b.n * plane;
  const float* gp = BWD ? go + b.n * plane : nullptr;
  const int pitch = b.ow + 8, rows = b.oh + 8, nel = pitch * rows;  // 72 x 12 or 12 x 72
  float* Eb = sm;
  float* Tb = Eb + 864;
  float* Gb = Tb + 864;
  for (int i = tid; i < nel; i += CS_NW * 32) {
    const int r = i / pitch, c = i % pitch;
    const int uy = b.oy0 - 4 + r, ux = b.ox0 - 4 + c;
    const int64_t o = (int64_t)clampi(uy, 0, H - 1) * W + clampi(ux, 0, W - 1);
    Eb[i] = __ldg(ep + o);
    Tb[i] = __ldg(tp + o);
    if (BWD) Gb[i] = (uy >= 0 && uy < H && ux >= 0 && ux < W) ? __ldg(gp + o) : 0.f;
  }
  __syncthreads();
  if (tid >= BD_LONG * BD_SHORT) return;
  const int lx = tid % b.ow, ly = tid / b.ow;
  const int x = b.ox0 + lx, y = b.oy0 + ly;
  if (x >= W || y < b.ymin || y >= b.ymax) return;
  float facc, acc, near0;
  band_pixel_sums<TYPE, FWD, BWD, false>(Eb, Tb, Gb, pitch, lx, ly, x, y, H, W, eps, facc, acc, near0);
  if (BWD && TYPE == 3 && near0 < SIGN_GUARD) {
    float f2, n2;
    band_pixel_sums<TYPE, false, true, true>(Eb, Tb, Gb, pitch, lx, ly, x, y, H, W, eps, f2, acc, n2);
  }
  const int64_t o = b.n * plane + (int64_t)y * W + x;
  if (FWD) {
    const float v = facc * ((TYPE == 2 ? 0.25f : 0.5f) * INV81);
    out[o] = v;
    if (mask != nullptr) {
      const float m = __ldg(mask + o);
      mnum = fmaf(m, v, mnum);
      mden += m;
    }
  }
  if (BWD) gi[o] = acc * (0.5f * eps * INV81);
}

// ---- the interior: strips x column tiles ---------------------------------------------------------------------------
__device__ __forceinline__ int tile_col0(const SymGeom& g, int t) {  // first interior column of column tile t (t = nct: end)
  if (g.vec) return 4 + 4 * (int)((int64_t)t * (g.ncol / 4) / g.nct);
  return 4 + (int)((int64_t)t * g.ncol / g.nct);
}

template <int TYPE, bool FWD, bool BWD>
__global__ void __launch_bounds__(CS_NW * 32, CS_MINB)
census_sym_kernel(const float* __restrict__ es, const float* __restrict__ ta, const float* __restrict__ go, float* __restrict__ out,
                  float* __restrict__ gi, const float* __restrict__ mask, const SymGeom g, float eps, float guard, double* __restrict__ partials,
                  unsigned* __restrict__ ticket, float* __restrict__ sums2, long long* __restrict__ timeline, int dbg) {
  extern __shared__ __align__(16) float smem[];
  float* E = smem;
  float* T = E + CS_TC * CS_PT;
  float* G = T + CS_TC * CS_PT;
  float* SO = G + CS_TC * CS_PT;        // staged forward sums  [column][row]
  float* SG = SO + CS_XC * CS_ROWS;     // staged backward sums [column][row]
  unsigned* flags = reinterpret_cast<unsigned*>(SG + CS_XC * CS_ROWS);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  float mnum = 0.f, mden = 0.f;
  auto stamp = [&](int k) {  // experiments only (timeline == nullptr in production): per warp, 8 slots; slot 7 = smid
    if (timeline != nullptr && lane == 0) {
      long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      long long* p = timeline + ((int64_t)blockIdx.x * 16 + wid) * 8;
      if (k == 0) {
        unsigned sm;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
        p[7] = sm;
      }
      p[k] = t;
    }
  };
  stamp(0);

  // The border band's CTAs come FIRST in the grid: one thread per band pixel is a long chain of dependent loads that
  // uses little of an SM, so it should share the SMs with the first tiles instead of running alone at the end of the
  // launch (measured: the band as the last CTAs extended a 120 us launch by 20 us).
  if ((int)blockIdx.x < g.nbandcta) {  // block-uniform
    band_block<TYPE, FWD, BWD>(smem, es, ta, go, out, gi, mask, g, eps, (int)blockIdx.x, tid, mnum, mden);
    if (FWD && mask != nullptr && !(dbg & 8)) finish_masked_sums((double)mnum, (double)mden, partials, ticket, sums2);
    stamp(4);
    return;
  }

  const int H = g.H, W = g.W;
  const int tile = blockIdx.x - g.nbandcta;
  const int ct = tile % g.nct, strip = (tile / g.nct) % g.nstrips;
  const int64_t n = tile / (g.nct * g.nstrips);
  const int c0 = tile_col0(g, ct), c1 = tile_col0(g, ct + 1), ncols = c1 - c0;  // output columns [c0, c1)
  const int R0 = strip * CS_USE;
  const int64_t plane = (int64_t)H * W;
  const float* ep = es + n * plane;
  const float* tp = ta + n * plane;
  const float* gp = BWD ? go + n * plane : nullptr;

  // ---- stage the tiles transposed: tile column j = image column c0 - 4 + j, tile row r = image row R0 + r
  {
    const int tcols = ncols + 8;
    // Tile rows below the image (R0 + r >= H, last strip only) get synthetic values instead of copies of the last row:
    // es rises and ta falls with the row and the column, so every pair that involves such a row has |dd| ~ 2 and never
    // looks like a near-tie -- 16 dy + 1000 dx != 0 for every offset (copies of one row would make dd = 0 for each of their pairs and send the warp to the slow
    // flagging path at every step); their grad_out is 0 and nothing is ever stored for them.
    if (g.vec) {
      // all of a thread's loads are issued before the first shared-memory store: one global round trip per tile
      constexpr int NIT = (CS_ROWS * (CS_TC / 4) + CS_NW * 32 - 1) / (CS_NW * 32);
      const int nitems = CS_ROWS * (tcols / 4);
      float4 ve[NIT], vt[NIT], vg[NIT];
#pragma unroll
      for (int it = 0; it < NIT; ++it) {
        const int idx = tid + it * (CS_NW * 32), r = idx % CS_ROWS, q = idx / CS_ROWS, y = R0 + r;
        if (idx < nitems && y < H && !(dbg & 1)) {
          const int64_t o = (int64_t)y * W + (c0 - 4 + 4 * q);
          ve[it] = ldg4(ep + o);
          vt[it] = ldg4(tp + o);
          if (BWD) vg[it] = ldg4(gp + o);
        }
      }
#pragma unroll
      for (int it = 0; it < NIT; ++it) {
        const int idx = tid + it * (CS_NW * 32), r = idx % CS_ROWS, q = idx / CS_ROWS, y = R0 + r;
        if (idx >= nitems) continue;
        float* de = E + (4 * q) * CS_PT + 4 + r;
        float* dt = T + (4 * q) * CS_PT + 4 + r;
        float* dg = G + (4 * q) * CS_PT + 4 + r;
        if (y < H && !(dbg & 1)) {
          de[0] = ve[it].x; de[CS_PT] = ve[it].y; de[2 * CS_PT] = ve[it].z; de[3 * CS_PT] = ve[it].w;
          dt[0] = vt[it].x; dt[CS_PT] = vt[it].y; dt[2 * CS_PT] = vt[it].z; dt[3 * CS_PT] = vt[it].w;
          if (BWD) {
            dg[0] = vg[it].x; dg[CS_PT] = vg[it].y; dg[2 * CS_PT] = vg[it].z; dg[3 * CS_PT] = vg[it].w;
          }
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float f = (float)(16 * y + 1000 * (4 * q + k));
            de[k * CS_PT] = f;
            dt[k * CS_PT] = -f;
            dg[k * CS_PT] = 0.f;
          }
        }
      }
    } else {
      for (int idx = tid; idx < CS_ROWS * tcols; idx += CS_NW * 32) {
        const int r = idx % CS_ROWS, j = idx / CS_ROWS, y = R0 + r;
        if (y < H) {
          const int64_t o = (int64_t)y * W + (c0 - 4 + j);
          E[j * CS_PT + 4 + r] = __ldg(ep + o);
          T[j * CS_PT + 4 + r] = __ldg(tp + o);
          if (BWD) G[j * CS_PT + 4 + r] = __ldg(gp + o);
        } else {
          const float f = (float)(16 * y + 1000 * j);
          E[j * CS_PT + 4 + r] = f;
          T[j * CS_PT + 4 + r] = -f;
          G[j * CS_PT + 4 + r] = 0.f;
        }
      }
    }
    for (int idx = tid; idx < 8 * tcols; idx += CS_NW * 32) {  // the rows above lane 0's and below lane 31's: finite values
      const int j = idx >> 3, k = idx & 7, o = j * CS_PT + (k < 4 ? k : CS_ROWS + k);
      E[o] = 0.f;
      T[o] = 0.f;
      G[o] = 0.f;
    }
    for (int idx = tid; idx < CS_TC * CS_FLAGW; idx += CS_NW * 32) flags[idx] = 0u;
  }
  __syncthreads();
  stamp(1);
  // The tiles of the next wave start with a 20 MB burst from DRAM (every SM stages two tiles at once) while this wave
  // uses no DRAM bandwidth at all during its walk: ask L2 for the tile that runs pf_stride tiles later.
  if (tile + g.pf_stride < g.ntiles) {
    const int t2 = tile + g.pf_stride;
    const int ct2 = t2 % g.nct, strip2 = (t2 / g.nct) % g.nstrips;
    const int64_t n2 = t2 / (g.nct * g.nstrips);
    const int a0 = tile_col0(g, ct2) - 4, a1 = tile_col0(g, ct2 + 1) + 4;   // columns [a0, a1)
    const int lines = ((a1 - a0) * 4 + 127) / 128 + 1;                       // 128-byte lines per row (unaligned start)
    const int rows2 = min(CS_ROWS, H - strip2 * CS_USE);
    for (int i = tid; i < rows2 * lines; i += CS_NW * 32) {
      const int r = i / lines, l = i % lines;
      const int64_t o = n2 * plane + (int64_t)(strip2 * CS_USE + r) * W + min(a0 + 32 * l, W - 1);
      asm volatile("prefetch.global.L2 [%0];" ::"l"(es + o));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(ta + o));
      if (BWD) asm volatile("prefetch.global.L2 [%0];" ::"l"(go + o));
    }
  }

  // ---- roles: slot x = tile column x = output column x - 4.  Warp 0 walks the run-in (slots 0..3: only the offsets that
  // reach columns >= c0, 2.25 columns' worth of pairs); warp w >= 1 walks the four output columns 4(w-1) .. 4w-1.
  int xb = 4 * wid, xe = min(4 * wid + 4, ncols + 4);
  if (wid == 0) xb = 0, xe = 4;
  if (xe < xb) xe = xb;

  float fI[4] = {0.f, 0.f, 0.f, 0.f}, aI[4] = {0.f, 0.f, 0.f, 0.f};  // sums of the pixels of the current column
  float fQ[4][4], aQ[4][4];                                            // ... of the next four columns (own rows)
#pragma unroll
  for (int d = 0; d < 4; ++d)
#pragma unroll
    for (int k = 0; k < 4; ++k) fQ[d][k] = aQ[d][k] = 0.f;
  const unsigned FULL = 0xffffffffu;
  float nmk[4] = {1.f, 1.f, 1.f, 1.f};  // smallest |dd| among the pairs of the current offset column, per own row (four
                                        // independent min chains: one chain through all 36 pairs serialises them)
  unsigned hit = 0u;  // bit dx: this lane saw a near-tie among the pairs of offset column dx of the current step

#pragma unroll 1
  for (int x = xb; x < xe; ++x) {
    const int dx0 = x < 4 ? 4 - x : 0;  // smallest column offset that matters (warp-uniform)
    float ei[4], ti[4], gI[4];
    {
      const float* c = E + x * CS_PT + 4 + 4 * lane;
      ld4(ei, c);
      ld4(ti, c + (T - E));
      if (BWD) ld4(gI, c + (G - E));
      else gI[0] = gI[1] = gI[2] = gI[3] = 0.f;
    }
    if (dx0 == 0) {  // same column: the four rows below each pixel
#pragma unroll
      for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int rq = k + 1; rq < 4; ++rq)
          pair_eval<TYPE, FWD, BWD>(ei[k], ti[k], gI[k], ei[rq], ti[rq], gI[rq], eps, fI[k], fI[rq], aI[k], aI[rq], nmk[k]);
      float e1[4], t1[4], g1[4];
      const float* c = E + x * CS_PT + 8 + 4 * lane;
      ld4(e1, c);
      ld4(t1, c + (T - E));
      if (BWD) ld4(g1, c + (G - E));
      else g1[0] = g1[1] = g1[2] = g1[3] = 0.f;
      float lf[4] = {0.f, 0.f, 0.f, 0.f}, la[4] = {0.f, 0.f, 0.f, 0.f};  // credits to the next lane's rows
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int j = 0; j <= k; ++j)  // row 4 lane + 4 + j: offset 4 + j - k in 1..4
          pair_eval<TYPE, FWD, BWD>(ei[k], ti[k], gI[k], e1[j], t1[j], g1[j], eps, fI[k], lf[j], aI[k], la[j], nmk[k]);
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        if (FWD) fI[m] += __shfl_up_sync(FULL, lf[m], 1);
        if (BWD) aI[m] += __shfl_up_sync(FULL, la[m], 1);
      }
      if (BWD && TYPE == 3) {
        hit |= fminf(fminf(nmk[0], nmk[1]), fminf(nmk[2], nmk[3])) < guard ? 1u : 0u;
        nmk[0] = nmk[1] = nmk[2] = nmk[3] = 1.f;
      }
    }
    // The four offset columns run through ONE copy of the pair code (an unrolled copy per column is 53 KB of
    // instructions and the warps stall on instruction fetch): the ring of accumulators is rotated by one column after
    // each, so the column being credited is always slot 0, and after four rotations the ring is back in place.  The 12
    // rows of the partner column are taken four at a time (the lane above's, the lane's own, the lane below's), which
    // keeps 12 instead of 36 partner values and 8 instead of 16 hand-over sums live.
#pragma unroll 1
    for (int dx = 1; dx <= 4; ++dx) {
      if (dx >= dx0) {
        const float* c = E + (x + dx) * CS_PT + 4 * lane;  // rows 4 lane - 4 .. 4 lane + 7
        float eq[4], tq[4], gq[4];
        {  // rows of the lane above: offsets j - k - 4 >= -4
          ld4(eq, c);
          ld4(tq, c + (T - E));
          if (BWD) ld4(gq, c + (G - E));
          else gq[0] = gq[1] = gq[2] = gq[3] = 0.f;
          float lf[4] = {0.f, 0.f, 0.f, 0.f}, la[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int j = k; j < 4; ++j)
              pair_eval<TYPE, FWD, BWD>(ei[k], ti[k], gI[k], eq[j], tq[j], gq[j], eps, fI[k], lf[j], aI[k], la[j], nmk[k]);
#pragma unroll
          for (int m = 0; m < 4; ++m) {
            if (FWD) fQ[0][m] += __shfl_down_sync(FULL, lf[m], 1);
            if (BWD) aQ[0][m] += __shfl_down_sync(FULL, la[m], 1);
          }
        }
        {  // the lane's own rows: offsets -3 .. 3
          ld4(eq, c + 4);
          ld4(tq, c + (T - E) + 4);
          if (BWD) ld4(gq, c + (G - E) + 4);
#pragma unroll
          for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int j = 0; j < 4; ++j)
              pair_eval<TYPE, FWD, BWD>(ei[k], ti[k], gI[k], eq[j], tq[j], gq[j], eps, fI[k], fQ[0][j], aI[k], aQ[0][j], nmk[k]);
        }
        {  // rows of the lane below: offsets 4 + j - k <= 4
          ld4(eq, c + 8);
          ld4(tq, c + (T - E) + 8);
          if (BWD) ld4(gq, c + (G - E) + 8);
          float lf[4] = {0.f, 0.f, 0.f, 0.f}, la[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int k = 0; k < 4; ++k)
#pragma unroll
            for (int j = 0; j <= k; ++j)
              pair_eval<TYPE, FWD, BWD>(ei[k], ti[k], gI[k], eq[j], tq[j], gq[j], eps, fI[k], lf[j], aI[k], la[j], nmk[k]);
#pragma unroll
          for (int m = 0; m < 4; ++m) {
            if (FWD) fQ[0][m] += __shfl_up_sync(FULL, lf[m], 1);
            if (BWD) aQ[0][m] += __shfl_up_sync(FULL, la[m], 1);
          }
        }
        if (BWD && TYPE == 3) {
          hit |= fminf(fminf(nmk[0], nmk[1]), fminf(nmk[2], nmk[3])) < guard ? 1u << dx : 0u;
          nmk[0] = nmk[1] = nmk[2] = nmk[3] = 1.f;
        }
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {  // rotate the ring: next column to slot 0
        const float f0 = fQ[0][k], a0 = aQ[0][k];
        fQ[0][k] = fQ[1][k]; fQ[1][k] = fQ[2][k]; fQ[2][k] = fQ[3][k]; fQ[3][k] = f0;
        aQ[0][k] = aQ[1][k]; aQ[1][k] = aQ[2][k]; aQ[2][k] = aQ[3][k]; aQ[3][k] = a0;
      }
    }
    if (BWD && TYPE == 3) {  // one vote per step; only the offset columns with a near-tie are scanned again
      unsigned owners = __ballot_sync(FULL, hit != 0u);
      while (owners) {  // warp-uniform loop over the lanes that saw a near-tie
        const int owner = __ffs(owners) - 1;
        owners &= owners - 1;
        const unsigned h = __shfl_sync(FULL, hit, owner);
#pragma unroll 1
        for (int dx = 0; dx <= 4; ++dx)
          if (h >> dx & 1u) flag_near_ties(E, T, flags, x, dx, owner, lane, eps);
      }
      hit = 0u;
    }
    if (x >= 4) {  // column x - 4 of the tile's outputs has met all the neighbours this warp walks over
      if (FWD) *reinterpret_cast<float4*>(SO + (x - 4) * CS_ROWS + 4 * lane) = make_float4(fI[0], fI[1], fI[2], fI[3]);
      if (BWD) *reinterpret_cast<float4*>(SG + (x - 4) * CS_ROWS + 4 * lane) = make_float4(aI[0], aI[1], aI[2], aI[3]);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      fI[k] = fQ[0][k]; fQ[0][k] = fQ[1][k]; fQ[1][k] = fQ[2][k]; fQ[2][k] = fQ[3][k]; fQ[3][k] = 0.f;
      aI[k] = aQ[0][k]; aQ[0][k] = aQ[1][k]; aQ[1][k] = aQ[2][k]; aQ[2][k] = aQ[3][k]; aQ[3][k] = 0.f;
    }
  }
  stamp(5);
  __syncthreads();
  stamp(2);
  // ---- carry: the ring holds this warp's credits for slots xe .. xe+3 -- the next warp's columns, staged without them
  if (xe > xb) {
#pragma unroll
    for (int d = 0; d < 4; ++d) {
      const int col = xe + d - 4;
      if (col >= 0 && col < ncols) {
        float4* po = reinterpret_cast<float4*>(SO + col * CS_ROWS + 4 * lane);
        float4* pg = reinterpret_cast<float4*>(SG + col * CS_ROWS + 4 * lane);
        const float* f = d == 0 ? fI : fQ[d == 0 ? 0 : d - 1];
        const float* a = d == 0 ? aI : aQ[d == 0 ? 0 : d - 1];
        if (FWD) {
          float4 v = *po;
          v.x += f[0]; v.y += f[1]; v.z += f[2]; v.w += f[3];
          *po = v;
        }
        if (BWD) {
          float4 v = *pg;
          v.x += a[0]; v.y += a[1]; v.z += a[2]; v.w += a[3];
          *pg = v;
        }
      }
    }
  }
  stamp(6);
  __syncthreads();
  // ---- exact pass over the flagged output pixels (census_sad gradient only)
  if (BWD && TYPE == 3) {
    for (int w = wid; w < ncols * CS_FLAGW; w += CS_NW) {
      const int col = w / CS_FLAGW, word = w % CS_FLAGW;
      unsigned bits = flags[(col + 4) * CS_FLAGW + word];
      while (bits) {
        const int b = __ffs(bits) - 1;
        bits &= bits - 1;
        const int r = 32 * word + b;
        if (r < 4 || r >= CS_ROWS - 4 || R0 + r >= H - 4) continue;  // halo lanes, rows of the border band
        const float v = exact_sad_sum(E, T, G, col + 4, r, eps, lane);
        if (lane == 0) SG[col * CS_ROWS + r] = v;
      }
    }
    __syncthreads();
  }
  stamp(3);
  // ---- write out row-major; the caller's masked-mean terms on the way
  {
    const float sf = (TYPE == 2 ? 0.25f : 0.5f) * INV81, sb = 0.5f * eps * INV81;
    float* outp = FWD ? out + n * plane : nullptr;
    float* gip = BWD ? gi + n * plane : nullptr;
    const float* mp = (FWD && mask != nullptr) ? mask + n * plane : nullptr;
    if (g.vec) {
      const int nq = ncols / 4;
      for (int item = wid; item < 4 * nq; item += CS_NW) {
        const int rg = item / nq, q = item % nq, r = 32 * rg + lane, y = R0 + r;
        if (r < 4 || r >= CS_ROWS - 4 || y >= H - 4) continue;
        const int64_t o = (int64_t)y * W + c0 + 4 * q;
        if (FWD) {
          const float* s = SO + (4 * q) * CS_ROWS + r;
          const float4 v = make_float4(s[0] * sf, s[CS_ROWS] * sf, s[2 * CS_ROWS] * sf, s[3 * CS_ROWS] * sf);
          if (!(dbg & 2)) *reinterpret_cast<float4*>(outp + o) = v;
          if (mp != nullptr) {
            const float4 m = ldg4(mp + o);
            mnum = fmaf(m.x, v.x, fmaf(m.y, v.y, fmaf(m.z, v.z, fmaf(m.w, v.w, mnum))));
            mden += (m.x + m.y) + (m.z + m.w);
          }
        }
        if (BWD) {
          const float* s = SG + (4 * q) * CS_ROWS + r;
          if (!(dbg & 2)) *reinterpret_cast<float4*>(gip + o) = make_float4(s[0] * sb, s[CS_ROWS] * sb, s[2 * CS_ROWS] * sb, s[3 * CS_ROWS] * sb);
        }
      }
    } else {
      for (int item = wid; item < 4 * ncols; item += CS_NW) {
        const int rg = item / ncols, col = item % ncols, r = 32 * rg + lane, y = R0 + r;
        if (r < 4 || r >= CS_ROWS - 4 || y >= H - 4) continue;
        const int64_t o = (int64_t)y * W + c0 + col;
        if (FWD) {
          const float v = SO[col * CS_ROWS + r] * sf;
          outp[o] = v;
          if (mp != nullptr) {
            const float m = __ldg(mp + o);
            mnum = fmaf(m, v, mnum);
            mden += m;
          }
        }
        if (BWD) gip[o] = SG[col * CS_ROWS + r] * sb;
      }
    }
  }
  if (FWD && mask != nullptr && !(dbg & 8)) finish_masked_sums((double)mnum, (double)mden, partials, ticket, sums2);  // block-uniform
  stamp(4);
}

static int sm_count_cs() {
  int dev = 0, v = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
  return v > 0 ? v : 148;
}

template <int TYPE, bool FWD, bool BWD>
static bool launch_variant(const float* es, const float* ta, const float* go, float* out, float* gi, const float* mask,
                           const SymGeom& g, float eps, unsigned grid, MsSlot& ms, float* sums2, cudaStream_t st) {
  auto kernel = census_sym_kernel<TYPE, FWD, BWD>;
  // two CTAs per SM need the largest shared-memory carve-out (2 x 107 KB); the default heuristic may pick a smaller one
  if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CS_SMEM) != cudaSuccess ||
      cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  kernel<<<grid, CS_NW * 32, CS_SMEM, st>>>(es, ta, go, out, gi, mask, g, eps, g_census_sym_noguard ? 0.f : SIGN_GUARD, ms.partials, ms.ticket, sums2, g_census_sym_timeline, g_census_sym_dbg);
  return true;
}

}  // namespace

// Forward (out != nullptr), backward (gi != nullptr, needs go) or both in one launch; with `mask` (forward required) also
// sums2 = (sum(mask * out), sum(mask)).  Returns false when this path does not take the call (nothing launched).
bool census_sym_launch(const float* es, const float* ta, const float* go, float* out, float* gi, const float* mask, float* sums2,
                       int64_t B, int64_t C, int64_t H, int64_t W, int type, float eps, cudaStream_t st) {
  if (g_census_sym == 2) {
    const int64_t px = B * H * W;
    // forward + backward in one call: the tile kernel with packed fp32 taps wins at every size measured (DESIGN §4.2)
    if (px < CS_MIN_PIXELS || (out != nullptr && gi != nullptr)) return false;
  }
  if (!g_census_sym || g_force_generic || C != 1 || B < 1 || H < 16 || W < 16 || H * W >= (int64_t)1 << 30 || (type != 2 && type != 3)) return false;
  if (!out && !gi) return false;
  if (gi && !go) return false;
  if (mask && (!out || !sums2)) return false;
  SymGeom g;
  g.H = (int)H;
  g.W = (int)W;
  g.ncol = (int)W - 8;
  uintptr_t al = reinterpret_cast<uintptr_t>(es) | reinterpret_cast<uintptr_t>(ta) | reinterpret_cast<uintptr_t>(go) |
                 reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(gi) | reinterpret_cast<uintptr_t>(mask);
  g.vec = (W % 4 == 0) && (al & 15) == 0;
  g.nstrips = (int)cdiv(H - 8, CS_USE);
  g.nct = g.vec ? (int)cdiv(g.ncol / 4, CS_XC / 4) : (int)cdiv(g.ncol, CS_XC);
  const int64_t ntiles = B * g.nstrips * g.nct;
  const int64_t nbandcta = (g_census_sym_dbg & 4) ? 0 : B * (2 * cdiv(W, BD_LONG) + 2 * cdiv(H - 8, BD_LONG));
  g.pf_stride = 2 * sm_count_cs();
  if (ntiles + nbandcta > (int64_t)INT32_MAX) return false;
  g.ntiles = (int)ntiles;
  g.nbandcta = (int)nbandcta;
  const unsigned grid = (unsigned)(ntiles + nbandcta);
  MsSlot ms = {nullptr, nullptr, nullptr};
  if (mask && !ms_acquire(grid, st, &ms)) return false;
  bool ok;
  if (type == 2) {
    if (out && gi) ok = launch_variant<2, true, true>(es, ta, go, out, gi, mask, g, eps, grid, ms, sums2, st);
    else if (out) ok = launch_variant<2, true, false>(es, ta, go, out, gi, mask, g, eps, grid, ms, sums2, st);
    else ok = launch_variant<2, false, true>(es, ta, go, out, gi, mask, g, eps, grid, ms, sums2, st);
  } else {
    if (out && gi) ok = launch_variant<3, true, true>(es, ta, go, out, gi, mask, g, eps, grid, ms, sums2, st);
    else if (out) ok = launch_variant<3, true, false>(es, ta, go, out, gi, mask, g, eps, grid, ms, sums2, st);
    else ok = launch_variant<3, false, true>(es, ta, go, out, gi, mask, g, eps, grid, ms, sums2, st);
  }
  ms_release(&ms, st);
  if (ok) count_launch();
  return ok;
}

}  // namespace ctd

// experiments only: per-CTA timestamps of the next census_sym launches go to `buf` (device memory, 128 int64 per CTA); NULL = off
CTD_API void ctd_debug_census_timeline(long long* buf) { ctd::g_census_sym_timeline = buf; }
