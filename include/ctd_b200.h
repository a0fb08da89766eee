/*
 * ctd_b200.h -- C ABI of libctd_b200.so, the B200 (sm_100a) implementation of the
 * per-pixel custom ops of "Connecting the Dots" (reference: torchext/ext/).
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  Each entry
 * point names the reference interface it replaces (paths relative to the reference
 * repository).  Two families:
 *
 *   ctd_<op>_<dtype>(..., stream)      DEVICE pointers; asynchronous launch on `stream`
 *                                      (cudaStream_t; NULL = legacy default stream);
 *                                      what ext_cuda.cpp's *_cuda / photometric_loss_*
 *                                      functions would call instead of ext_kernel.cu.
 *   ctd_host_<op>_<dtype>(...)         HOST pointers (pageable or pinned); copies in,
 *                                      runs the same kernels, copies out, returns when the
 *                                      result is in host memory; what ext_cpu.cpp's *_cpu
 *                                      functions would call instead of iterate_cpu.
 *
 * Every function returns CTD_OK (0) or a CTD_ERR_* code and never terminates the process
 * (the reference's CUDA_CHECK calls exit(-1), common_cuda.h:11-20).  ctd_last_error()
 * returns a thread-local message for the last failure.  There is no CPU fallback: without
 * a CUDA device every compute entry point returns CTD_ERR_CUDA.
 *
 * Layouts are the reference's: contiguous row-major, es/ta/grad [B,C,H,W], out [B,1,H,W],
 * xyz [B,H,W,3], K [3,3], cost volume [D,H,W] per image.  Index outputs are int64,
 * CrossCheck masks are uint8 (ext_cpu.cpp:31,50,76).
 */
#ifndef CTD_B200_H
#define CTD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* ctd_stream_t; /* a cudaStream_t */

enum {
  CTD_OK = 0,
  CTD_ERR_INVALID = 1, /* bad argument (shape, type id, null pointer) */
  CTD_ERR_CUDA = 2,    /* CUDA runtime error, message in ctd_last_error() */
  CTD_ERR_NOMEM = 3    /* workspace allocation failed */
};

/* loss type ids, torchext/ext/ext.h:196-199 */
enum { CTD_LOSS_MSE = 0, CTD_LOSS_SAD = 1, CTD_LOSS_CENSUS_MSE = 2, CTD_LOSS_CENSUS_SAD = 3 };

const char* ctd_last_error(void);
/* library version and the SM architecture the kernels were compiled for ("sm_100a") */
const char* ctd_version(void);
/* number of kernel launches issued by this library in the calling process so far */
uint64_t ctd_launch_count(void);
/* test/tuning switches: "force_generic" = 1 routes every op through its generic kernel */
int ctd_set_option(const char* name, int value);

/* ---- PhotometricLossForward: ext.h:201-266, ext_cuda.cpp:92-104 (photometric_loss_forward) */
int ctd_photometric_fwd_f32(const float* es, const float* ta, float* out, int64_t B, int64_t C,
                            int64_t H, int64_t W, int block_size, int type, float eps,
                            ctd_stream_t stream);
int ctd_photometric_fwd_f64(const double* es, const double* ta, double* out, int64_t B, int64_t C,
                            int64_t H, int64_t W, int block_size, int type, float eps,
                            ctd_stream_t stream);
/* ---- PhotometricLossBackward: ext.h:268-344, ext_cuda.cpp:109-123 (photometric_loss_backward).
 * grad_in [B,C,H,W] is fully overwritten (no zero-initialisation needed, no atomics). */
int ctd_photometric_bwd_f32(const float* es, const float* ta, const float* grad_out, float* grad_in,
                            int64_t B, int64_t C, int64_t H, int64_t W, int block_size, int type,
                            float eps, ctd_stream_t stream);
int ctd_photometric_bwd_f64(const double* es, const double* ta, const double* grad_out,
                            double* grad_in, int64_t B, int64_t C, int64_t H, int64_t W,
                            int block_size, int type, float eps, ctd_stream_t stream);

/* ---- forward + backward in one call (ext.h:201-344), for callers whose grad_out does not depend on the loss
 * map -- the reference's only caller builds it from the mask alone (model/networks.py:377).  The census modes
 * run a single fused kernel (the backward's window terms already contain the forward's); results are identical
 * to calling ctd_photometric_fwd_f32 then ctd_photometric_bwd_f32. */
int ctd_photometric_fwd_bwd_f32(const float* es, const float* ta, const float* grad_out, float* out,
                                float* grad_in, int64_t B, int64_t C, int64_t H, int64_t W, int block_size,
                                int type, float eps, ctd_stream_t stream);

/* The same plus the caller's masked-mean terms (model/networks.py:377) from the same pass:
 * sums2[0] = sum(mask * out), sums2[1] = sum(mask), deterministic.  mask [B,1,H,W]. */
int ctd_photometric_fwd_bwd_masked_f32(const float* es, const float* ta, const float* grad_out, const float* mask,
                                       float* out, float* grad_in, float* sums2, int64_t B, int64_t C, int64_t H,
                                       int64_t W, int block_size, int type, float eps, ctd_stream_t stream);

/* ---- SSIM photometric loss (an addition: the reference has no SSIM op).  Same window as the photometric loss:
 * taps (clamp(h + i - bs/2), clamp(w + j - bs/2)), i, j in [0, bs), N = bs^2; with x = es, y = ta and population
 * statistics over the window, S = (2 mx my + c1)(2 vxy + c2) / ((mx^2 + my^2 + c1)(vxx + vyy + c2)) and
 * out[n,0,h,w] = sum_c (1 - S_c) / 2.  c1 > 0 and c2 > 0 (usual values 0.01^2, 0.03^2).  The backward is the gradient
 * w.r.t. es for grad_out [B,1,H,W]; grad_in [B,C,H,W] is fully overwritten, no atomics. */
int ctd_ssim_fwd_f32(const float* es, const float* ta, float* out, int64_t B, int64_t C, int64_t H, int64_t W,
                     int block_size, double c1, double c2, ctd_stream_t stream);
int ctd_ssim_fwd_f64(const double* es, const double* ta, double* out, int64_t B, int64_t C, int64_t H, int64_t W,
                     int block_size, double c1, double c2, ctd_stream_t stream);
int ctd_ssim_bwd_f32(const float* es, const float* ta, const float* grad_out, float* grad_in, int64_t B, int64_t C,
                     int64_t H, int64_t W, int block_size, double c1, double c2, ctd_stream_t stream);
int ctd_ssim_bwd_f64(const double* es, const double* ta, const double* grad_out, double* grad_in, int64_t B, int64_t C,
                     int64_t H, int64_t W, int block_size, double c1, double c2, ctd_stream_t stream);
/* forward + backward + sums2 = (sum(mask * out), sum(mask)) in one pass (one kernel for odd block sizes 3..11),
 * deterministic; mask [B,1,H,W] */
int ctd_ssim_fwd_bwd_masked_f32(const float* es, const float* ta, const float* grad_out, const float* mask, float* out,
                                float* grad_in, float* sums2, int64_t B, int64_t C, int64_t H, int64_t W,
                                int block_size, double c1, double c2, ctd_stream_t stream);

/* ---- the disparity warp in front of the loss: model/networks.py:362-371 (RectifiedPatternSimilarityLoss.tforward),
 * grid_sample(pattern, grid(disp), bilinear, padding_mode='border', align_corners=False) with the reference's (W-1)
 * grid normalisation.  pattern [Bp,1,Hp,Wp] (Bp = 1 or B), disp [B,1,H,W] -> out [B,1,H,W]; backward: gradient
 * w.r.t. disp (the pattern is a constant of the model). */
int ctd_warp_pattern_fwd_f32(const float* pattern, const float* disp, float* out, int64_t B, int64_t Bp, int64_t Hp,
                             int64_t Wp, int64_t H, int64_t W, ctd_stream_t stream);
int ctd_warp_pattern_bwd_f32(const float* pattern, const float* disp, const float* grad_out, float* grad_disp,
                             int64_t B, int64_t Bp, int64_t Hp, int64_t Wp, int64_t H, int64_t W, ctd_stream_t stream);

/* ---- geometric loss of the stage-2 trainer, one direction: model/networks.py:474-498
 * (ProjectionDepthSimilarityLoss.fwd over ProjectionBaseLoss.unproject/transform/project, networks.py:436-472).
 * depthA, depthB [B,1,H,W]; ray [H*W,3] (the module's uv @ Ki^T table); K [3,3]; RA, RB [B,3,3]; tA, tB [B,3];
 * all DEVICE pointers.  sums2[0] = sum |d - grid_sample(depthB)| (clamped to [0, clamp] when clamp > 0),
 * sums2[1] = B*H*W, deterministic.  Gradients of sums2[0] * scale: grad_depthA [B,1,H,W] is written
 * (direct_accumulate = 0) or added to (1); grad_depthB receives the bilinear scatter by atomicAdd and must be
 * initialised by the caller.  Either gradient pointer may be NULL. */
int ctd_depth_similarity_f32(const float* depthA, const float* depthB, const float* ray, const float* K,
                             const float* RA, const float* tA, const float* RB, const float* tB,
                             float* grad_depthA, float* grad_depthB, float* sums2, int64_t B, int64_t H, int64_t W,
                             float clamp, float scale, int direct_accumulate, ctd_stream_t stream);

/* ---- disparity (smoothness / edge) loss of the stage-1 trainer: model/networks.py:380-412 (DisparityLoss.tforward)
 * over the 5x5 Sobel filter with replicate padding (networks.py:537-565).  disp, edge, grad_disp, grad_edge
 * [B,1,H,W], DEVICE pointers; edge may be NULL (the reference's edge=None branch: mean of the clamped gradient
 * magnitude).  sums2[0] = sum of the per-pixel loss, sums2[1] = B*H*W, deterministic; the gradients are those of
 * sums2[0] * scale, fully overwritten, no atomics.  grad_disp / grad_edge may be NULL. */
int ctd_disparity_loss_f32(const float* disp, const float* edge, float* grad_disp, float* grad_edge, float* sums2,
                           int64_t B, int64_t H, int64_t W, float scale, ctd_stream_t stream);

/* ---- XCorrVolFunctor: ext.h:120-191, ext_cuda.cpp:73-86 (xcorrvol_cuda).  The reference has no
 * batch dimension; here in0,in1 are [B,C,H,W] and out is [B,D,H,W] (B=1 is the reference call). */
int ctd_xcorrvol_f32(const float* in0, const float* in1, float* out, int64_t B, int64_t C, int64_t H,
                     int64_t W, int64_t n_disps, int block_size, ctd_stream_t stream);
int ctd_xcorrvol_f64(const double* in0, const double* in1, double* out, int64_t B, int64_t C,
                     int64_t H, int64_t W, int64_t n_disps, int block_size, ctd_stream_t stream);

/* ---- block-matching disparity from the XCorrVol cost volume (an addition: the reference has no consumer of the volume),
 * without writing the volume.  With V[b,d,h,w] what ctd_xcorrvol_* writes for the same arguments (n_disps = D):
 *   d*[b,h,w]        = the first d in [0, D) with V[b,d,h,w] = max_d V[b,d,h,w] (ties -> smallest d; +0.0 == -0.0),
 *   score[b,0,h,w]   = V[b,d*,h,w], the peak normalised cross-correlation (a confidence),
 *   disp[b,0,h,w]    = d* (subpixel = 0), or d* + delta (subpixel = 1) with c-, c0, c+ the scores at d*-1, d*, d*+1,
 *                      den = c- - 2 c0 + c+, delta = (c- - c+) / (2 den) clamped to [-0.5, 0.5]; delta = 0 when d* = 0,
 *                      d* = D-1 or den >= 0.
 * disp and score [B,1,H,W], DEVICE pointers; score may be NULL.  n_disps >= 1 unless B*H*W = 0 (then CTD_OK, nothing runs).
 * The integer disparity and the score equal the argmax and the maximum of the volume ctd_xcorrvol_* computes for the same
 * inputs with the default options: fp32, C = 1, block 3/5/7/9 run one fused pass over the separable kernel's outputs
 * (workspace grows with B*H*W, not B*D*H*W); every other case, and force_generic, runs a generic kernel, the exact argmax
 * of the generic volume.  Not mirrored: the A/B options xcorr_direct and xcorr_nofix (the disparity always uses the
 * separable kernel with its fix-up), and images that one separable launch cannot take even alone (H > 1048560, more than
 * 65535 chunks of 16 disparities, or H * (16 ceil(D/16) + 4 ceil(W/4)) >= 2^31 window-statistics positions), where the
 * volume falls back to its direct or generic kernel and the disparity to the generic one -- equal to within the volume's
 * 1e-5 there, not bit for bit.  The batch size alone never leaves the separable path: both ops cut a batch into launches
 * of as many images as one launch takes.  In the fused path the sub-pixel scores are re-evaluated
 * in the centred form, within ~1e-5 of the volume's.  The inputs must be finite: for non-finite inputs the
 * result is unspecified (the call does not fault). */
int ctd_xcorr_disparity_f32(const float* in0, const float* in1, float* disp, float* score, int64_t B, int64_t C, int64_t H,
                            int64_t W, int64_t n_disps, int block_size, int subpixel, ctd_stream_t stream);
int ctd_xcorr_disparity_f64(const double* in0, const double* in1, double* disp, double* score, int64_t B, int64_t C, int64_t H,
                            int64_t W, int64_t n_disps, int block_size, int subpixel, ctd_stream_t stream);

/* ---- semi-global matching over a score volume (an addition: Hirschmueller, PAMI 2008).  vol [B,D,H,W], higher is better
 * (the convention of ctd_xcorrvol_*; pass a cost volume negated).  p1, p2 are converted once to the volume's dtype.  For
 * each path direction r = (dy, dx) and q = p - r:
 *   L_r(p, d) = V(p, d)                    if q is outside the image (a path starts there),
 *   L_r(p, d) = V(p, d) + (m - M)          otherwise, with M = max_k L_r(q, k) and
 *               m = max(L_r(q, d), L_r(q, d-1) - p1, L_r(q, d+1) - p1, M - p2), leaving out neighbours outside [0, D).
 * Path order: paths = 4: (0,+1) (0,-1) (+1,0) (-1,0); paths = 8: those, then (+1,+1) (+1,-1) (-1,+1) (-1,-1).
 *   agg[b,d,h,w]   = A = (((L_0 + L_1) + L_2) + ...), summed in that order (required, caller-owned, must not overlap vol),
 *   disp, score    = the winner-take-all of A exactly as ctd_xcorr_disparity_* states it for a volume (first maximum, score
 *                    A at d*, optional fp64 three-point sub-pixel offset), [B,1,H,W]; each may be NULL.
 * Every value is bit-equal to that definition (no multiplies, max is exact).  CTD_ERR_INVALID for paths other than 4 or
 * 8, non-finite penalties, p1 < 0, p2 < p1, D < 1 (unless B*H*W = 0: then CTD_OK and nothing runs), D > 1024, agg
 * overlapping vol.  DEVICE pointers; no scratch memory, no atomics, capture-safe.  The inputs must be finite: for
 * non-finite inputs the result is unspecified (the call does not fault). */
int ctd_sgm_f32(const float* vol, float* agg, float* disp, float* score, int64_t B, int64_t D, int64_t H, int64_t W,
                double p1, double p2, int paths, int subpixel, ctd_stream_t stream);
int ctd_sgm_f64(const double* vol, double* agg, double* disp, double* score, int64_t B, int64_t D, int64_t H, int64_t W,
                double p1, double p2, int paths, int subpixel, ctd_stream_t stream);

/* ---- census-transform stereo matching (an addition: Zabih & Woodfill 1994).  in0, in1 [B,C,H,W].  The window is
 * (wh, ww), both odd, 2 <= wh*ww <= 65; rh = wh/2, rw = ww/2.  block_size = bs is odd, 1 <= bs <= 15; r = bs/2.
 *   1. Census transform.  T[b,c,h,w] is a uint64.  Number the window taps (i, j), i in [0,wh), j in [0,ww), row-major,
 *      skipping the centre (rh, rw).  Bit k, for the k-th tap, is
 *      x[b,c,clamp(h+i-rh,0,H-1),clamp(w+j-rw,0,W-1)] < x[b,c,h,w].  Bits from wh*ww - 1 up are 0.  The comparison is
 *      IEEE <, so a NaN on either side gives 0: non-finite input is defined.
 *   2. Per-pixel Hamming cost.  Hm[b,d,h,w] = sum_c popcount(T0[b,c,h,w] XOR T1[b,c,h,clamp(w-d,0,W-1)]).
 *   3. Aggregated cost.  S[b,d,h,w] = sum_{i,j in [0,bs)} Hm[b,d,clamp(h+i-r,0,H-1),clamp(w+j-r,0,W-1)] (a
 *      replicate-padded box filter of the bs = 1 volume).
 *   4. Score volume.  V = -S in the input's dtype: higher is better, the convention of ctd_xcorrvol_* and ctd_sgm_*.  |V|
 *      <= C*(wh*ww-1)*bs^2, and calls where that bound exceeds 2^24 are rejected, so fp32 holds every value exactly.
 *   5. Disparity.  (disp, score) = the winner-take-all of V as ctd_xcorr_disparity_* states it for a volume: the first
 *      maximum of V (the smallest d among equal least costs), score = V at d*, and the optional fp64 three-point
 *      sub-pixel offset, computed from the same integers, so the fused result is bit-equal to that of the volume.
 * ctd_census_transform_* writes T (out [B,C,H,W] uint64).  ctd_census_vol_* writes V (out [B,n_disps,H,W]).
 * ctd_census_disparity_* writes disp [B,1,H,W] and score [B,1,H,W] (score may be NULL) without writing V.
 * CTD_ERR_INVALID, checked before any device work, for: an even or non-positive window side, wh*ww < 2 or > 65; an even
 * block_size or one outside 1..15; the 2^24 bound; negative sizes; null pointers; n_disps < 1 when B*H*W > 0; an
 * output that overlaps an input (or disp overlapping score).  B*H*W = 0 (B*C*H*W = 0 for the transform) is CTD_OK with
 * nothing launched.  DEVICE pointers; descriptor scratch (2*B*C*H*W*8 bytes) comes from the library's stream-ordered
 * pool; no atomics, no host synchronisation, capture-safe; 64-bit indexing.  One kernel path per entry point:
 * "force_generic" does not apply. */
int ctd_census_transform_f32(const float* in, uint64_t* out, int64_t B, int64_t C, int64_t H, int64_t W, int wh, int ww,
                             ctd_stream_t stream);
int ctd_census_transform_f64(const double* in, uint64_t* out, int64_t B, int64_t C, int64_t H, int64_t W, int wh, int ww,
                             ctd_stream_t stream);
int ctd_census_vol_f32(const float* in0, const float* in1, float* out, int64_t B, int64_t C, int64_t H, int64_t W,
                       int64_t n_disps, int wh, int ww, int block_size, ctd_stream_t stream);
int ctd_census_vol_f64(const double* in0, const double* in1, double* out, int64_t B, int64_t C, int64_t H, int64_t W,
                       int64_t n_disps, int wh, int ww, int block_size, ctd_stream_t stream);
int ctd_census_disparity_f32(const float* in0, const float* in1, float* disp, float* score, int64_t B, int64_t C, int64_t H,
                             int64_t W, int64_t n_disps, int wh, int ww, int block_size, int subpixel, ctd_stream_t stream);
int ctd_census_disparity_f64(const double* in0, const double* in1, double* disp, double* score, int64_t B, int64_t C,
                             int64_t H, int64_t W, int64_t n_disps, int wh, int ww, int block_size, int subpixel,
                             ctd_stream_t stream);

/* ---- left-right consistency and uniqueness checks over a score volume (an addition: the post-processing of Hirschmueller's
 * SGM and of OpenCV's StereoSGBM).  vol [B,D,H,W], higher is better (the convention of ctd_xcorrvol_*, ctd_census_vol_*
 * and ctd_sgm_*); V[b,d,h,w] scores left pixel w against right pixel w - d.
 *   1. Left view.  disp, score = the winner-take-all of V exactly as ctd_xcorr_disparity_* states it for a volume: d*L =
 *      the first d with the largest V, score = V at d*L, optional fp64 three-point sub-pixel offset.
 *   2. Right view.  For right pixel x, Dx = min(D, W - x) and VR[d,h,x] = V[d,h,x+d], d < Dx (the diagonal x + d <= W - 1:
 *      never the clamped columns a volume holds for d > w).  dR* = the first d in [0, Dx) with the largest VR,
 *      score_right = VR at dR*, disp_right = dR* plus the same offset with c-, c+ = V[dR*-1, h, x+dR*-1],
 *      V[dR*+1, h, x+dR*+1]; the offset is 0 when dR* = 0, dR* = Dx - 1 or den >= 0.
 *   3. valid[b,0,h,w] = 1 when both hold, else 0:
 *      LR:          max_diff < 0 (check off), or x = w - d*L >= 0 and |d*L - dR*(x)| <= max_diff (integer indices);
 *      uniqueness:  uniqueness == 0 (check off), or {d : |d - d*L| >= 2} is empty, or
 *                   (double)V[d*L] - (double)second >= uniqueness, second = the maximum of V over that set.
 * Only maxima, compares and those fp64 operations are involved, so every output is bit-equal to the definition.  Outputs
 * [B,1,H,W] (valid as uint8), DEVICE pointers, each may be NULL.  CTD_ERR_INVALID, checked before any device work, for:
 * negative sizes; a negative or non-finite uniqueness; D < 1 when B*H*W > 0; a null vol; an output overlapping vol or
 * another output.  B*H*W = 0 is CTD_OK with nothing launched.  One pass over the volume; the right disparities of a row go
 * through (grid x W x 4 bytes of) scratch from the library's stream-ordered pool; no atomics, no host synchronisation,
 * capture-safe; 64-bit indexing.  The volume must not hold NaN: for it the result is unspecified (the call does not fault). */
int ctd_disparity_check_f32(const float* vol, float* disp, float* score, float* disp_right, float* score_right,
                            uint8_t* valid, int64_t B, int64_t D, int64_t H, int64_t W, int max_diff, double uniqueness,
                            int subpixel, ctd_stream_t stream);
int ctd_disparity_check_f64(const double* vol, double* disp, double* score, double* disp_right, double* score_right,
                            uint8_t* valid, int64_t B, int64_t D, int64_t H, int64_t W, int max_diff, double uniqueness,
                            int subpixel, ctd_stream_t stream);

/* ---- speckle filter of a disparity map (an addition: OpenCV's filterSpeckles, the speckleWindowSize / speckleRange step
 * of StereoSGBM, the peak filter of Hirschmueller's SGM): drop small connected regions of nearly equal disparity.
 *   Inputs.  disp [B,1,H,W], float or double; valid, the same shape, uint8, nonzero meaning valid, NULL meaning every
 *            pixel is valid; an integer max_size >= 0; a finite max_diff >= 0.
 *   Adjacency.  Pixels p and q of the same image are adjacent when all of these hold: they are 4-neighbours
 *            (|dh| + |dw| = 1); both are valid; |(double)disp[p] - (double)disp[q]| <= max_diff, evaluated in fp64.  A NaN
 *            disparity is therefore adjacent to nothing.  Adjacency is not transitive in value: 0, 1, 2 in a row with
 *            max_diff = 1 form one component.
 *   Components.  They are the connected components of that graph.  A valid pixel with no adjacent pixel is a component of
 *            size 1.
 *   Output.  valid_out[p] = valid[p] && size(component of p) > max_size (uint8, 0 or 1), and disp is not modified.  This
 *            equals OpenCV's filterSpeckles(disp, newVal, max_size, max_diff) with invalid pixels preset to newVal.
 *            max_size = 0 returns valid unchanged.
 *   Exactness.  Component membership does not depend on the algorithm that finds it, and sizes are integer counts.  So
 *            the output is bit-equal to the definition, deterministic, and independent of the order in which atomics land.
 * DEVICE pointers.  valid_out == NULL makes the call a no-op.  B*H*W = 0 is CTD_OK with nothing launched.  CTD_ERR_INVALID,
 * checked before any device work, for: negative sizes; H*W > INT32_MAX (labels are image-local int32); a null disp;
 * max_size < 0; a negative or non-finite max_diff; valid_out overlapping disp or valid.  Union-find labelling in four
 * launches whatever the sizes; labels and sizes (8 bytes per pixel of int32) come from the library's stream-ordered
 * scratch pool; integer atomics only, no host synchronisation, capture-safe; 64-bit indexing over the batch. */
int ctd_speckle_filter_f32(const float* disp, const uint8_t* valid, uint8_t* valid_out, int64_t B, int64_t H, int64_t W,
                           int64_t max_size, double max_diff, ctd_stream_t stream);
int ctd_speckle_filter_f64(const double* disp, const uint8_t* valid, uint8_t* valid_out, int64_t B, int64_t H, int64_t W,
                           int64_t max_size, double max_diff, ctd_stream_t stream);

/* ---- correlation soft-argmax disparity (an addition: the differentiable matching head of DispNetC / ActiveStereoNet), fused
 * forward and backward that never write the B x D x H x W score volume.
 *   Inputs.  f0, f1: [B,C,H,W] (or [C,H,W]), same shape, dtype (float or double) and device, contiguous; n_disps = D >= 1;
 *            temperature = tau, finite and > 0.
 *   Scores.  For pixel (b,h,w), let Dw = min(D, w + 1).  Only w - d >= 0 is a correspondence: there is no clamped column
 *            and no zero padding.  For d < Dw, s_d = (sum_c f0[b,c,h,w] * f1[b,c,h,w-d]) / C.  This is the DispNetC /
 *            FlowNet correlation normalisation.  Higher is better, the convention of xcorrvol and census_vol.
 *   Soft-argmax.  m = max_d s_d/tau; lse = m + log sum_{d<Dw} exp(s_d/tau - m); p_d = exp(s_d/tau - lse);
 *            disp = sum_{d<Dw} d * p_d.  Output disp is [B,1,H,W] (or [1,H,W]) in the input dtype.  At w = 0, disp = 0.
 *   Gradient.  d disp / d s_d = p_d * (d - disp) / tau, chained through s_d to both f0 and f1.  Either input may not
 *            require grad.  Double backward is not supported (once_differentiable).
 *   Non-finite input is outside the contract.  The result is unspecified, but the call must not fault.
 * Sums of products in a different order differ in the last bits, so this op is checked against a tolerance, not bit for
 * bit.
 * DEVICE pointers.  fwd writes disp and lse ([B,1,H,W] each, lse saved for bwd).  bwd takes grad_disp [B,1,H,W] and writes
 * grad_f0 and grad_f1 ([B,C,H,W], overwritten); either may be NULL (that half is skipped), both NULL is a no-op.
 * B*H*W = 0 is CTD_OK with nothing launched.  CTD_ERR_INVALID, checked before any device work, for: negative sizes; C < 1
 * or D < 1 when B*H*W > 0; a temperature that is non-positive or non-finite; C or H > INT32_MAX, W > INT32_MAX / 4; null
 * required pointers; any output overlapping an input or another output.  One launch for fwd, one per gradient for bwd;
 * no scratch memory, no atomics (the gradients are bit-identical from run to run), no host synchronisation,
 * capture-safe; 64-bit indexing over the batch. */
int ctd_corr_softargmax_fwd_f32(const float* f0, const float* f1, float* disp, float* lse, int64_t B, int64_t C, int64_t H,
                                int64_t W, int64_t n_disps, double temperature, ctd_stream_t stream);
int ctd_corr_softargmax_fwd_f64(const double* f0, const double* f1, double* disp, double* lse, int64_t B, int64_t C,
                                int64_t H, int64_t W, int64_t n_disps, double temperature, ctd_stream_t stream);
int ctd_corr_softargmax_bwd_f32(const float* f0, const float* f1, const float* disp, const float* lse,
                                const float* grad_disp, float* grad_f0, float* grad_f1, int64_t B, int64_t C, int64_t H,
                                int64_t W, int64_t n_disps, double temperature, ctd_stream_t stream);
int ctd_corr_softargmax_bwd_f64(const double* f0, const double* f1, const double* disp, const double* lse,
                                const double* grad_disp, double* grad_f0, double* grad_f1, int64_t B, int64_t C, int64_t H,
                                int64_t W, int64_t n_disps, double temperature, ctd_stream_t stream);

/* ---- ProjNNFunctor: ext.h:65-117, ext_cuda.cpp:47-69 (proj_nn_cuda).  K is a DEVICE pointer to
 * 9 values (row-major 3x3), like the reference's K tensor. */
int ctd_proj_nn_f32(const float* xyz0, const float* xyz1, const float* K, int64_t* out, int64_t B,
                    int64_t H, int64_t W, int patch_size, ctd_stream_t stream);
int ctd_proj_nn_f64(const double* xyz0, const double* xyz1, const double* K, int64_t* out, int64_t B,
                    int64_t H, int64_t W, int patch_size, ctd_stream_t stream);

/* ---- NNFunctor<T,3>: ext.h:13-46, ext_cuda.cpp:9-26 (nn_cuda).  in0 [N0,3], in1 [N1,3]. */
int ctd_nn_f32(const float* in0, const float* in1, int64_t* out, int64_t N0, int64_t N1,
               ctd_stream_t stream);
int ctd_nn_f64(const double* in0, const double* in1, int64_t* out, int64_t N0, int64_t N1,
               ctd_stream_t stream);

/* ---- CrossCheckFunctor: ext.h:48-63, ext_cuda.cpp:31-43 (crosscheck_cuda).  N1 is used only to
 * reject out-of-range gathers (they yield 0; the reference reads out of bounds there). */
int ctd_crosscheck(const int64_t* in0, const int64_t* in1, uint8_t* out, int64_t N0, int64_t N1,
                   ctd_stream_t stream);

/* ---- LCN: model/networks.py:507-533 (LCN.tforward).  x [N,1,H,W] -> lcn, std [N,1,H,W]. */
int ctd_lcn_f32(const float* x, float* lcn, float* std, int64_t N, int64_t H, int64_t W, int radius,
                float epsilon, ctd_stream_t stream);
int ctd_lcn_f64(const double* x, double* lcn, double* std, int64_t N, int64_t H, int64_t W,
                int radius, double epsilon, ctd_stream_t stream);

/* ---- RectifiedPatternSimilarityLoss.tforward + backward to the disparity, model/networks.py:358-378, as ONE kernel
 * (census modes, block 9): grid_sample(pattern, grid(disp), border) formed inside the loss kernel's tile loader, loss map,
 * masked-mean terms sums2 = (sum(mask * out), sum(mask)) and d loss / d disp for `grad_out` (w.r.t. the loss map).
 * pattern [Bp,1,Hp,Wp] with Bp = 1 or B; everything else [B,1,H,W]. */
int ctd_pattern_similarity_f32(const float* pattern, const float* disp, const float* ta, const float* grad_out,
                               const float* mask, float* pattern_proj, float* out, float* grad_disp, float* sums2,
                               int64_t B, int64_t Bp, int64_t Hp, int64_t Wp, int64_t H, int64_t W, int type, float eps,
                               ctd_stream_t stream);

/* ---- LCN backward: what autograd produces for networks.LCN (model/networks.py:523-533) w.r.t. its input, given the
 * forward's input x, its outputs (lcn, std) and upstream gradients for both outputs (either may be NULL = zero).
 * radius <= 8 (CTD_ERR_INVALID above; the forward takes any radius); any number of images N. */
int ctd_lcn_bwd_f32(const float* x, const float* lcn, const float* std, const float* grad_lcn, const float* grad_std,
                    float* grad_x, int64_t N, int64_t H, int64_t W, int radius, float epsilon, ctd_stream_t stream);

/* ---- the data generator's offline LCN: data/lcn/lcn.pyx:16-58 `normalize(img, kernel_size, epsilon)` (called at
 * data/create_syn_data.py:182) for a batch of B images [M,N] -- no padding (a border of kernel_size pixels stays 0),
 * centred two-pass variance, std = sqrt(var); bit-identical to the Cython build. */
int ctd_lcn_cython_f32(const float* img, float* lcn, float* std, int64_t B, int64_t M, int64_t N, int kernel_size,
                       float epsilon, ctd_stream_t stream);

/* ---- masked loss reduction of the caller, model/networks.py:377: val = (mask*diff).sum() / mask.sum().
 * out2[0] = sum(mask*diff), out2[1] = sum(mask), deterministic.  `workspace`: device memory of
 * ctd_masked_sums_workspace_bytes() bytes, zero-filled once before first use, one per concurrent stream. */
int64_t ctd_masked_sums_workspace_bytes(void);
int ctd_masked_sums_f32(const float* diff, const float* mask, int64_t n, float* out2, void* workspace,
                        ctd_stream_t stream);

/* ---- host-buffer entry points (fp32): same arguments, HOST pointers, synchronous.  They stage
 * through a per-thread grow-only device workspace on the current device. */
int ctd_host_photometric_fwd_f32(const float* es, const float* ta, float* out, int64_t B, int64_t C,
                                 int64_t H, int64_t W, int block_size, int type, float eps);
int ctd_host_photometric_bwd_f32(const float* es, const float* ta, const float* grad_out,
                                 float* grad_in, int64_t B, int64_t C, int64_t H, int64_t W,
                                 int block_size, int type, float eps);
/* forward and backward in one staged call: es/ta cross the bus once */
int ctd_host_photometric_fwd_bwd_f32(const float* es, const float* ta, const float* grad_out,
                                     float* out, float* grad_in, int64_t B, int64_t C, int64_t H,
                                     int64_t W, int block_size, int type, float eps);
/* the whole use the reference's caller makes of the loss (model/networks.py:376-377) in one staged call: loss map
 * (`out`, may be NULL: then it is not downloaded), d loss / d es for the caller's grad_out, and the masked-mean terms
 * sums2[0] = sum(mask * loss), sums2[1] = sum(mask) (host float[2]) */
int ctd_host_photometric_fwd_bwd_masked_f32(const float* es, const float* ta, const float* grad_out,
                                            const float* mask, float* out, float* grad_in, float* sums2,
                                            int64_t B, int64_t C, int64_t H, int64_t W, int block_size,
                                            int type, float eps);
int ctd_host_xcorrvol_f32(const float* in0, const float* in1, float* out, int64_t B, int64_t C,
                          int64_t H, int64_t W, int64_t n_disps, int block_size);
int ctd_host_proj_nn_f32(const float* xyz0, const float* xyz1, const float* K, int64_t* out,
                         int64_t B, int64_t H, int64_t W, int patch_size);
int ctd_host_nn_f32(const float* in0, const float* in1, int64_t* out, int64_t N0, int64_t N1);
int ctd_host_crosscheck(const int64_t* in0, const int64_t* in1, uint8_t* out, int64_t N0, int64_t N1);
int ctd_host_lcn_f32(const float* x, float* lcn, float* std, int64_t N, int64_t H, int64_t W,
                     int radius, float epsilon);
/* Deferred mode for the calling thread: between begin and end the ctd_host_* calls only enqueue their copies and
 * kernels (they return at once), so consecutive calls overlap on the bus; every result is in host memory when
 * ctd_host_end_batch() returns.  Input buffers must stay untouched, output buffers unread, until then.
 * An input that several photometric calls of one batch read (same host address and size: the image pair of two
 * loss types, the gradient weights) is uploaded once.  An input that is an OUTPUT of an earlier call of the same batch
 * (LCN's std used as the loss mask, ProjNN's indices fed to CrossCheck) is taken from that call's device buffer when
 * address and size match exactly (no copy at all); any other overlap with an output still in flight first waits for
 * the downloads, then uploads what the host holds.  Later calls of a batch may overwrite an earlier call's inputs or
 * outputs: the batch's results are those of the same calls made one at a time. */
int ctd_host_begin_batch(void);
int ctd_host_end_batch(void);
/* Two batches in flight: ctd_host_end_batch_async() returns once the batch is enqueued, ctd_host_wait_batch() waits for the
 * OLDEST batch not waited for yet (CTD_OK at once if there is none); a thread may have two such batches outstanding -- the
 * third ctd_host_begin_batch waits for the oldest itself.  With steps issued as begin / calls / end_async / wait (for
 * the previous step), the uploads of step k + 1 cross the bus under the downloads of step k.  Results of a batch are in
 * host memory after its wait; until then its host inputs must not change, its host outputs must not be read -- or be
 * passed as inputs to a later batch.  ctd_host_end_batch() (and any ctd_host_* call outside a batch) waits for
 * everything outstanding. */
int ctd_host_end_batch_async(void);
int ctd_host_wait_batch(void);
/* host-to-device bytes the calling thread's current (or last) batch copied, and bytes it did not have to copy again */
void ctd_host_batch_stats(uint64_t* h2d_bytes, uint64_t* h2d_bytes_saved);
/* Repeated batches (opt-in: ctd_set_option("host_graphs", 1)): a batch whose calls (entry points, arguments, host
 * addresses) equal those of an earlier batch of the thread, with every host buffer in pinned memory, is captured into
 * a CUDA graph the second time and replayed from the third on -- ctd_host_end_batch then issues ONE graph launch
 * instead of the batch's copies, kernels and events.  The calls of a replayed batch return at once; host inputs are
 * read when ctd_host_end_batch runs (the contract above: they must not change while the batch is open).  A batch that
 * stops matching is issued the ordinary way from the point of divergence.  Measured on the bench's step: the same
 * step time (the step is bound by the bus), the host thread's time in the calls drops from 0.09 ms to 0.01 ms (profiles/r02_e2e_chunks.json).
 * Counters for the calling thread: graphs captured, graph launches (the capturing batch included), expectations given up. */
void ctd_host_graph_stats(uint64_t* captured, uint64_t* launched, uint64_t* bailed);
/* release the calling thread's staging workspace */
void ctd_host_release(void);

#ifdef __cplusplus
}
#endif
#endif /* CTD_B200_H */
