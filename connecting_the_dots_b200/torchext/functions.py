"""The reference's op API (torchext/functions.py:5-147), same names, signatures, defaults and return
types, dispatching to the B200 kernels.  CUDA tensors go to ext_cuda (libctd_b200.so); CPU tensors
reach ext_cpu, which raises -- there is no CPU implementation.

Only photometric_loss is differentiable (w.r.t. `es`); the index / cost-volume ops return None
gradients like the reference (functions.py:15-17,33-35,50-52,69-71).
"""
import torch

from . import ext_cpu
from . import ext_cuda

LOSS_TYPES = {"mse": 0, "sad": 1, "census_mse": 2, "census_sad": 3}  # ext.h:196-199


def _native(t, cuda_name, cpu_name):
    return getattr(ext_cuda, cuda_name) if t.is_cuda else getattr(ext_cpu, cpu_name)


def _cuda_only(t, op):
    if not t.is_cuda:
        raise RuntimeError("torchext.%s: connecting_the_dots_b200 has no CPU implementation" % op)


class NNFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, in0, in1):
        return _native(in0, "nn_cuda", "nn_cpu")(in0, in1)

    @staticmethod
    def backward(ctx, grad_out):
        return None, None


def nn(in0, in1):
    """For every row of in0 [N0,3] the index of its nearest row of in1 [N1,3] (int64, -1 if none)."""
    return NNFunction.apply(in0, in1)


class CrossCheckFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, in0, in1):
        return _native(in0, "crosscheck_cuda", "crosscheck_cpu")(in0, in1)

    @staticmethod
    def backward(ctx, grad_out):
        return None, None


def crosscheck(in0, in1):
    """uint8 mask: in0[i] = j >= 0 and in1[j] == i (mutual consistency of two index maps)."""
    return CrossCheckFunction.apply(in0, in1)


class ProjNNFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xyz0, xyz1, K, patch_size):
        return _native(xyz0, "proj_nn_cuda", "proj_nn_cpu")(xyz0, xyz1, K, patch_size)

    @staticmethod
    def backward(ctx, grad_out):
        return None, None, None, None


def proj_nn(xyz0, xyz1, K, patch_size):
    """Project xyz0 with K, search a patch_size^2 pixel patch of xyz1 for the nearest 3-D point."""
    return ProjNNFunction.apply(xyz0, xyz1, K, patch_size)


class XCorrVolFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, in0, in1, n_disps, block_size):
        return _native(in0, "xcorrvol_cuda", "xcorrvol_cpu")(in0, in1, n_disps, block_size)

    @staticmethod
    def backward(ctx, grad_out):
        return None, None, None, None


def xcorrvol(in0, in1, n_disps, block_size):
    """Normalised cross-correlation cost volume [n_disps,H,W] of in0 against in1 shifted by d."""
    return XCorrVolFunction.apply(in0, in1, n_disps, block_size)


def xcorr_disparity(in0, in1, n_disps, block_size, subpixel=True):
    """Block-matching disparity from the xcorrvol cost volume, without writing the volume: (disp, score), [B,1,H,W] for a
    [B,C,H,W] pair ([1,H,W] for the reference's [C,H,W]), in the input's dtype, not differentiable.  d* is the first d with
    the largest score (winner-take-all), score the peak correlation there; with subpixel, disp = d* + the vertex offset of
    the parabola through the scores at d* - 1, d*, d* + 1 (disparity_from_volume states it).  d* and score equal
    disparity_from_volume(xcorrvol(in0, in1, n_disps, block_size)) exactly.  CUDA tensors only, float32 or float64."""
    _cuda_only(in0, "xcorr_disparity")
    return ext_cuda.xcorr_disparity_cuda(in0, in1, n_disps, block_size, subpixel)


def _subpixel(src, d, lim):
    """The sub-pixel offset of the winner-take-all disparity d [B,1,H,W] of src [B,D,H,W], in float64: with c-, c0, c+ =
    src at d - 1, d, d + 1 and den = c- - 2 c0 + c+, clamp((c- - c+) / (2 den), -0.5, 0.5), and 0 where d = 0,
    d >= lim - 1 (lim: the disparities the pixel has) or den >= 0."""
    D = src.size(1)
    cm = src.gather(1, (d - 1).clamp(min=0)).double()
    c0 = src.gather(1, d).double()
    cp = src.gather(1, (d + 1).clamp(max=D - 1)).double()
    den = cm - 2 * c0 + cp
    ok = (d > 0) & (d < lim - 1) & (den < 0)
    return torch.where(ok, (cm - cp) / (2 * torch.where(ok, den, -1.0)), 0.0).clamp(-0.5, 0.5)


def disparity_from_volume(vol, subpixel=True):
    """Winner-take-all disparity of a cost volume [B,D,H,W] (or [D,H,W]) in plain torch, any device: the definition of
    xcorr_disparity and its test oracle.  d* = the first d with vol[:, d] equal to the maximum over d; score = vol at d*;
    with subpixel, c-, c0, c+ = vol at d* - 1, d*, d* + 1, den = c- - 2 c0 + c+ and disp = d* + clamp((c- - c+) / (2 den),
    -0.5, 0.5), in float64, the offset 0 where d* = 0, d* = D - 1 or den >= 0.  Returns (disp, score), [B,1,H,W] (or
    [1,H,W]), in vol's dtype.  For finite volumes; a column holding NaN gives d* = D - 1 (no error)."""
    v = vol if vol.dim() == 4 else vol.unsqueeze(0)
    D = v.size(1)
    if D < 1:
        raise RuntimeError("disparity_from_volume: the volume has no disparities")
    idx = torch.arange(D, device=v.device).view(1, D, 1, 1)
    # the first maximum (a column holding NaN has none: it gets d = D - 1, outside the finite-input contract)
    d = torch.where(v == v.amax(dim=1, keepdim=True), idx, D).amin(dim=1, keepdim=True).clamp(max=D - 1)
    score = v.gather(1, d)
    disp = d.to(torch.float64)
    if subpixel:
        disp = disp + _subpixel(v, d, D)
    disp = disp.to(vol.dtype)
    if vol.dim() == 3:
        disp, score = disp[0], score[0]
    return disp, score


def _disparity_check_args(op, vol, uniqueness):
    if vol.dim() not in (3, 4):
        raise RuntimeError("%s: vol has to be D x H x W (or B x D x H x W)" % op)
    u = float(uniqueness)
    if not (u >= 0.0 and u != float("inf")):
        raise RuntimeError("%s: uniqueness must be finite and >= 0, got %r" % (op, uniqueness))
    return u


def disparity_check(vol, max_diff=1, uniqueness=0.0, subpixel=True):
    """Left-right consistency and uniqueness checks of the winner-take-all disparity of a score volume vol [B,D,H,W] (or
    [D,H,W]; higher is better, the convention of xcorrvol, census_vol and sgm_aggregate), in one pass over the volume.
    Returns (disp, score, valid), [B,1,H,W] (or [1,H,W]): disp and score equal disparity_from_volume(vol, subpixel) bit for
    bit, valid (torch.bool) marks the pixels that pass both checks as disparity_check_pytorch states them.  max_diff < 0
    turns the LR check off, uniqueness = 0 the uniqueness check.  Not differentiable.  CUDA tensors only, float32 or
    float64."""
    _cuda_only(vol, "disparity_check")
    u = _disparity_check_args("disparity_check", vol, uniqueness)
    return ext_cuda.disparity_check_cuda(vol, int(max_diff), u, subpixel)


def right_disparity_from_volume(vol, subpixel=True):
    """Winner-take-all disparity of the right view of a score volume [B,D,H,W] (or [D,H,W]) in plain torch, any device:
    part of disparity_check's definition and its test oracle.  For right pixel x, Dx = min(D, W - x) and VR[d,h,x] =
    V[d,h,x+d] for d < Dx.  dR* = the first d in [0, Dx) with the largest VR, score = VR at dR*; with subpixel, c-, c0, c+
    = VR at dR* - 1, dR*, dR* + 1 and disparity_from_volume's fp64 offset, 0 where dR* = 0, dR* = Dx - 1 or den >= 0.
    Returns (disp, score), [B,1,H,W] (or [1,H,W]), in vol's dtype.  For volumes without NaN."""
    v = vol if vol.dim() == 4 else vol.unsqueeze(0)
    B, D, H, W = v.shape
    if D < 1:
        raise RuntimeError("right_disparity_from_volume: the volume has no disparities")
    idx = torch.arange(D, device=v.device).view(1, D, 1, 1)
    x = torch.arange(W, device=v.device).view(1, 1, 1, W)
    cols = x + idx                                                  # [1,D,1,W]
    ok = cols < W
    vr = v.gather(3, cols.clamp(max=W - 1).expand(B, D, H, W))      # VR where ok, a clamped column elsewhere
    best = torch.where(ok, vr, float("-inf")).amax(dim=1, keepdim=True)
    d = torch.where(ok & (vr == best), idx, D).amin(dim=1, keepdim=True)
    score = vr.gather(1, d)
    disp = d.to(torch.float64)
    if subpixel:
        disp = disp + _subpixel(vr, d, (W - x).clamp(max=D))
    disp = disp.to(vol.dtype)
    if vol.dim() == 3:
        disp, score = disp[0], score[0]
    return disp, score


def disparity_check_pytorch(vol, max_diff=1, uniqueness=0.0, subpixel=True):
    """The definition of disparity_check in plain torch, any device, and its test oracle.  (disp, score) =
    disparity_from_volume(vol, subpixel); with d*L the integer left disparity and dR* that of right_disparity_from_volume,
    valid = LR and uniqueness, where LR: max_diff < 0, or x = w - d*L >= 0 and |d*L - dR*(x)| <= max_diff; uniqueness:
    uniqueness == 0, or no d has |d - d*L| >= 2, or (double)vol[d*L] - (double)max{vol[d] : |d - d*L| >= 2} >= uniqueness."""
    u = _disparity_check_args("disparity_check", vol, uniqueness)
    v = vol if vol.dim() == 4 else vol.unsqueeze(0)
    B, D, H, W = v.shape
    disp, score = disparity_from_volume(v, subpixel)
    dl = disparity_from_volume(v, False)[0].long()
    dr = right_disparity_from_volume(v, False)[0].long()
    valid = torch.ones_like(dl, dtype=torch.bool)
    if max_diff >= 0:
        x = torch.arange(W, device=v.device).view(1, 1, 1, W) - dl
        valid &= (x >= 0) & ((dl - dr.gather(3, x.clamp(min=0))).abs() <= max_diff)
    if u != 0:
        far = (torch.arange(D, device=v.device).view(1, D, 1, 1) - dl).abs() >= 2
        second = torch.where(far, v, float("-inf")).amax(dim=1, keepdim=True)
        valid &= ~far.any(dim=1, keepdim=True) | (score.double() - second.double() >= u)
    if vol.dim() == 3:
        disp, score, valid = disp[0], score[0], valid[0]
    return disp, score, valid


def _speckle_args(op, disp, valid, max_size, max_diff):
    if disp.dim() not in (3, 4) or disp.size(-3) != 1:
        raise RuntimeError("%s: disp has to be 1 x H x W (or B x 1 x H x W)" % op)
    ext_cuda._real_suffix(disp, op)
    if valid is not None:
        if valid.dtype != torch.bool or tuple(valid.shape) != tuple(disp.shape):
            raise RuntimeError("%s: valid has to be a bool tensor of disp's shape" % op)
        if valid.device != disp.device:
            raise RuntimeError("%s: disp and valid must be on the same device" % op)
    n, md = int(max_size), float(max_diff)
    if n != max_size or n < 0:
        raise RuntimeError("%s: max_size must be an integer >= 0, got %r" % (op, max_size))
    if not (md >= 0.0 and md != float("inf")):
        raise RuntimeError("%s: max_diff must be finite and >= 0, got %r" % (op, max_diff))
    return n, md


def speckle_filter(disp, valid=None, max_size=100, max_diff=1.0):
    """Speckle filter of a disparity map disp [B,1,H,W] (or [1,H,W]): drop the connected regions of nearly equal disparity
    with at most max_size pixels, as speckle_filter_pytorch states it.  valid (bool, disp's shape; None: every pixel) marks
    the pixels that take part.  Returns valid_out (bool, disp's shape); disp is not modified.  Not differentiable.  CUDA
    tensors only, float32 or float64."""
    _cuda_only(disp, "speckle_filter")
    n, md = _speckle_args("speckle_filter", disp, valid, max_size, max_diff)
    return ext_cuda.speckle_filter_cuda(disp, valid, n, md)


def speckle_filter_pytorch(disp, valid=None, max_size=100, max_diff=1.0):
    """The definition of speckle_filter in plain torch, any device, and its test oracle.

    Inputs: disp [B,1,H,W] (or [1,H,W]), float32 or float64; valid, the same shape, bool, None meaning every pixel is
    valid; an integer max_size >= 0; a finite max_diff >= 0.
    Adjacency: pixels p and q of the same image are adjacent when all of these hold: they are 4-neighbours
    (|dh| + |dw| = 1); both are valid; |(double)disp[p] - (double)disp[q]| <= max_diff, evaluated in fp64.  A NaN disparity
    is therefore adjacent to nothing.  Adjacency is not transitive in value: 0, 1, 2 in a row with max_diff = 1 form one
    component.
    Components: they are the connected components of that graph.  A valid pixel with no adjacent pixel is a component of
    size 1.
    Output: valid_out[p] = valid[p] && size(component of p) > max_size, and disp is not modified.  This equals OpenCV's
    filterSpeckles(disp, newVal, max_size, max_diff) with invalid pixels preset to newVal.  max_size = 0 returns valid
    unchanged.
    Exactness: component membership does not depend on the algorithm that finds it, and sizes are integer counts.  So the
    output is bit-equal to the definition, deterministic, and independent of the order in which atomics land.

    Components are found by min-label hooking with pointer jumping (scatter_reduce "amin") until a fixed point."""
    n, md = _speckle_args("speckle_filter", disp, valid, max_size, max_diff)
    d = disp.reshape(-1, disp.size(-2), disp.size(-1)).double()
    ok = torch.ones(d.shape, dtype=torch.bool, device=d.device) if valid is None else valid.reshape(d.shape)
    B, H, W = d.shape
    idx = torch.arange(B * H * W, device=d.device).view(B, H, W)
    right = ok[:, :, :-1] & ok[:, :, 1:] & ((d[:, :, :-1] - d[:, :, 1:]).abs() <= md)
    down = ok[:, :-1] & ok[:, 1:] & ((d[:, :-1] - d[:, 1:]).abs() <= md)
    src = torch.cat([idx[:, :, :-1][right], idx[:, :-1][down]])
    dst = torch.cat([idx[:, :, 1:][right], idx[:, 1:][down]])
    lab = idx.view(-1)  # lab[x] <= x, a pixel of x's component; lab[lab] == lab after every round
    while True:
        ls, ld = lab[src], lab[dst]
        m = torch.minimum(ls, ld)
        new = lab.scatter_reduce(0, ls, m, "amin").scatter_reduce(0, ld, m, "amin")  # hook each edge's roots to the smaller
        while True:
            jumped = new[new]
            if torch.equal(jumped, new):
                break
            new = jumped
        if torch.equal(new, lab):  # every edge joins two pixels of one label: lab is the component's smallest pixel
            break
        lab = new
    size = torch.bincount(lab, minlength=lab.numel())[lab].view(B, H, W)
    return (ok & (size > n)).view(disp.shape)


SGM_PATHS = {4:((0, 1), (0, -1), (1, 0), (-1, 0)),
             8: ((0, 1), (0, -1), (1, 0), (-1, 0), (1, 1), (1, -1), (-1, 1), (-1, -1))}


def sgm_aggregate(vol, p1, p2, paths=8):
    """Semi-global matching (Hirschmueller, PAMI 2008) over a score volume vol [B,D,H,W] (or [D,H,W]; higher is better, the
    convention of xcorrvol: pass a cost volume negated): the aggregated volume A, same shape and dtype, equal bit for bit to
    sgm_aggregate_pytorch, which states the definition.  Not differentiable.  CUDA tensors only, float32 or float64."""
    _cuda_only(vol, "sgm_aggregate")
    return ext_cuda.sgm_cuda(vol, p1, p2, paths, want_disparity=False)[0]


def sgm_disparity(vol, p1, p2, paths=8, subpixel=True):
    """(disp, score) = disparity_from_volume(sgm_aggregate(vol, p1, p2, paths), subpixel), bit for bit, with the
    winner-take-all fused into the last aggregation pass; A is allocated and dropped.  [B,1,H,W] (or [1,H,W]), not
    differentiable, CUDA tensors only, float32 or float64."""
    _cuda_only(vol, "sgm_disparity")
    _, disp, score = ext_cuda.sgm_cuda(vol, p1, p2, paths, subpixel)
    return disp, score


def _sgm_check(vol, p1, p2, paths):
    if paths not in SGM_PATHS:
        raise RuntimeError("sgm: paths must be 4 or 8, got %r" % (paths,))
    if vol.dim() not in (3, 4) or vol.size(-3) < 1:
        raise RuntimeError("sgm: vol has to be D x H x W (or B x D x H x W) with D >= 1")
    if vol.dtype not in (torch.float32, torch.float64):
        raise NotImplementedError("sgm: float32 or float64 volumes only")
    t1, t2 = (torch.tensor(float(p), dtype=vol.dtype, device=vol.device) for p in (p1, p2))
    if not (torch.isfinite(t1) and torch.isfinite(t2) and 0 <= t1 <= t2):
        raise RuntimeError("sgm: penalties must be finite with 0 <= p1 <= p2 (p1 = %r, p2 = %r)" % (p1, p2))
    return t1, t2


def sgm_aggregate_pytorch(vol, p1, p2, paths=8):
    """The definition of sgm_aggregate in plain torch, any device, in vol's dtype, and its test oracle.  For each path
    direction r = (dy, dx) in the order of SGM_PATHS[paths] and q = p - r: L_r(p, d) = V(p, d) where q is outside the image,
    else L_r(p, d) = V(p, d) + (m - M) with M = max_k L_r(q, k) and m = max(L_r(q, d), L_r(q, d-1) - p1, L_r(q, d+1) - p1,
    M - p2) over the neighbours inside [0, D); p1, p2 converted once to vol's dtype.  A = (((L_0 + L_1) + L_2) + ...)."""
    t1, t2 = _sgm_check(vol, p1, p2, paths)
    v = vol if vol.dim() == 4 else vol.unsqueeze(0)
    B, D, H, W = v.shape

    def step(lq, cur, valid):
        # lq: L_r(q, .) aligned with cur [B,D,N]; valid [N]: q inside the image
        M = lq.amax(dim=1, keepdim=True)
        ninf = torch.full_like(lq[:, :1], float("-inf"))
        dn = torch.cat([ninf, lq[:, :-1]], 1) - t1     # L(q, d-1) - p1
        up = torch.cat([lq[:, 1:], ninf], 1) - t1      # L(q, d+1) - p1
        m = torch.maximum(torch.maximum(lq, dn), torch.maximum(up, M - t2))
        return torch.where(valid, cur + (m - M), cur)

    agg = None
    for dy, dx in SGM_PATHS[paths]:
        L = torch.empty_like(v)
        if dy == 0:    # along rows: lines are [B,D,H] columns of pixels
            ws = range(W) if dx > 0 else range(W - 1, -1, -1)
            prev = None
            for w in ws:
                L[..., w] = v[..., w] if prev is None else step(prev, v[..., w], torch.ones(H, dtype=torch.bool, device=v.device))
                prev = L[..., w]
        else:          # row by row, the predecessor row shifted by dx
            hs = range(H) if dy > 0 else range(H - 1, -1, -1)
            prev = None
            cols = torch.arange(W, device=v.device)
            valid = (cols - dx >= 0) & (cols - dx < W)
            for h in hs:
                if prev is None:
                    L[:, :, h] = v[:, :, h]
                else:
                    lq = prev if dx == 0 else torch.roll(prev, dx, dims=2)   # lq[..., w] = prev[..., w - dx]
                    L[:, :, h] = step(lq, v[:, :, h], valid)
                prev = L[:, :, h]
        agg = L if agg is None else agg + L
    return agg if vol.dim() == 4 else agg[0]


def _census_check(op, window, block_size=1, C=0):
    """The argument checks of the census entry points, with the C ABI's wording: (wh, ww) odd with 2 <= wh*ww <= 65,
    block_size odd in [1, 15], C*(wh*ww-1)*block_size^2 <= 2^24."""
    try:
        wh, ww = (int(v) for v in window)
    except (TypeError, ValueError):
        raise RuntimeError("%s: window has to be a pair (wh, ww), got %r" % (op, window))
    bs = int(block_size)
    if wh < 1 or ww < 1 or wh % 2 == 0 or ww % 2 == 0:
        raise RuntimeError("%s: window sides must be odd and positive, got %dx%d" % (op, wh, ww))
    if not 2 <= wh * ww <= 65:
        raise RuntimeError("%s: window %dx%d must have 2 to 65 taps" % (op, wh, ww))
    if not (1 <= bs <= 15 and bs % 2 == 1):
        raise RuntimeError("%s: block_size must be odd in [1,15], got %d" % (op, bs))
    bound = C * (wh * ww - 1) * bs * bs
    if bound > 1 << 24:
        raise RuntimeError("%s: C*(wh*ww-1)*block_size^2 = %d exceeds 2^24 (scores would not be exact in float32)" % (op, bound))
    return wh, ww, bs


def _census_inputs(op, in0, in1, n_disps, window, block_size):
    if in0.dim() not in (3, 4) or tuple(in0.shape) != tuple(in1.shape) or in0.dtype != in1.dtype:
        raise RuntimeError("%s: in0 and in1 have to be C x H x W (or B x C x H x W) of the same shape and dtype" % op)
    wh, ww, bs = _census_check(op, window, block_size, in0.size(-3))
    B = in0.size(0) if in0.dim() == 4 else 1
    if int(n_disps) < 1 and B * in0.size(-2) * in0.size(-1) > 0:
        raise RuntimeError("%s: n_disps must be >= 1 (D = 0)" % op)
    return wh, ww, bs


def census_transform(x, window=(7, 9)):
    """Census transform of each channel of x [B,C,H,W] (or [C,H,W]) over a window (wh, ww): int64 of x's shape holding the
    uint64 bit pattern (bit 63 makes it negative), equal to census_transform_pytorch, which states the definition.  Not
    differentiable.  CUDA tensors only, float32 or float64."""
    _cuda_only(x, "census_transform")
    wh, ww, _ = _census_check("census_transform", window)
    return ext_cuda.census_transform_cuda(x, wh, ww)


def census_vol(in0, in1, n_disps, window=(7, 9), block_size=1):
    """Census matching-score volume V [B,n_disps,H,W] (or [n_disps,H,W]) of in0 against in1 shifted by d, in the inputs'
    dtype: minus the block_size^2 box sum of the Hamming distances of the census descriptors.  Higher is better (the
    convention of xcorrvol), so sgm_disparity(census_vol(...), p1, p2) works as it is.  Equal bit for bit to
    census_vol_pytorch, which states the definition.  Not differentiable.  CUDA tensors only, float32 or float64."""
    _cuda_only(in0, "census_vol")
    wh, ww, bs = _census_inputs("census_vol", in0, in1, n_disps, window, block_size)
    return ext_cuda.census_vol_cuda(in0, in1, n_disps, wh, ww, bs)


def census_disparity(in0, in1, n_disps, window=(7, 9), block_size=9, subpixel=True):
    """(disp, score) = disparity_from_volume(census_vol(in0, in1, n_disps, window, block_size), subpixel), bit for bit
    including the sub-pixel offset, without writing the volume.  [B,1,H,W] (or [1,H,W]), not differentiable, CUDA tensors
    only, float32 or float64."""
    _cuda_only(in0, "census_disparity")
    wh, ww, bs = _census_inputs("census_disparity", in0, in1, n_disps, window, block_size)
    return ext_cuda.census_disparity_cuda(in0, in1, n_disps, wh, ww, bs, subpixel)


def census_transform_pytorch(x, window=(7, 9)):
    """The definition of census_transform in plain torch, any device, and its test oracle.  Number the taps (i, j) of the
    window, i in [0, wh), j in [0, ww), row-major, skipping the centre (wh//2, ww//2); bit k of T[b,c,h,w] is
    x[b,c,clamp(h+i-wh//2),clamp(w+j-ww//2)] < x[b,c,h,w] (IEEE <: NaN on either side gives 0).  Higher bits are 0."""
    wh, ww, _ = _census_check("census_transform", window)
    xb = x if x.dim() == 4 else x.unsqueeze(0)
    H, W = xb.shape[-2:]
    rh, rw = wh // 2, ww // 2
    taps = [(i, j) for i in range(wh) for j in range(ww) if (i, j) != (rh, rw)]
    ti = torch.tensor([i - rh for i, _ in taps], device=x.device)
    tj = torch.tensor([j - rw for _, j in taps], device=x.device)
    rows = (torch.arange(H, device=x.device) + ti[:, None]).clamp(0, H - 1)     # [K,H]
    cols = (torch.arange(W, device=x.device) + tj[:, None]).clamp(0, W - 1)     # [K,W]
    bits = (xb[:, :, rows[:, :, None], cols[:, None, :]] < xb.unsqueeze(2)).long()  # [B,C,K,H,W]
    shifts = torch.arange(len(taps), device=x.device).view(1, 1, -1, 1, 1)
    t = (bits << shifts).sum(2)  # disjoint bits: the sum is their OR (bit 63 is the int64 sign)
    return t if x.dim() == 4 else t[0]


_POPCOUNT8 = torch.tensor([bin(i).count("1") for i in range(256)], dtype=torch.int32)


def census_vol_pytorch(in0, in1, n_disps, window=(7, 9), block_size=1):
    """The definition of census_vol in plain torch, any device, in the inputs' dtype, and its test oracle.  With T0, T1 =
    census_transform_pytorch(in0, in1): Hm[b,d,h,w] = sum_c popcount(T0[b,c,h,w] ^ T1[b,c,h,clamp(w-d,0,W-1)]);
    S[b,d,h,w] = sum over i, j in [0, bs) of Hm[b,d,clamp(h+i-bs//2),clamp(w+j-bs//2)]; V = -S.  census_disparity's
    definition is disparity_from_volume(census_vol_pytorch(...))."""
    wh, ww, bs = _census_inputs("census_vol", in0, in1, n_disps, window, block_size)
    if in0.dtype not in (torch.float32, torch.float64):
        raise NotImplementedError("census_vol: float32 or float64 inputs only")
    a = in0 if in0.dim() == 4 else in0.unsqueeze(0)
    b = in1 if in1.dim() == 4 else in1.unsqueeze(0)
    B, C, H, W = a.shape
    D, r = int(n_disps), bs // 2
    t0, t1 = census_transform_pytorch(a, (wh, ww)), census_transform_pytorch(b, (wh, ww))
    lut = _POPCOUNT8.to(a.device)
    cols = torch.arange(W, device=a.device)
    box_r = (torch.arange(H, device=a.device) + torch.arange(-r, r + 1, device=a.device)[:, None]).clamp(0, H - 1)  # [bs,H]
    box_c = (cols + torch.arange(-r, r + 1, device=a.device)[:, None]).clamp(0, W - 1)                               # [bs,W]
    vol = torch.empty(B, D, H, W, dtype=in0.dtype, device=in0.device)
    for d in range(D):
        x = (t0 ^ t1[..., (cols - d).clamp(min=0)]).contiguous()
        hm = lut[x.view(torch.uint8).long()].view(B, C, H, W, 8).sum((1, 4))   # [B,H,W]
        if r:
            hm = hm[:, box_r].sum(1)          # [B,bs,H,W] -> rows summed
            hm = hm[:, :, box_c].sum(2)       # [B,H,bs,W] -> columns summed
        vol[:, d] = -(hm.to(in0.dtype))
    return vol if in0.dim() == 4 else vol[0]


class PhotometricLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, es, ta, block_size, type, eps):
        ctx.save_for_backward(es, ta)
        ctx.block_size, ctx.type, ctx.eps = block_size, type, eps
        return _native(es, "photometric_loss_forward", "photometric_loss_forward")(es, ta, block_size, type, eps)

    @staticmethod
    def backward(ctx, grad_out):
        es, ta = ctx.saved_tensors
        fn = _native(grad_out, "photometric_loss_backward", "photometric_loss_backward")
        grad_es = fn(es, ta, grad_out.contiguous(), ctx.block_size, ctx.type, ctx.eps)
        return grad_es, None, None, None, None


def _loss_type_id(type):
    try:
        return LOSS_TYPES[type.lower()]
    except KeyError:
        raise Exception("invalid loss type")


def photometric_loss(es, ta, block_size, type="mse", eps=0.1):
    """Block-window photometric loss map [B,1,H,W]; type in mse | sad | census_mse | census_sad."""
    return PhotometricLossFunction.apply(es, ta, block_size, _loss_type_id(type), eps)


def photometric_loss_pytorch(es, ta, block_size, type="mse", eps=0.1):
    """Plain-torch evaluation of the same loss (differentiable by autograd, any device); the
    counterpart of the reference's functions.py:120-147, written as a loop over window offsets on a
    replicate-padded copy instead of an unfold, so it needs O(1) extra image copies."""
    kind = type.lower()
    if kind not in LOSS_TYPES:
        raise Exception("invalid loss type")
    lo = block_size // 2
    hi = block_size - 1 - lo
    H, W = es.shape[2], es.shape[3]
    es_p = torch.nn.functional.pad(es, (lo, hi, lo, hi), mode="replicate")
    ta_p = torch.nn.functional.pad(ta, (lo, hi, lo, hi), mode="replicate")

    def soft_step(x):
        return 0.5 * (1 + x / torch.sqrt(x * x + eps))

    total = None
    for dy in range(block_size):
        for dx in range(block_size):
            e = es_p[:, :, dy:dy + H, dx:dx + W]
            t = ta_p[:, :, dy:dy + H, dx:dx + W]
            d = (soft_step(e - es) - soft_step(t - ta)) if kind.startswith("census") else (e - t)
            term = (d * d if kind.endswith("mse") else d.abs()).sum(dim=1, keepdim=True)
            total = term if total is None else total + term
    return total / block_size ** 2


class WeightedPhotometricLossFunction(torch.autograd.Function):
    """`(mask * photometric_loss(es, ta)).sum() / mask.sum()` -- the way the reference's only caller consumes the
    loss map (model/networks.py:377) -- as ONE op.  Its upstream gradient is a scalar, so the backward's grad_out is
    the mask up to that scalar and is known before the loss map exists: loss map, gradient and both sums come out of
    one fused pass (ctd_photometric_fwd_bwd_masked_f32, a single kernel for the census modes) and autograd's backward
    is a scalar multiply.  SURVEY section 8(f) rank 1, without the warp.  Returns (value, loss_map); mask is not
    differentiated (it is LCN's std in the reference)."""

    @staticmethod
    def forward(ctx, es, ta, mask, block_size, type, eps):
        _cuda_only(es, "weighted_photometric_loss")
        mask = mask.detach().contiguous()
        # grad_out = mask: the gradient comes back unnormalised and is divided by sum(mask) in backward
        out, grad_es, sums = ext_cuda.photometric_loss_forward_backward_masked(es.detach(), ta.detach(), mask, mask, block_size, type, eps)
        ctx.save_for_backward(grad_es, sums)
        ctx.mark_non_differentiable(out)
        return sums[0] / sums[1], out

    @staticmethod
    def backward(ctx, g_val, g_map):
        grad_es, sums = ctx.saved_tensors
        return grad_es * (g_val / sums[1]), None, None, None, None, None


def weighted_photometric_loss(es, ta, mask, block_size, type="mse", eps=0.1):
    """Masked mean of the photometric loss map and the map itself: (value, loss_map [B,1,H,W])."""
    return WeightedPhotometricLossFunction.apply(es, ta, mask, block_size, _loss_type_id(type), eps)


SSIM_C1, SSIM_C2 = 0.01 ** 2, 0.03 ** 2


class SSIMLossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, es, ta, block_size, c1, c2):
        _cuda_only(es, "ssim_loss")
        es, ta = es.detach(), ta.detach()
        ctx.save_for_backward(es, ta)
        ctx.block_size, ctx.c1, ctx.c2 = block_size, c1, c2
        return ext_cuda.ssim_forward(es, ta, block_size, c1, c2)

    @staticmethod
    def backward(ctx, grad_out):
        es, ta = ctx.saved_tensors
        return ext_cuda.ssim_backward(es, ta, grad_out.contiguous(), ctx.block_size, ctx.c1, ctx.c2), None, None, None, None


def ssim_loss(es, ta, block_size, c1=SSIM_C1, c2=SSIM_C2):
    """SSIM photometric loss map [B,1,H,W]: for every pixel and channel the structural similarity S of es and ta over the
    block_size^2 window of photometric_loss (taps clamp(h + i - block_size//2), clamp(w + j - block_size//2), i, j in
    [0, block_size): replicate-clamped at the border), with population statistics
        S = (2 mx my + c1)(2 vxy + c2) / ((mx^2 + my^2 + c1)(vxx + vyy + c2)),
    and out = sum over channels of (1 - S) / 2 (not clamped).  c1, c2 > 0.  Differentiable w.r.t. es (ta gets no
    gradient).  CUDA tensors only, float32 or float64."""
    return SSIMLossFunction.apply(es, ta, block_size, c1, c2)


def ssim_loss_pytorch(es, ta, block_size, c1=SSIM_C1, c2=SSIM_C2):
    """Plain-torch evaluation of ssim_loss (differentiable by autograd, any device): the same loop over window offsets on
    a replicate-padded copy as photometric_loss_pytorch, with centred second moments."""
    lo = block_size // 2
    hi = block_size - 1 - lo
    H, W = es.shape[2], es.shape[3]
    es_p = torch.nn.functional.pad(es, (lo, hi, lo, hi), mode="replicate")
    ta_p = torch.nn.functional.pad(ta, (lo, hi, lo, hi), mode="replicate")
    taps = [(es_p[:, :, dy:dy + H, dx:dx + W], ta_p[:, :, dy:dy + H, dx:dx + W]) for dy in range(block_size) for dx in range(block_size)]
    n = block_size ** 2
    mx = sum(e for e, _ in taps) / n
    my = sum(t for _, t in taps) / n
    vxx = sum((e - mx) ** 2 for e, _ in taps) / n
    vyy = sum((t - my) ** 2 for _, t in taps) / n
    vxy = sum((e - mx) * (t - my) for e, t in taps) / n
    s = (2 * mx * my + c1) * (2 * vxy + c2) / ((mx * mx + my * my + c1) * (vxx + vyy + c2))
    return ((1 - s) / 2).sum(dim=1, keepdim=True)


class WeightedSSIMLossFunction(torch.autograd.Function):
    """`(mask * ssim_loss(es, ta)).sum() / mask.sum()` as ONE op, like WeightedPhotometricLossFunction: loss map,
    gradient and both sums from one fused pass (ctd_ssim_fwd_bwd_masked_f32); autograd's backward is a scalar multiply.
    Returns (value, loss_map); mask is not differentiated."""

    @staticmethod
    def forward(ctx, es, ta, mask, block_size, c1, c2):
        _cuda_only(es, "weighted_ssim_loss")
        mask = mask.detach().contiguous()
        # grad_out = mask: the gradient comes back unnormalised and is divided by sum(mask) in backward
        out, grad_es, sums = ext_cuda.ssim_forward_backward_masked(es.detach(), ta.detach(), mask, mask, block_size, c1, c2)
        ctx.save_for_backward(grad_es, sums)
        ctx.mark_non_differentiable(out)
        return sums[0] / sums[1], out

    @staticmethod
    def backward(ctx, g_val, g_map):
        grad_es, sums = ctx.saved_tensors
        return grad_es * (g_val / sums[1]), None, None, None, None, None


def weighted_ssim_loss(es, ta, mask, block_size, c1=SSIM_C1, c2=SSIM_C2):
    """Masked mean of the SSIM loss map and the map itself: (value, loss_map [B,1,H,W]); float32 CUDA tensors."""
    return WeightedSSIMLossFunction.apply(es, ta, mask, block_size, c1, c2)


class WarpPatternFunction(torch.autograd.Function):
    """The disparity warp of the reference pattern (model/networks.py:362-371): one gather kernel instead of
    building uv grids and calling grid_sample; differentiable w.r.t. disp."""

    @staticmethod
    def forward(ctx, pattern, disp):
        _cuda_only(disp, "warp_pattern")
        pattern, disp = pattern.detach().contiguous(), disp.detach().contiguous()
        ctx.save_for_backward(pattern, disp)
        return ext_cuda.warp_pattern_forward(pattern, disp)

    @staticmethod
    def backward(ctx, grad_out):
        pattern, disp = ctx.saved_tensors
        return None, ext_cuda.warp_pattern_backward(pattern, disp, grad_out.contiguous())


def warp_pattern(pattern, disp):
    """pattern [Bp,1,Hp,Wp] sampled at (u - disp, v) with the reference's grid convention -> [B,1,H,W]."""
    return WarpPatternFunction.apply(pattern, disp)


class PatternSimilarityFunction(torch.autograd.Function):
    """RectifiedPatternSimilarityLoss.tforward (model/networks.py:358-378) with its backward to the disparity as ONE
    kernel (census modes, block 9): the disparity warp of the pattern happens inside the loss kernel's tile loader, so
    pattern_proj and d loss / d es never make a round trip through HBM as separate kernels' outputs and inputs.  The upstream
    gradient of the value is a scalar; autograd's backward is a scalar multiply."""

    @staticmethod
    def forward(ctx, disp, pattern, im, mask, type, eps):
        d = disp.detach().contiguous()
        m = mask.detach().contiguous()
        proj, out, gd, sums = ext_cuda.pattern_similarity(pattern.detach().contiguous(), d, im.detach().contiguous(), m, m, type, eps)
        ctx.save_for_backward(gd, sums)
        ctx.mark_non_differentiable(proj, out)
        return sums[0] / sums[1], proj, out

    @staticmethod
    def backward(ctx, g_val, g_proj, g_map):
        gd, sums = ctx.saved_tensors
        return gd * (g_val / sums[1]), None, None, None, None, None


def pattern_similarity_loss(disp, pattern, im, std=None, loss_type="census_sad", loss_eps=0.5, block_size=9, fused=False):
    """RectifiedPatternSimilarityLoss.tforward (model/networks.py:358-378).  Returns (val, pattern_proj).
    Default: three kernels (warp; fused loss forward + backward + masked mean; in autograd's backward the warp's gradient).
    fused=True (census modes, block 9, CUDA float32 -- the reference's configuration, networks.py:344,376): ONE kernel forward
    + backward (PatternSimilarityFunction).  Measured on B200 at batch 8 x 480x640 (profiles/r02_ops_b8.json): 175 us for
    the one kernel against 164 us for the three -- the tile loader warps 1.7 pixels per output pixel (halo) behind two
    dependent global loads, which costs more than the 27 us of the two stand-alone warp kernels -- so it is not the default."""
    mask = torch.ones_like(im) if std is None else std
    ty = _loss_type_id(loss_type)
    if (fused and ty >= 2 and block_size == 9 and disp.is_cuda and disp.dtype == torch.float32 and disp.dim() == 4 and disp.size(1) == 1
            and disp.size(2) >= 9 and disp.size(3) >= 9):
        val, pattern_proj, _ = PatternSimilarityFunction.apply(disp, pattern, im, mask, ty, loss_eps)
        return val, pattern_proj
    pattern_proj = warp_pattern(pattern, disp)
    val, _ = weighted_photometric_loss(pattern_proj, im.contiguous(), mask, block_size, loss_type, loss_eps)
    return val, pattern_proj


class ProjectionDepthSimilarityFunction(torch.autograd.Function):
    """The geometric loss of the stage-2 trainer, ProjectionDepthSimilarityLoss.tforward (model/networks.py:474-503,
    called per frame pair at model/exp_synphge.py:185-200): unproject, two rigid transforms, projection, bilinear
    sampling of the other frame's depth and the (clamped) absolute difference, both directions.  In the reference
    that is 4 bmm, 2 grid_sample and ~20 elementwise kernels plus their autograd twins; here two launches produce
    the loss and both depth gradients (the upstream gradient of a scalar loss is a scalar, applied in backward).
    Poses, K and the ray table are not differentiated (they are data in the reference)."""

    @staticmethod
    def forward(ctx, depth0, depth1, R0, t0, R1, t1, K, ray, clamp):
        _cuda_only(depth0, "projection_depth_similarity_loss")
        c = lambda t: t.detach().contiguous()
        sums, g0, g1 = ext_cuda.depth_similarity(c(depth0), c(depth1), c(ray), c(K), c(R0), c(t0), c(R1), c(t1), clamp)
        ctx.save_for_backward(g0, g1)
        return sums[0, 0] / sums[0, 1] + sums[1, 0] / sums[1, 1]

    @staticmethod
    def backward(ctx, g):
        g0, g1 = ctx.saved_tensors
        return g0 * g, g1 * g, None, None, None, None, None, None, None


def projection_depth_similarity_loss(depth0, depth1, R0, t0, R1, t1, K, ray, clamp=-1):
    """l0 + l1 of ProjectionDepthSimilarityLoss.tforward(depth0, depth1, R0, t0, R1, t1) (model/networks.py:500-503).
    K [3,3] and ray [H*W,3] are the module's constants (networks.py:421-434: ray = uv1 @ Ki^T in float32)."""
    return ProjectionDepthSimilarityFunction.apply(depth0, depth1, R0, t0, R1, t1, K, ray, clamp)


def projection_rays(Ki, im_height, im_width):
    """The ray table of ProjectionBaseLoss.__init__ (model/networks.py:427-434): pixel centres (u, v, 1) times
    Ki^T, computed in float64 by numpy and stored as float32 [H*W,3]."""
    import numpy as np
    u, v = np.meshgrid(range(im_width), range(im_height))
    uv = np.stack((u, v, np.ones_like(u)), axis=2).reshape(-1, 3)
    ray = uv @ np.asarray(Ki, dtype=np.float64).T if not torch.is_tensor(Ki) else uv @ Ki.cpu().numpy().T
    return torch.from_numpy(ray.reshape(-1, 3).astype(np.float32))


class DisparityLossFunction(torch.autograd.Function):
    """DisparityLoss.tforward (model/networks.py:395-411, called at model/exp_synph.py:116): 5x5 Sobel gradient
    magnitude of the disparity under a two-Laplacian mixture weighted by the edge probability (or, without an edge
    map, its clamped mean).  One kernel computes the loss and the gradients w.r.t. disp and edge; autograd's backward
    is a scalar multiply."""

    @staticmethod
    def forward(ctx, disp, edge):
        _cuda_only(disp, "disparity_loss")
        sums, gd, ge = ext_cuda.disparity_loss(disp.detach().contiguous(), None if edge is None else edge.detach().contiguous())
        ctx.has_edge = edge is not None
        ctx.save_for_backward(gd, ge if ge is not None else gd)
        return sums[0] / sums[1]

    @staticmethod
    def backward(ctx, g):
        gd, ge = ctx.saved_tensors
        return gd * g, (ge * g if ctx.has_edge else None)


def disparity_loss(disp, edge=None):
    """DisparityLoss()(disp, edge) of the reference (model/networks.py:380-412)."""
    return DisparityLossFunction.apply(disp, edge)


class LCNFunction(torch.autograd.Function):
    """Fused local contrast normalisation (model/networks.py:507-533) with its gradient: the forward is one kernel, the
    backward (ctd_lcn_bwd_f32) is what autograd produces through the reference's torch ops for upstream gradients of
    both outputs.  (In the reference the gradient flows to an input image nobody reads, exp_synph.py:80-91.)"""

    @staticmethod
    def forward(ctx, x, radius, epsilon):
        _cuda_only(x, "lcn")
        out, std = ext_cuda.lcn_forward(x, radius, epsilon)
        ctx.radius, ctx.epsilon = radius, epsilon
        if x.dtype == torch.float32 and x.requires_grad:
            ctx.save_for_backward(x.detach(), out, std)
        else:
            ctx.mark_non_differentiable(out, std)
        return out, std

    @staticmethod
    def backward(ctx, g_lcn, g_std):
        x, out, std = ctx.saved_tensors
        gl = None if g_lcn is None else g_lcn.contiguous()
        gs = None if g_std is None else g_std.contiguous()
        return ext_cuda.lcn_backward(x, out, std, gl, gs, ctx.radius, ctx.epsilon), None, None


def lcn(x, radius=5, epsilon=0.05):
    """(x - box_mean) / (box_std + epsilon) over a (2*radius+1)^2 reflection-padded window -> (lcn, std)."""
    return LCNFunction.apply(x, radius, epsilon)


def lcn_normalize(img, kernel_size=4, epsilon=0.01):
    """The data generator's offline LCN, data/lcn/lcn.pyx:16-58 `normalize(img, kernel_size, epsilon)` (called at
    data/create_syn_data.py:182): img [M,N] (or a batch [B,M,N]) -> (img_lcn, img_std), a border of kernel_size pixels left
    at 0, std = sqrt of the centred two-pass variance.  Bit-identical to the Cython build; CUDA tensors only."""
    _cuda_only(img, "lcn_normalize")
    return ext_cuda.lcn_cython(img.contiguous(), kernel_size, epsilon)


def pyramid_pattern_similarity_loss(disps, patterns, ims, stds, loss_type="census_sad", loss_eps=0.5, block_size=9):
    """The photometric part of the trainer's loss_forward (model/exp_synph.py:107-111) over the image pyramid
    (exp_synph.py:25-27: 480x640 halved three times): for every scale s, RectifiedPatternSimilarityLoss(disps[s],
    ims[s], stds[s]) with that scale's pattern (exp_synph.py:62-71).  `patterns` is one [1,1,Hp,Wp] tensor per scale (or
    one tensor used for all).  Returns (vals: list of scalar tensors, pattern_proj of scale 0, detached) as the reference
    keeps them; 3 kernels per scale forward+backward (warp, fused loss + gradient + masked mean, warp gradient), all
    capture-safe, so the whole pyramid replays as one CUDA graph."""
    if torch.is_tensor(patterns):
        patterns = [patterns] * len(disps)
    if not (len(disps) == len(patterns) == len(ims) == len(stds)):
        raise RuntimeError("pyramid_pattern_similarity_loss: one disparity, pattern, image and std per scale")
    vals, proj0 = [], None
    for s, (d, p, im, sd) in enumerate(zip(disps, patterns, ims, stds)):
        val, proj = pattern_similarity_loss(d, p, im, sd, loss_type, loss_eps, block_size)
        if s == 0:
            proj0 = proj.detach()
        vals.append(val)
    return vals, proj0


def masked_mean_terms(diff, mask):
    """(sum(mask*diff), sum(mask)) as a float32 [2] tensor: the two scalars of the caller's
    `(mask*diff).sum() / mask.sum()` (model/networks.py:377); under batch sharding they are what gets
    all-reduced.  Not differentiable (use photometric_loss's own backward with grad_out = mask / sum)."""
    return ext_cuda.masked_sums(diff.detach(), mask.detach())
