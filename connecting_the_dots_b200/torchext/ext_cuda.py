"""The reference's native CUDA entry points, re-bound onto libctd_b200.so.

Mirrors the pybind11 module `ext_cuda` of the reference (torchext/ext/ext_cuda.cpp:126-135): same
function names, argument order and meaning, same Python-visible exception types (RuntimeError for
contiguity / device / shape violations like AT_ASSERTM, NotImplementedError for dtypes other than
float32/float64).  Differences, all deliberate (SURVEY.md section 7, "reference hazards"): outputs are
allocated on the INPUT's device, kernels run on torch's CURRENT stream under a device guard, CUDA
errors raise instead of exit(-1), es/ta shape and K shape are checked, an invalid loss type raises
instead of returning uninitialised memory, xcorrvol also accepts a batched [B,C,H,W] pair, and
photometric_loss_backward overwrites its result (no zero fill, no atomics).
"""
import torch

from .. import _lib

_SUFFIX = {torch.float32: "_f32", torch.float64: "_f64"}


def _check(cond, msg):
    if not cond:
        raise RuntimeError(msg)


def _check_input_cuda(t, name):
    _check(isinstance(t, torch.Tensor), "%s must be a tensor" % name)
    _check(t.is_cuda, "%s must be a CUDA tensor" % name)
    _check(t.is_contiguous(), "%s must be contiguous" % name)


def _real_suffix(t, op):
    try:
        return _SUFFIX[t.dtype]
    except KeyError:
        raise NotImplementedError('"%s" not implemented for \'%s\'' % (op, str(t.dtype).replace("torch.", "").capitalize()))


def _same(a, b, na, nb):
    _check(a.dtype == b.dtype, "%s and %s must have the same dtype" % (na, nb))
    _check(a.device == b.device, "%s and %s must be on the same device" % (na, nb))


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _image_pair(in0, in1, op):
    """Checks of an image pair [C,H,W] or [B,C,H,W]: (dtype suffix, B, C, H, W, batched)."""
    _check_input_cuda(in0, "in0")
    _check_input_cuda(in1, "in1")
    _check(in0.dim() in (3, 4), "in0 has to be C x H x W (or B x C x H x W)")
    _check(tuple(in0.shape) == tuple(in1.shape), "in0 and in1 have to be the same shape")
    _same(in0, in1, "in0", "in1")
    sfx = _real_suffix(in0, op)
    batched = in0.dim() == 4
    C, H, W = in0.shape[-3:]
    return sfx, in0.size(0) if batched else 1, C, H, W, batched


def _maps(ref, B, H, W, batched, dtype=None):
    """One per-pixel output map on ref's device, [B,1,H,W] (or [1,H,W]), in ref's dtype unless one is given."""
    return torch.empty((B, 1, H, W) if batched else (1, H, W), dtype=dtype or ref.dtype, device=ref.device)


def nn_cuda(in0, in1):
    """ext_cuda.cpp:9-26.  in0 [N0,3], in1 [N1,3] -> int64 [N0] nearest-neighbour indices (or -1)."""
    _check_input_cuda(in0, "in0")
    _check_input_cuda(in1, "in1")
    _check(in0.dim() == 2, "in0 has to be N0 x 3")
    _check(in1.dim() == 2, "in1 has to be N1 x 3")
    _check(in0.size(1) == in1.size(1), "in0 and in1 have to be the same shape")
    _check(in0.size(1) == 3, "dim hast to be 3")
    _same(in0, in1, "in0", "in1")
    sfx = _real_suffix(in0, "nn")
    out = torch.empty((in0.size(0),), dtype=torch.int64, device=in0.device)
    with torch.cuda.device(in0.device):
        _lib.call("ctd_nn" + sfx, in0.data_ptr(), in1.data_ptr(), out.data_ptr(), in0.size(0), in1.size(0), _stream(in0))
    return out


def crosscheck_cuda(in0, in1):
    """ext_cuda.cpp:31-43.  in0 int64 [N0], in1 int64 [N1] -> uint8 [N0] mutual-consistency mask."""
    _check_input_cuda(in0, "in0")
    _check_input_cuda(in1, "in1")
    _check(in0.dim() == 1, "in0 has to be 1-D")
    _check(in1.dim() == 1, "in1 has to be 1-D")
    _check(in0.dtype == torch.int64 and in1.dtype == torch.int64, "crosscheck expects int64 index tensors")
    _check(in0.device == in1.device, "in0 and in1 must be on the same device")
    out = torch.empty((in0.size(0),), dtype=torch.uint8, device=in0.device)
    with torch.cuda.device(in0.device):
        _lib.call("ctd_crosscheck", in0.data_ptr(), in1.data_ptr(), out.data_ptr(), in0.size(0), in1.size(0), _stream(in0))
    return out


def proj_nn_cuda(xyz0, xyz1, K, patch_size):
    """ext_cuda.cpp:47-69.  xyz0, xyz1 [B,H,W,3], K [3,3] -> int64 [B,H,W] flat indices into xyz1 (or -1)."""
    _check_input_cuda(xyz0, "xyz0")
    _check_input_cuda(xyz1, "xyz1")
    _check_input_cuda(K, "K")
    _check(xyz0.dim() == 4 and xyz1.dim() == 4, "xyz0 and xyz1 have to be B x H x W x 3")
    _check(tuple(xyz0.shape) == tuple(xyz1.shape), "xyz0 and xyz1 have to be the same shape")
    _check(xyz0.size(3) == 3, "last dimension has to be 3")
    _check(K.numel() == 9, "K has to be 3 x 3")
    _same(xyz0, xyz1, "xyz0", "xyz1")
    _same(xyz0, K, "xyz0", "K")
    sfx = _real_suffix(xyz0, "proj_nn")
    B, H, W = xyz0.shape[:3]
    out = torch.empty((B, H, W), dtype=torch.int64, device=xyz0.device)
    with torch.cuda.device(xyz0.device):
        _lib.call("ctd_proj_nn" + sfx, xyz0.data_ptr(), xyz1.data_ptr(), K.data_ptr(), out.data_ptr(), B, H, W,
                  int(patch_size), _stream(xyz0))
    return out


def xcorrvol_cuda(in0, in1, n_disps, block_size):
    """ext_cuda.cpp:73-86.  in0, in1 [C,H,W] -> [n_disps,H,W]; batched: [B,C,H,W] -> [B,n_disps,H,W]."""
    sfx, B, C, H, W, batched = _image_pair(in0, in1, "xcorrvol")
    out = torch.empty((B, int(n_disps), H, W) if batched else (int(n_disps), H, W), dtype=in0.dtype, device=in0.device)
    with torch.cuda.device(in0.device):
        _lib.call("ctd_xcorrvol" + sfx, in0.data_ptr(), in1.data_ptr(), out.data_ptr(), B, C, H, W, int(n_disps),
                  int(block_size), _stream(in0))
    return out


def xcorr_disparity_cuda(in0, in1, n_disps, block_size, subpixel=True):
    """Winner-take-all disparity of xcorrvol_cuda's volume without writing it (ctd_xcorr_disparity_*).  in0, in1 [C,H,W]
    -> (disp, score) [1,H,W]; batched: [B,C,H,W] -> [B,1,H,W]."""
    sfx, B, C, H, W, batched = _image_pair(in0, in1, "xcorr_disparity")
    disp, score = _maps(in0, B, H, W, batched), _maps(in0, B, H, W, batched)
    with torch.cuda.device(in0.device):
        _lib.call("ctd_xcorr_disparity" + sfx, in0.data_ptr(), in1.data_ptr(), disp.data_ptr(), score.data_ptr(), B, C, H, W,
                  int(n_disps), int(block_size), int(bool(subpixel)), _stream(in0))
    return disp, score


def sgm_cuda(vol, p1, p2, paths=8, subpixel=True, want_disparity=True):
    """Semi-global matching over a score volume (ctd_sgm_*).  vol [B,D,H,W] (or [D,H,W]) -> (agg, disp, score): agg like
    vol, disp and score [B,1,H,W] (or [1,H,W]), or None without want_disparity."""
    _check_input_cuda(vol, "vol")
    _check(vol.dim() in (3, 4), "vol has to be D x H x W (or B x D x H x W)")
    sfx = _real_suffix(vol, "sgm")
    batched = vol.dim() == 4
    B = vol.size(0) if batched else 1
    D, H, W = vol.shape[-3:]
    agg = torch.empty_like(vol)
    disp = score = None
    if want_disparity:
        disp, score = _maps(vol, B, H, W, batched), _maps(vol, B, H, W, batched)
    with torch.cuda.device(vol.device):
        _lib.call("ctd_sgm" + sfx, vol.data_ptr(), agg.data_ptr(), disp.data_ptr() if want_disparity else None,
                  score.data_ptr() if want_disparity else None, B, D, H, W, float(p1), float(p2), int(paths),
                  int(bool(subpixel)), _stream(vol))
    return agg, disp, score


def disparity_check_cuda(vol, max_diff=1, uniqueness=0.0, subpixel=True):
    """Left-right consistency and uniqueness checks over a score volume (ctd_disparity_check_*).  vol [B,D,H,W] (or
    [D,H,W]) -> (disp, score, valid), [B,1,H,W] (or [1,H,W]); valid is torch.bool."""
    _check_input_cuda(vol, "vol")
    _check(vol.dim() in (3, 4), "vol has to be D x H x W (or B x D x H x W)")
    sfx = _real_suffix(vol, "disparity_check")
    batched = vol.dim() == 4
    B = vol.size(0) if batched else 1
    D, H, W = vol.shape[-3:]
    disp, score, valid = _maps(vol, B, H, W, batched), _maps(vol, B, H, W, batched), _maps(vol, B, H, W, batched, torch.bool)
    with torch.cuda.device(vol.device):
        _lib.call("ctd_disparity_check" + sfx, vol.data_ptr(), disp.data_ptr(), score.data_ptr(), None, None, valid.data_ptr(),
                  B, D, H, W, int(max_diff), float(uniqueness), int(bool(subpixel)), _stream(vol))
    return disp, score, valid


def speckle_filter_cuda(disp, valid, max_size, max_diff):
    """Speckle filter of a disparity map (ctd_speckle_filter_*).  disp [B,1,H,W] (or [1,H,W]), valid None or bool of the
    same shape -> valid_out, torch.bool of disp's shape."""
    _check_input_cuda(disp, "disp")
    _check(disp.dim() in (3, 4) and disp.size(-3) == 1, "disp has to be 1 x H x W (or B x 1 x H x W)")
    sfx = _real_suffix(disp, "speckle_filter")
    if valid is not None:
        _check_input_cuda(valid, "valid")
        _check(valid.dtype == torch.bool and tuple(valid.shape) == tuple(disp.shape), "valid has to be a bool tensor of disp's shape")
        _check(valid.device == disp.device, "disp and valid must be on the same device")
    H, W = disp.shape[-2:]
    out = torch.empty(disp.shape, dtype=torch.bool, device=disp.device)
    with torch.cuda.device(disp.device):
        _lib.call("ctd_speckle_filter" + sfx, disp.data_ptr(), None if valid is None else valid.data_ptr(), out.data_ptr(),
                  disp.size(0) if disp.dim() == 4 else 1, H, W, int(max_size), float(max_diff), _stream(disp))
    return out


def census_transform_cuda(x, wh, ww):
    """Census transform (ctd_census_transform_*): x [B,C,H,W] (or [C,H,W]) -> int64 of the same shape holding the uint64
    bit patterns."""
    _check_input_cuda(x, "x")
    _check(x.dim() in (3, 4), "x has to be C x H x W (or B x C x H x W)")
    sfx = _real_suffix(x, "census_transform")
    B, C, H, W = x.shape if x.dim() == 4 else (1,) + tuple(x.shape)
    out = torch.empty(x.shape, dtype=torch.int64, device=x.device)
    with torch.cuda.device(x.device):
        _lib.call("ctd_census_transform" + sfx, x.data_ptr(), out.data_ptr(), B, C, H, W, int(wh), int(ww), _stream(x))
    return out


def census_vol_cuda(in0, in1, n_disps, wh, ww, block_size):
    """Census matching-score volume (ctd_census_vol_*): in0, in1 [B,C,H,W] -> [B,n_disps,H,W] (or [C,H,W] ->
    [n_disps,H,W]), in the inputs' dtype."""
    sfx, B, C, H, W, batched = _image_pair(in0, in1, "census_vol")
    out = torch.empty((B, int(n_disps), H, W) if batched else (int(n_disps), H, W), dtype=in0.dtype, device=in0.device)
    with torch.cuda.device(in0.device):
        _lib.call("ctd_census_vol" + sfx, in0.data_ptr(), in1.data_ptr(), out.data_ptr(), B, C, H, W, int(n_disps), int(wh),
                  int(ww), int(block_size), _stream(in0))
    return out


def census_disparity_cuda(in0, in1, n_disps, wh, ww, block_size, subpixel=True):
    """Winner-take-all disparity of census_vol_cuda's volume without writing it (ctd_census_disparity_*): (disp, score),
    [B,1,H,W] (or [1,H,W])."""
    sfx, B, C, H, W, batched = _image_pair(in0, in1, "census_disparity")
    disp, score = _maps(in0, B, H, W, batched), _maps(in0, B, H, W, batched)
    with torch.cuda.device(in0.device):
        _lib.call("ctd_census_disparity" + sfx, in0.data_ptr(), in1.data_ptr(), disp.data_ptr(), score.data_ptr(), B, C, H, W,
                  int(n_disps), int(wh), int(ww), int(block_size), int(bool(subpixel)), _stream(in0))
    return disp, score


def _photometric_args(es, ta, type):
    _check_input_cuda(es, "es")
    _check_input_cuda(ta, "ta")
    _check(es.dim() == 4, "es has to be B x C x H x W")
    _check(tuple(es.shape) == tuple(ta.shape), "es and ta have to be the same shape")
    _same(es, ta, "es", "ta")
    _check(int(type) in (0, 1, 2, 3), "invalid loss type")
    return _real_suffix(es, "photometric_loss")


def photometric_loss_forward(es, ta, block_size, type, eps):
    """ext_cuda.cpp:92-104.  es, ta [B,C,H,W] -> [B,1,H,W]; type 0 mse, 1 sad, 2 census_mse, 3 census_sad."""
    sfx = _photometric_args(es, ta, type)
    B, C, H, W = es.shape
    out = torch.empty((B, 1, H, W), dtype=es.dtype, device=es.device)
    with torch.cuda.device(es.device):
        _lib.call("ctd_photometric_fwd" + sfx, es.data_ptr(), ta.data_ptr(), out.data_ptr(), B, C, H, W,
                  int(block_size), int(type), float(eps), _stream(es))
    return out


def photometric_loss_backward(es, ta, grad_out, block_size, type, eps):
    """ext_cuda.cpp:109-123.  grad_out [B,1,H,W] -> gradient w.r.t. es, [B,C,H,W]."""
    sfx = _photometric_args(es, ta, type)
    _check_input_cuda(grad_out, "grad_out")
    B, C, H, W = es.shape
    _check(grad_out.numel() == B * H * W, "grad_out has to be B x 1 x H x W")
    _same(es, grad_out, "es", "grad_out")
    grad_in = torch.empty((B, C, H, W), dtype=es.dtype, device=es.device)
    with torch.cuda.device(es.device):
        _lib.call("ctd_photometric_bwd" + sfx, es.data_ptr(), ta.data_ptr(), grad_out.data_ptr(), grad_in.data_ptr(),
                  B, C, H, W, int(block_size), int(type), float(eps), _stream(es))
    return grad_in


def photometric_loss_forward_backward(es, ta, grad_out, block_size, type, eps):
    """Both halves in one call (ctd_photometric_fwd_bwd_f32; the census modes run a single fused kernel).
    Returns (loss map [B,1,H,W], gradient w.r.t. es [B,C,H,W]); fp32 only."""
    _photometric_args(es, ta, type)
    _check(es.dtype == torch.float32, "photometric_loss_forward_backward is float32 only")
    _check_input_cuda(grad_out, "grad_out")
    B, C, H, W = es.shape
    _check(grad_out.numel() == B * H * W, "grad_out has to be B x 1 x H x W")
    _same(es, grad_out, "es", "grad_out")
    out = torch.empty((B, 1, H, W), dtype=es.dtype, device=es.device)
    grad_in = torch.empty((B, C, H, W), dtype=es.dtype, device=es.device)
    with torch.cuda.device(es.device):
        _lib.call("ctd_photometric_fwd_bwd_f32", es.data_ptr(), ta.data_ptr(), grad_out.data_ptr(), out.data_ptr(),
                  grad_in.data_ptr(), B, C, H, W, int(block_size), int(type), float(eps), _stream(es))
    return out, grad_in


def photometric_loss_forward_backward_masked(es, ta, grad_out, mask, block_size, type, eps):
    """photometric_loss_forward_backward plus sums = (sum(mask * loss), sum(mask)) from the same kernels
    (ctd_photometric_fwd_bwd_masked_f32).  Returns (loss map, gradient w.r.t. es, sums float32 [2])."""
    _photometric_args(es, ta, type)
    _check(es.dtype == torch.float32, "photometric_loss_forward_backward_masked is float32 only")
    _check_input_cuda(grad_out, "grad_out")
    _check_input_cuda(mask, "mask")
    B, C, H, W = es.shape
    _check(grad_out.numel() == B * H * W and mask.numel() == B * H * W, "grad_out and mask have to be B x 1 x H x W")
    _check(mask.dtype == torch.float32 and grad_out.dtype == torch.float32, "grad_out and mask have to be float32")
    _same(es, grad_out, "es", "grad_out")
    _same(es, mask, "es", "mask")
    out = torch.empty((B, 1, H, W), dtype=es.dtype, device=es.device)
    grad_in = torch.empty((B, C, H, W), dtype=es.dtype, device=es.device)
    sums = torch.empty(2, dtype=torch.float32, device=es.device)
    with torch.cuda.device(es.device):
        _lib.call("ctd_photometric_fwd_bwd_masked_f32", es.data_ptr(), ta.data_ptr(), grad_out.data_ptr(), mask.data_ptr(),
                  out.data_ptr(), grad_in.data_ptr(), sums.data_ptr(), B, C, H, W, int(block_size), int(type), float(eps), _stream(es))
    return out, grad_in, sums


def _ssim_args(es, ta):
    _check_input_cuda(es, "es")
    _check_input_cuda(ta, "ta")
    _check(es.dim() == 4, "es has to be B x C x H x W")
    _check(tuple(es.shape) == tuple(ta.shape), "es and ta have to be the same shape")
    _same(es, ta, "es", "ta")
    return _real_suffix(es, "ssim_loss")


def _ssim_grad_out(es, grad_out):
    _check_input_cuda(grad_out, "grad_out")
    B, C, H, W = es.shape
    _check(grad_out.numel() == B * H * W, "grad_out has to be B x 1 x H x W")
    _same(es, grad_out, "es", "grad_out")


def ssim_forward(es, ta, block_size, c1, c2):
    """SSIM loss map (ctd_ssim_fwd_*): es, ta [B,C,H,W] -> [B,1,H,W] = sum over channels of (1 - SSIM) / 2 over the
    replicate-clamped block_size^2 window of photometric_loss."""
    sfx = _ssim_args(es, ta)
    B, C, H, W = es.shape
    out = torch.empty((B, 1, H, W), dtype=es.dtype, device=es.device)
    with torch.cuda.device(es.device):
        _lib.call("ctd_ssim_fwd" + sfx, es.data_ptr(), ta.data_ptr(), out.data_ptr(), B, C, H, W, int(block_size),
                  float(c1), float(c2), _stream(es))
    return out


def ssim_backward(es, ta, grad_out, block_size, c1, c2):
    """Gradient of ssim_forward w.r.t. es for grad_out [B,1,H,W] -> [B,C,H,W] (ctd_ssim_bwd_*)."""
    sfx = _ssim_args(es, ta)
    _ssim_grad_out(es, grad_out)
    B, C, H, W = es.shape
    grad_in = torch.empty((B, C, H, W), dtype=es.dtype, device=es.device)
    with torch.cuda.device(es.device):
        _lib.call("ctd_ssim_bwd" + sfx, es.data_ptr(), ta.data_ptr(), grad_out.data_ptr(), grad_in.data_ptr(), B, C, H, W,
                  int(block_size), float(c1), float(c2), _stream(es))
    return grad_in


def ssim_forward_backward_masked(es, ta, grad_out, mask, block_size, c1, c2):
    """Loss map, gradient w.r.t. es and sums = (sum(mask * loss), sum(mask)) from one pass
    (ctd_ssim_fwd_bwd_masked_f32).  Returns (loss map [B,1,H,W], gradient [B,C,H,W], sums float32 [2]); fp32 only."""
    _ssim_args(es, ta)
    _check(es.dtype == torch.float32, "ssim_forward_backward_masked is float32 only")
    _ssim_grad_out(es, grad_out)
    _check_input_cuda(mask, "mask")
    B, C, H, W = es.shape
    _check(mask.numel() == B * H * W, "mask has to be B x 1 x H x W")
    _check(mask.dtype == torch.float32, "mask has to be float32")
    _same(es, mask, "es", "mask")
    out = torch.empty((B, 1, H, W), dtype=es.dtype, device=es.device)
    grad_in = torch.empty((B, C, H, W), dtype=es.dtype, device=es.device)
    sums = torch.empty(2, dtype=torch.float32, device=es.device)
    with torch.cuda.device(es.device):
        _lib.call("ctd_ssim_fwd_bwd_masked_f32", es.data_ptr(), ta.data_ptr(), grad_out.data_ptr(), mask.data_ptr(),
                  out.data_ptr(), grad_in.data_ptr(), sums.data_ptr(), B, C, H, W, int(block_size), float(c1), float(c2),
                  _stream(es))
    return out, grad_in, sums


def _warp_args(pattern, disp):
    _check_input_cuda(pattern, "pattern")
    _check_input_cuda(disp, "disp")
    _check(pattern.dim() == 4 and pattern.size(1) == 1, "pattern has to be Bp x 1 x Hp x Wp")
    _check(disp.dim() == 4 and disp.size(1) == 1, "disp has to be B x 1 x H x W")
    _check(pattern.size(0) in (1, disp.size(0)), "pattern batch has to be 1 or the batch of disp")
    _check(pattern.dtype == torch.float32 and disp.dtype == torch.float32, "warp_pattern is float32 only")
    _same(pattern, disp, "pattern", "disp")


def warp_pattern_forward(pattern, disp):
    """model/networks.py:362-371: grid_sample(pattern, grid(disp), padding_mode='border') -> [B,1,H,W]."""
    _warp_args(pattern, disp)
    B, _, H, W = disp.shape
    Bp, _, Hp, Wp = pattern.shape
    out = torch.empty_like(disp)
    with torch.cuda.device(disp.device):
        _lib.call("ctd_warp_pattern_fwd_f32", pattern.data_ptr(), disp.data_ptr(), out.data_ptr(), B, Bp, Hp, Wp, H, W, _stream(disp))
    return out


def warp_pattern_backward(pattern, disp, grad_out):
    """Gradient of warp_pattern_forward w.r.t. disp."""
    _warp_args(pattern, disp)
    _check_input_cuda(grad_out, "grad_out")
    _check(grad_out.numel() == disp.numel() and grad_out.dtype == torch.float32, "grad_out has to match disp")
    B, _, H, W = disp.shape
    Bp, _, Hp, Wp = pattern.shape
    gd = torch.empty_like(disp)
    with torch.cuda.device(disp.device):
        _lib.call("ctd_warp_pattern_bwd_f32", pattern.data_ptr(), disp.data_ptr(), grad_out.data_ptr(), gd.data_ptr(), B, Bp, Hp, Wp,
                  H, W, _stream(disp))
    return gd


def pattern_similarity(pattern, disp, ta, grad_out, mask, type, eps):
    """model/networks.py:358-378 as ONE kernel (ctd_pattern_similarity_f32; census modes, block 9): returns (pattern_proj,
    loss map, d loss / d disp for grad_out, sums float32 [2] = (sum(mask * loss), sum(mask)))."""
    _warp_args(pattern, disp)
    for t, n in ((ta, "ta"), (grad_out, "grad_out"), (mask, "mask")):
        _check_input_cuda(t, n)
        _check(t.dtype == torch.float32 and t.numel() == disp.numel(), n + " has to be float32 and match disp")
        _same(disp, t, "disp", n)
    B, _, H, W = disp.shape
    Bp, _, Hp, Wp = pattern.shape
    proj, out, gd = torch.empty_like(disp), torch.empty_like(disp), torch.empty_like(disp)
    sums = torch.empty(2, dtype=torch.float32, device=disp.device)
    with torch.cuda.device(disp.device):
        _lib.call("ctd_pattern_similarity_f32", pattern.data_ptr(), disp.data_ptr(), ta.data_ptr(), grad_out.data_ptr(), mask.data_ptr(),
                  proj.data_ptr(), out.data_ptr(), gd.data_ptr(), sums.data_ptr(), B, Bp, Hp, Wp, H, W, int(type), float(eps), _stream(disp))
    return proj, out, gd, sums


def depth_similarity(depth0, depth1, ray, K, R0, t0, R1, t1, clamp=-1.0):
    """model/networks.py:500-503 (ProjectionDepthSimilarityLoss.tforward): both directions of the projected depth
    difference, loss sums and gradients in two kernels.  depth0/1 [B,1,H,W]; ray [H*W,3] or [1,H*W,3]; K [3,3] or
    [1,3,3]; R0/R1 [B,3,3]; t0/t1 [B,3].  Returns (sums [2,2] = per direction {sum diff, pixel count},
    grad_depth0, grad_depth1) with the gradients of l0 + l1 (each a mean over B*H*W)."""
    for t, name in ((depth0, "depth0"), (depth1, "depth1"), (ray, "ray"), (K, "K"), (R0, "R0"), (t0, "t0"), (R1, "R1"), (t1, "t1")):
        _check_input_cuda(t, name)
        _check(t.dtype == torch.float32, "depth_similarity is float32 only")
        _same(depth0, t, "depth0", name)
    _check(depth0.dim() == 4 and depth0.size(1) == 1, "depth0 has to be B x 1 x H x W")
    _check(depth1.shape == depth0.shape, "depth0 and depth1 have to have the same shape")
    B, _, H, W = depth0.shape
    _check(ray.numel() == H * W * 3, "ray has to be H*W x 3")
    _check(K.numel() == 9, "K has to be 3 x 3")
    _check(R0.numel() == B * 9 and R1.numel() == B * 9, "R0, R1 have to be B x 3 x 3")
    _check(t0.numel() == B * 3 and t1.numel() == B * 3, "t0, t1 have to be B x 3")
    sums = torch.empty(2, 2, dtype=torch.float32, device=depth0.device)
    g0 = torch.empty_like(depth0)
    g1 = torch.zeros_like(depth1)
    scale = 1.0 / max(B * H * W, 1)
    with torch.cuda.device(depth0.device):
        st = _stream(depth0)
        # direction 0 -> 1: g0 gets every pixel's own gradient (store), g1 the bilinear scatter (atomics on zeros)
        _lib.call("ctd_depth_similarity_f32", depth0.data_ptr(), depth1.data_ptr(), ray.data_ptr(), K.data_ptr(), R0.data_ptr(),
                  t0.data_ptr(), R1.data_ptr(), t1.data_ptr(), g0.data_ptr(), g1.data_ptr(), sums[0].data_ptr(), B, H, W,
                  float(clamp), scale, 0, st)
        # direction 1 -> 0: roles swapped, own gradients are added to g1, the scatter lands on g0
        _lib.call("ctd_depth_similarity_f32", depth1.data_ptr(), depth0.data_ptr(), ray.data_ptr(), K.data_ptr(), R1.data_ptr(),
                  t1.data_ptr(), R0.data_ptr(), t0.data_ptr(), g1.data_ptr(), g0.data_ptr(), sums[1].data_ptr(), B, H, W,
                  float(clamp), scale, 1, st)
    return sums, g0, g1


def disparity_loss(disp, edge=None):
    """model/networks.py:395-411 (DisparityLoss.tforward) in one kernel.  disp [B,1,H,W]; edge [B,1,H,W] or None.
    Returns (sums [2] = {sum of the per-pixel loss, pixel count}, grad_disp, grad_edge or None) with the gradients
    of the mean."""
    _check_input_cuda(disp, "disp")
    _check(disp.dim() == 4 and disp.size(1) == 1, "disp has to be B x 1 x H x W")
    _check(disp.dtype == torch.float32, "disparity_loss is float32 only")
    if edge is not None:
        _check_input_cuda(edge, "edge")
        _check(edge.shape == disp.shape and edge.dtype == torch.float32, "edge has to match disp")
        _same(disp, edge, "disp", "edge")
    B, _, H, W = disp.shape
    sums = torch.empty(2, dtype=torch.float32, device=disp.device)
    gd = torch.empty_like(disp)
    ge = torch.empty_like(disp) if edge is not None else None
    with torch.cuda.device(disp.device):
        _lib.call("ctd_disparity_loss_f32", disp.data_ptr(), edge.data_ptr() if edge is not None else 0, gd.data_ptr(),
                  ge.data_ptr() if ge is not None else 0, sums.data_ptr(), B, H, W, 1.0 / max(B * H * W, 1), _stream(disp))
    return sums, gd, ge


def lcn_forward(x, radius, epsilon):
    """model/networks.py:523-533 as one kernel.  x [N,1,H,W] -> (lcn, std), both [N,1,H,W]."""
    _check_input_cuda(x, "x")
    _check(x.dim() == 4 and x.size(1) == 1, "x has to be N x 1 x H x W")
    sfx = _real_suffix(x, "lcn")
    N, _, H, W = x.shape
    out = torch.empty_like(x)
    std = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.call("ctd_lcn" + sfx, x.data_ptr(), out.data_ptr(), std.data_ptr(), N, H, W, int(radius), float(epsilon),
                  _stream(x))
    return out, std


def lcn_backward(x, lcn, std, grad_lcn, grad_std, radius, epsilon):
    """Gradient of model/networks.py:523-533 w.r.t. its input (what autograd produces through the reference's torch
    ops), from the forward's input and outputs and the upstream gradients of (lcn, std); either gradient may be None.
    float32, [N,1,H,W]."""
    for t, n in ((x, "x"), (lcn, "lcn"), (std, "std")):
        _check_input_cuda(t, n)
        _check(t.dtype == torch.float32, "lcn_backward is float32 only")
    _check(x.dim() == 4 and x.size(1) == 1 and lcn.shape == x.shape and std.shape == x.shape, "x, lcn, std have to be N x 1 x H x W")
    for t, n in ((grad_lcn, "grad_lcn"), (grad_std, "grad_std")):
        if t is not None:
            _check_input_cuda(t, n)
            _check(t.shape == x.shape and t.dtype == torch.float32, n + " has to match x")
    N, _, H, W = x.shape
    gx = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.call("ctd_lcn_bwd_f32", x.data_ptr(), lcn.data_ptr(), std.data_ptr(), 0 if grad_lcn is None else grad_lcn.data_ptr(),
                  0 if grad_std is None else grad_std.data_ptr(), gx.data_ptr(), N, H, W, int(radius), float(epsilon), _stream(x))
    return gx


def lcn_cython(img, kernel_size, epsilon):
    """data/lcn/lcn.pyx:16-58 `normalize` for one image [M,N] or a batch [B,M,N]: (lcn, std), zeros in the border."""
    _check_input_cuda(img, "img")
    _check(img.dtype == torch.float32 and img.dim() in (2, 3), "img has to be float32 [M,N] or [B,M,N]")
    B = 1 if img.dim() == 2 else img.size(0)
    M, N = img.shape[-2:]
    out, std = torch.empty_like(img), torch.empty_like(img)
    with torch.cuda.device(img.device):
        _lib.call("ctd_lcn_cython_f32", img.data_ptr(), out.data_ptr(), std.data_ptr(), B, M, N, int(kernel_size), float(epsilon), _stream(img))
    return out, std


_reduce_ws = {}


def masked_sums(diff, mask):
    """model/networks.py:377 numerator and denominator in one deterministic kernel:
    returns float32 [2] = (sum(mask * diff), sum(mask)).  val = r[0] / r[1]."""
    _check_input_cuda(diff, "diff")
    _check_input_cuda(mask, "mask")
    _check(diff.dtype == torch.float32 and mask.dtype == torch.float32, "masked_sums expects float32")
    _check(diff.numel() == mask.numel(), "diff and mask have to be the same size")
    _same(diff, mask, "diff", "mask")
    key = (diff.device, torch.cuda.current_stream(diff.device).cuda_stream)
    ws = _reduce_ws.get(key)
    if ws is None:
        ws = _reduce_ws[key] = torch.zeros(int(_lib.lib().ctd_masked_sums_workspace_bytes()), dtype=torch.uint8, device=diff.device)
    out = torch.empty(2, dtype=torch.float32, device=diff.device)
    with torch.cuda.device(diff.device):
        _lib.call("ctd_masked_sums_f32", diff.data_ptr(), mask.data_ptr(), diff.numel(), out.data_ptr(), ws.data_ptr(), _stream(diff))
    return out
