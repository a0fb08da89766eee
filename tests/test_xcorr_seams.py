"""GPU tests of XCorrVol and its fused disparity at their dispatch seams (-m gpu).

xcorrvol.cu cuts a call of either op into separable launches of at most xcorr_images_per_launch(D, H, W) images (the
hit-list bound, gridDim.z = images x disparity chunks <= 65535, window-statistics positions < 2^31) and moves the input,
volume, disparity and score pointers with each launch.  Only an image that one launch cannot take alone leaves the
separable path: the volume then runs xcorrvol_direct (chunks of 1024 images) or xcorrvol_generic, the disparity
xcorr_disparity_generic.  The other GPU tests stay at batch 8 or less, inside one launch.  These tests run each split and
each fallback at legal sizes and check:
  * the volume against the C oracle, on the images at every launch boundary (full-width bands of rows, the image's top
    and bottom rows among them, or whole images where they are small);
  * the disparity against disparity_from_volume(volume) under the contract of include/ctd_b200.h: d* and the score
    bit-equal where both ops take the same path, the sub-pixel offset within what the header's ~1e-5 on the
    re-evaluated scores allows;
  * where the batch is split, every image's volume, disparity and score bit-equal to a call on that image alone (one
    launch): the cheapest full check of the per-launch pointer arithmetic.
Each test records its kernels and asserts which of them ran with which grid.z per launch; where the profiler's trace
misses launches, only that assertion is skipped.
"""
import functools
import math

import pytest
import torch

import oracle
from conftest import assert_close
from test_dispatch_seams import _expect, _expect_chunks, _grids, _kernels, _seen

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

XS_DT, XD_DC, ST_H = 16, 32, 16      # xcorrvol.cu: disparities per separable CTA, per direct CTA; statistics tile rows
HIT_OUTPUTS = ((1 << 24) - 1024) * 32  # outputs per launch that keep the fix-up's hit list at 1/32 of them
SEP, DIRECT, GENERIC = "xcorr_sep_kernel", "xcorrvol_direct", "xcorrvol_generic"
DGENERIC, FINISH = "xcorr_disparity_generic", "xcorr_wta_finish_kernel"
KERNELS = (SEP, DIRECT, GENERIC, DGENERIC, FINISH)
EPS = 1e-5  # include/ctd_b200.h: the fused path's sub-pixel scores are within ~1e-5 of the volume's


def cdiv(a, b):
    return -(-a // b)


def images_per_launch(D, H, W):
    """xcorr_images_per_launch: the hit-list bound, gridDim.z <= 65535, statistics positions < 2^31."""
    ws1 = cdiv(D, XS_DT) * XS_DT + cdiv(W, 4) * 4
    return max(1, min(HIT_OUTPUTS // (D * H * W), 65535 // cdiv(D, XS_DT), (2 ** 31 - 1) // (H * ws1)))


def _lib():
    from connecting_the_dots_b200 import _lib
    return _lib


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _option(name, value):
    _lib().set_option(name, value)


def _boundaries(B, nb):
    """First and last image of every launch of at most nb images."""
    return sorted({i for b0 in range(0, B, nb) for i in (b0, min(b0 + nb, B) - 1)})


# ---------------------------------------------------------------- inputs
@functools.lru_cache(maxsize=1)
def _full_batch(B):
    """synth.make_batch(B): the synthetic LCN'd pair, eight frames and row-rolled copies, every image distinct."""
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(B)
    return d["ta"], d["pat_lcn"]


def _tiled(B, H, W, step):
    """[B,1,H,W] pairs on the device cut from one flattened synthetic LCN'd frame, image n starting `step * n` values
    further on: distinct images with the frame's flat and textured windows."""
    from connecting_the_dots_b200 import synth
    d = synth.make_pair(0)
    src = [torch.from_numpy(d[k].ravel()).to(DEV) for k in ("ta", "pat_lcn")]
    out = [torch.empty(B, 1, H, W, device=DEV) for _ in src]
    pos = torch.arange(H * W, device=DEV)
    chunk = max(1, (1 << 25) // (H * W))
    for b0 in range(0, B, chunk):
        n = torch.arange(b0, min(b0 + chunk, B), device=DEV)
        idx = (pos[None] + step * n[:, None]) % src[0].numel()
        for s, o in zip(src, out):
            o[b0:b0 + len(n)] = s[idx].view(-1, 1, H, W)
    return out


# ---------------------------------------------------------------- checks
def _oracle_band(a, b, D, bs, r0, r1):
    """oracle.xcorrvol rows r0..r1-1 of one image pair a, b [H,W] (numpy), from the oracle run on the band plus bs // 2
    rows of context above and below: windows clamp only at the image's own top and bottom rows, so this is exact."""
    R, H = bs // 2, a.shape[0]
    lo, hi = max(r0 - R, 0), min(r1 + R, H)
    return oracle.xcorrvol(a[None, lo:hi], b[None, lo:hi], D, bs)[:, r0 - lo:r1 - lo]


def _check_oracle(vol, a, b, D, bs, images, rows, what):
    """vol[n] (device) against the oracle for every image n in `images`, on the row bands `rows` ((r0, r1) pairs);
    a, b: the inputs, [B,1,H,W] numpy arrays or device tensors."""
    for n in images:
        an, bn = (x[n, 0].cpu().numpy() if torch.is_tensor(x) else x[n, 0] for x in (a, b))
        for r0, r1 in rows:
            assert_close(vol[n, :, r0:r1].cpu().numpy(), _oracle_band(an, bn, D, bs, r0, r1),
                         what="%s: image %d rows %d..%d" % (what, n, r0, r1 - 1))


def _wta(vol, subpixel):
    """disparity_from_volume(vol) in chunks of images (the definition is per pixel; this bounds its temporaries)."""
    from connecting_the_dots_b200.torchext import functions as F
    chunk = max(1, (1 << 26) // vol[0].numel())
    parts = [F.disparity_from_volume(vol[i:i + chunk], subpixel) for i in range(0, vol.size(0), chunk)]
    return torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts])


def _equal(got, ref, what):
    bad = int((got != ref).sum())
    assert bad == 0, "%s: %d of %d values differ, max |diff| %.3e" % (what, bad, got.numel(), float((got - ref).abs().max()))


def _check_subpixel(ds, di, vol, what):
    """ds: the sub-pixel disparity of the fused call, di: its integer d* (already checked bit-equal to the volume's).
    The offset is the vertex of the parabola through c-, c0, c+; scores within EPS of the volume's move it by at most
    3 EPS / (|den| - 4 EPS), and the two disparities are each rounded to float32 once.  Checked where |den| >= 1e-3."""
    D = vol.size(1)
    ulp = 2.0 ** (math.ceil(math.log2(max(D, 2))) - 24)  # two half ulps of a value below 2^ceil(log2 D)
    ref, _ = _wta(vol, True)
    chunk = max(1, (1 << 26) // vol[0].numel())
    for i in range(0, vol.size(0), chunk):
        v, d = vol[i:i + chunk], di[i:i + chunk].long()
        cm, c0, cp = (v.gather(1, (d + k).clamp(0, D - 1)).double() for k in (-1, 0, 1))
        den = (cm - 2 * c0 + cp).abs()
        err = (ds[i:i + chunk].double() - ref[i:i + chunk].double()).abs()
        sel = den >= 1e-3
        excess = (err - 3 * EPS / (den - 4 * EPS) - ulp)[sel]
        assert excess.numel() == 0 or float(excess.max()) <= 0, \
            "%s: sub-pixel disparity off by up to %.3e beyond the bound" % (what, float(excess.max()))


def _sep_launches(ks, B, nb, D, wta, what):
    """The separable path ran in launches of at most nb images: grid.z = images x ceil(D / 16), and the disparity's
    last pass once per launch."""
    _expect(ks, [SEP, FINISH] if wta else [SEP], KERNELS, what)
    _expect_chunks(ks, SEP, B, nb, what, zper=cdiv(D, XS_DT))
    if wta and _seen(ks, what):
        assert len(_grids(ks, FINISH)) == cdiv(B, nb), "%s: %s ran %d times" % (what, FINISH, len(_grids(ks, FINISH)))


def _check_disparity(tx, a, b, vol, D, bs, nb, what):
    """xcorr_disparity in separable launches of at most nb images against disparity_from_volume(vol), where the volume
    ran the same separable kernel: d* and the score bit-equal, the sub-pixel disparity within the bound of
    _check_subpixel.  Returns the sub-pixel (disp, score)."""
    (di, si), ks = _kernels(lambda: tx.xcorr_disparity(a, b, D, bs, False))
    _sep_launches(ks, a.size(0), nb, D, True, what + " disparity")
    rd, rs = _wta(vol, False)
    _equal(di, rd, what + ": integer disparity vs the volume's argmax")
    _equal(si, rs, what + ": score vs the volume's maximum")
    del rd, rs
    ds, ss = tx.xcorr_disparity(a, b, D, bs, True)
    _equal(ss, si, what + ": score with and without subpixel")
    _check_subpixel(ds, di, vol, what)
    return ds, ss


def _check_single_images(tx, a, b, vol, disp, score, D, bs, what):
    """vol[n], disp[n] and score[n] of the batched call bit-equal to a call on image n alone (one separable launch), for
    every image, in groups that bound the extra memory."""
    L, st = _lib(), _stream()
    B, _, H, W = a.shape
    group = max(1, min(B, (1 << 27) // (D * H * W)))
    v1, d1, s1 = torch.empty(group, D, H, W, device=DEV), torch.empty(group, 1, H, W, device=DEV), torch.empty(group, 1, H, W, device=DEV)
    px, vx = H * W * 4, D * H * W * 4  # bytes per image of an input / disparity map, of a volume
    for b0 in range(0, B, group):
        n = min(group, B - b0)
        for i in range(n):
            p0, p1 = a.data_ptr() + (b0 + i) * px, b.data_ptr() + (b0 + i) * px
            L.call("ctd_xcorrvol_f32", p0, p1, v1.data_ptr() + i * vx, 1, 1, H, W, D, bs, st)
            L.call("ctd_xcorr_disparity_f32", p0, p1, d1.data_ptr() + i * px, s1.data_ptr() + i * px, 1, 1, H, W, D, bs, 1, st)
        for name, one, full in (("volume", v1, vol), ("disparity", d1, disp), ("score", s1, score)):
            assert torch.equal(one[:n], full[b0:b0 + n]), "%s: %s of images %d..%d differs from one-image calls: %d values" % (
                what, name, b0, b0 + n - 1, int((one[:n] != full[b0:b0 + n]).sum()))


# ---------------------------------------------------------------- 1. batch split at full size
def _band_rows(k, H):
    """One band of three rows per boundary image, turn about: the top rows, the bottom rows, the middle."""
    return [((0, 3), (H - 3, H), (H // 2 - 1, H // 2 + 2))[k % 3]]


@pytest.mark.parametrize("bs", (3, 5, 7, 9))
def test_batch_split_full_size(tx, bs):
    """27 images at 480x640, D = 128: launches of 13, 13 and 1 images (grid.z 104, 104, 8) for the volume and the
    disparity.  The volume against the oracle at every launch boundary, the disparity against the volume, every image
    against a call on it alone."""
    B, H, W, D = 27, 480, 640, 128
    nb = images_per_launch(D, H, W)
    assert nb == 13
    an, bn = _full_batch(B)
    a, b = torch.from_numpy(an).to(DEV), torch.from_numpy(bn).to(DEV)
    what = "27x480x640 D128 bs%d" % bs
    vol, ks = _kernels(lambda: tx.xcorrvol(a, b, D, bs))
    _sep_launches(ks, B, nb, D, False, what)
    for k, n in enumerate(_boundaries(B, nb)):
        _check_oracle(vol, an, bn, D, bs, [n], _band_rows(k + bs, H), what)
    disp, score = _check_disparity(tx, a, b, vol, D, bs, nb, what)
    _check_single_images(tx, a, b, vol, disp, score, D, bs, what)


def test_batch_split_hit_list_overflow(tx):
    """The 27-image call at block 5 with the fix-up's hit list forced to size 0 (xcorr_hitcap): every launch hands its
    untrusted outputs to the overflow fallback kernel.  Same launches, and the same volume and disparity as with the
    list, bit for bit; the volume against the oracle at the launch boundaries."""
    B, H, W, D, bs = 27, 480, 640, 128, 5
    nb = images_per_launch(D, H, W)
    an, bn = _full_batch(B)
    a, b = torch.from_numpy(an).to(DEV), torch.from_numpy(bn).to(DEV)
    listed = tx.xcorrvol(a, b, D, bs)
    listed_d = tx.xcorr_disparity(a, b, D, bs)
    _option("xcorr_hitcap", 0)
    try:
        vol, ks = _kernels(lambda: tx.xcorrvol(a, b, D, bs))
        _sep_launches(ks, B, nb, D, False, "hitcap 0")
        (disp, score), ks = _kernels(lambda: tx.xcorr_disparity(a, b, D, bs))
        _sep_launches(ks, B, nb, D, True, "hitcap 0 disparity")
    finally:
        _option("xcorr_hitcap", -1)
    _equal(vol, listed, "hitcap 0: volume vs the listed fix-up")
    _equal(disp, listed_d[0], "hitcap 0: disparity vs the listed fix-up")
    _equal(score, listed_d[1], "hitcap 0: score vs the listed fix-up")
    del listed
    for k, n in enumerate(_boundaries(B, nb)):
        _check_oracle(vol, an, bn, D, bs, [n], _band_rows(k, H), "hitcap 0")


def test_batch_split_under_capture(tx):
    """The 27-image calls of both ops (block 9) captured into one CUDA graph and replayed twice on a side stream: the
    three launches of each call replay bit-equal to the eager calls."""
    B, H, W, D, bs = 27, 480, 640, 128, 9
    nb = images_per_launch(D, H, W)
    an, bn = _full_batch(B)
    a, b = torch.from_numpy(an).to(DEV), torch.from_numpy(bn).to(DEV)
    (vol, (disp, score)), ks = _kernels(lambda: (tx.xcorrvol(a, b, D, bs), tx.xcorr_disparity(a, b, D, bs)))
    _expect(ks, [SEP, FINISH], KERNELS, "eager calls")
    if _seen(ks, "eager calls"):
        assert [g[2] for g in _grids(ks, SEP)] == [104, 104, 8] * 2, ks
    gv, gd, gs = torch.empty_like(vol), torch.empty_like(disp), torch.empty_like(score)
    L = _lib()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        st = _stream()
        L.call("ctd_xcorrvol_f32", a.data_ptr(), b.data_ptr(), gv.data_ptr(), B, 1, H, W, D, bs, st)
        L.call("ctd_xcorr_disparity_f32", a.data_ptr(), b.data_ptr(), gd.data_ptr(), gs.data_ptr(), B, 1, H, W, D, bs, 1, st)
    side = torch.cuda.Stream()
    for rep in range(2):
        for t in (gv, gd, gs):
            t.fill_(float("nan"))
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            g.replay()
        side.synchronize()
        for name, got, ref in (("volume", gv, vol), ("disparity", gd, disp), ("score", gs, score)):
            assert torch.equal(got, ref), "replay %d: %s differs from the eager call" % (rep, name)
    del g


# ---------------------------------------------------------------- 2. bounds that used to leave the separable path
def _check_split(tx, a, b, D, bs, nb, rows, what):
    """A batch that the grid or the statistics bound splits: separable launches of nb images for both ops, the volume
    against the oracle on `rows` of the launch-boundary images, the disparity bit-equal to the volume's argmax, every
    image bit-equal to a call on it alone."""
    B = a.size(0)
    vol, ks = _kernels(lambda: tx.xcorrvol(a, b, D, bs))
    _sep_launches(ks, B, nb, D, False, what)
    _check_oracle(vol, a, b, D, bs, _boundaries(B, nb), rows, what)
    disp, score = _check_disparity(tx, a, b, vol, D, bs, nb, what)
    _check_single_images(tx, a, b, vol, disp, score, D, bs, what)


def test_split_by_grid_bound(tx):
    """16385 images of 16x16, D = 64: one launch would need gridDim.z = 16385 x 4 > 65535.  Launches of 16383 and 2
    images (the hit-list bound alone allows 32766)."""
    B, H, W, D, bs = 16385, 16, 16, 64, 9
    assert HIT_OUTPUTS // (D * H * W) == 32766 and B * cdiv(D, XS_DT) > 65535
    nb = images_per_launch(D, H, W)
    assert nb == 16383
    a, b = _tiled(B, H, W, 997)
    _check_split(tx, a, b, D, bs, nb, [(0, H)], "16385x16x16 D64")


def test_split_by_statistics_bound(tx):
    """1639 images of 65535x4, D = 1, block 3: the in1 statistics plane of one launch would hold 1639 x 65535 x 20 >=
    2^31 positions (ws1 = 16 + 4).  Launches of 1638 and 1 images; the oracle checks whole images."""
    B, H, W, D, bs = 1639, 65535, 4, 1, 3
    ws1 = cdiv(D, XS_DT) * XS_DT + cdiv(W, 4) * 4
    assert ws1 == 20 and B * H * ws1 >= 2 ** 31 and HIT_OUTPUTS // (D * H * W) >= B
    nb = images_per_launch(D, H, W)
    assert nb == 1638
    a, b = _tiled(B, H, W, 1237)
    _check_split(tx, a, b, D, bs, nb, [(0, H)], "1639x65535x4 D1")


# ---------------------------------------------------------------- 3. per-image limits: the fallbacks
def test_tall_image_runs_generic(tx):
    """One image of 1048577 rows: ceil(H / 16) = 65537 statistics row tiles, more than one launch takes, and H > 65535
    rules out the direct kernel.  Both ops run their generic kernels, so the disparity (sub-pixel included) is
    bit-equal to the volume's argmax."""
    B, H, W, D, bs = 1, 1048577, 8, 4, 9
    assert cdiv(H, ST_H) > 65535
    a, b = _tiled(B, H, W, 0)
    vol, ks = _kernels(lambda: tx.xcorrvol(a, b, D, bs))
    _expect(ks, [GENERIC], KERNELS, "H 1048577")
    _check_oracle(vol, a, b, D, bs, [0], [(0, 6), (1048560 - 3, 1048560 + 3), (H - 6, H)], "H 1048577")
    for sub in (False, True):
        (d, s), ks = _kernels(lambda: tx.xcorr_disparity(a, b, D, bs, sub))
        _expect(ks, [DGENERIC], KERNELS, "H 1048577 disparity")
        rd, rs = _wta(vol, sub)
        _equal(d, rd, "H 1048577 subpixel=%s: disparity vs the volume's" % sub)
        _equal(s, rs, "H 1048577 subpixel=%s: score vs the volume's" % sub)


@pytest.mark.parametrize("B,H,W,D", [(1, 65537, 8, 4), (1024, 8, 8, 2080)], ids=["H65537", "D2080"])
def test_direct_refusal_runs_generic(tx, B, H, W, D):
    """With xcorr_direct the volume skips the separable kernel; the direct kernel then refuses H > 65535 (grid.y) and
    1024-image chunks with 1024 x ceil(D / 32) > 65535 (grid.z), and the generic kernel runs."""
    bs = 9
    assert H > 65535 or min(B, 1024) * cdiv(D, XD_DC) > 65535
    a, b = _tiled(B, H, W, 331)
    _option("xcorr_direct", 1)
    try:
        vol, ks = _kernels(lambda: tx.xcorrvol(a, b, D, bs))
    finally:
        _option("xcorr_direct", 0)
    what = "xcorr_direct %dx%dx%d D%d" % (B, H, W, D)
    _expect(ks, [GENERIC], KERNELS, what)
    rows = [(0, H)] if H <= 64 else [(0, 6), (H // 2 - 3, H // 2 + 3), (H - 6, H)]
    _check_oracle(vol, a, b, D, bs, sorted({0, B // 2, B - 1}), rows, what)
