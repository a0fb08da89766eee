"""Block-matching disparity from the XCorrVol cost volume (xcorrvol.cu: ctd_xcorr_disparity_*, torchext.xcorr_disparity).

The definition is disparity_from_volume, the plain-torch winner-take-all over a volume: the CPU tests pin it to a brute-force
numpy loop over oracle volumes.  The GPU tests hold the fused kernels to disparity_from_volume(xcorrvol(...)) on the same
inputs: the integer disparity and the score bit-equal, the sub-pixel offset within what the 1e-5 score tolerance allows.
"""
import re
import subprocess

import numpy as np
import pytest
import torch

import oracle

DEV = "cuda:0"


def _F():
    from connecting_the_dots_b200.torchext import functions
    return functions


def wta_brute(vol, subpixel):
    """The definition, one pixel at a time: vol [D,H,W] -> (disp, score) [H,W], float64."""
    D, H, W = vol.shape
    disp, score = np.zeros((H, W)), np.zeros((H, W))
    for h in range(H):
        for w in range(W):
            col = [float(v) for v in vol[:, h, w]]
            m = max(col)
            d = col.index(m)  # the first maximum
            delta = 0.0
            if subpixel and 0 < d < D - 1:
                cm, c0, cp = col[d - 1], col[d], col[d + 1]
                den = cm - 2 * c0 + cp
                if den < 0:
                    delta = min(max((cm - cp) / (2 * den), -0.5), 0.5)
            disp[h, w], score[h, w] = d + delta, m
    return disp, score


def lcn_pair(n, H, W):
    from connecting_the_dots_b200 import synth
    d = synth.make_pair(n, H, W)
    return d["ta"][None], d["pat_lcn"][None]


# ---------------------------------------------------------------- CPU: the definition
@pytest.mark.parametrize("subpixel", (True, False))
def test_disparity_from_volume_matches_brute_force(subpixel):
    F = _F()
    a, b = lcn_pair(0, 24, 64)
    vols = [oracle.xcorrvol(a, b, 32, 9)]            # left border: clamped in1 windows, exact ties between disparities
    rng = np.random.RandomState(1)
    q = np.round(rng.rand(9, 6, 7) * 3) / 3          # coarse values: repeated maxima, flat tops (den = 0), peaks at both ends
    q[:, 0, 0], q[:, 0, 1], q[:, 0, 2] = 0, np.arange(9), -np.arange(9.0)   # constant, d* = D - 1, d* = 0
    q[:, 1, 0] = [0, 1, 3, 3, 1, 0, 3, 0, 0]          # a tie of three: the first wins, den < 0 there
    vols.append(q.astype(np.float32))
    vols.append(oracle.xcorrvol(a[:, :8, :12].copy(), b[:, :8, :12].copy(), 5, 3).astype(np.float64))
    for vol in vols:
        ref_disp, ref_score = wta_brute(vol, subpixel)
        disp, score = F.disparity_from_volume(torch.from_numpy(vol), subpixel)
        assert disp.shape == (1,) + vol.shape[1:] and disp.dtype == torch.from_numpy(vol).dtype
        assert np.array_equal(score[0].numpy(), ref_score.astype(vol.dtype))
        np.testing.assert_allclose(disp[0].numpy(), ref_disp, rtol=0, atol=1e-5 if vol.dtype == np.float32 else 1e-12)
        d4, s4 = F.disparity_from_volume(torch.from_numpy(vol)[None], subpixel)   # batched [B,D,H,W] -> [B,1,H,W]
        assert d4.shape == (1, 1) + vol.shape[1:] and torch.equal(d4[0], disp) and torch.equal(s4[0], score)
    # the cases the volumes above had to contain
    dq = F.disparity_from_volume(torch.from_numpy(vols[1]), False)[0][0].numpy()
    assert dq[0, 0] == 0 and dq[0, 1] == 8 and dq[0, 2] == 0 and dq[1, 0] == 2
    assert (np.sort(vols[0], axis=0)[-1] == np.sort(vols[0], axis=0)[-2]).any(), "no tie in the oracle volume"
    nan = torch.from_numpy(vols[1].copy())
    nan[3, 2, 2] = float("nan")                       # outside the contract, but the oracle answers instead of failing
    assert F.disparity_from_volume(nan, True)[0][0, 2, 2] == 8


def test_xcorr_disparity_api_without_gpu(tx):
    from connecting_the_dots_b200 import _lib
    x = torch.rand(1, 1, 12, 12)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        tx.xcorr_disparity(x, x, 4, 3)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        tx.XCorrDisparity(4, 3)(x, x)
    m = tx.XCorrDisparity()
    assert (m.n_disps, m.block_size, m.subpixel) == (128, 9, True)
    with pytest.raises(_lib.CtdError, match="block_size"):
        _lib.call("ctd_xcorr_disparity_f32", 16, 16, 16, 16, 1, 1, 8, 8, 4, 0, 1, None)
    with pytest.raises(_lib.CtdError, match="negative size"):
        _lib.call("ctd_xcorr_disparity_f64", 16, 16, 16, 16, 1, 1, -8, 8, 4, 3, 1, None)
    with pytest.raises(_lib.CtdError, match="n_disps"):
        _lib.call("ctd_xcorr_disparity_f32", 16, 16, 16, 16, 1, 1, 8, 8, 0, 3, 1, None)
    with pytest.raises(_lib.CtdError, match="null pointer"):
        _lib.call("ctd_xcorr_disparity_f32", 16, 16, None, 16, 1, 1, 8, 8, 4, 3, 1, None)
    with pytest.raises(_lib.CtdError, match="null pointer"):
        _lib.call("ctd_xcorr_disparity_f32", None, 16, 16, None, 1, 1, 8, 8, 4, 3, 1, None)
    # an empty batch is a no-op, with any n_disps
    _lib.call("ctd_xcorr_disparity_f32", None, None, None, None, 0, 1, 8, 8, 0, 9, 1, None)
    _lib.call("ctd_xcorr_disparity_f64", None, None, None, None, 2, 1, 0, 8, 4, 9, 0, None)


def test_xcorr_disparity_kernels_have_no_floating_point_atomics(tx):
    """The disparity kernels merge partial maxima with 64-bit integer atomics on (score bits, d) keys: the only atomics
    in them are integer ones."""
    from connecting_the_dots_b200 import _lib
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    new = re.compile(r"xcorr_wta_finish_kernel|xcorr_disparity_generic|xcorr_(sep|eval|fixup)_kernelI.*yEE")
    atomics, kernels, kernel = [], set(), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            kernel = m.group(1) if new.search(m.group(1)) else None
            if kernel:
                kernels.add(kernel)
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d+\s+)?((?:ATOM|RED)[A-Z0-9_.]*)", line)
        if m and kernel:
            atomics.append((kernel, m.group(1)))
    assert len(kernels) >= 2 + 3 * 4, sorted(kernels)   # finish x4 block sizes, generic x2, sep / eval / fixup variants
    assert any("MAX.64" in op for _, op in atomics), "no 64-bit integer max found"
    for k, op in atomics:
        assert not re.search(r"F16|F32|F64|BF16|\.FT", op), (k, op)


# ---------------------------------------------------------------- GPU
def cu(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


def fused_and_volume(tx, a, b, D, bs, subpixel=False):
    """(disp, score) of the fused call and of disparity_from_volume over xcorrvol's volume, same inputs."""
    got = tx.xcorr_disparity(a, b, D, bs, subpixel)
    ref = tx.disparity_from_volume(tx.xcorrvol(a, b, D, bs), subpixel)
    return got, ref


def assert_exact(tx, a, b, D, bs, what):
    (d, s), (rd, rs) = fused_and_volume(tx, a, b, D, bs)
    assert d.shape == rd.shape and s.shape == rs.shape and d.dtype == a.dtype, what
    bad = (d != rd).sum().item()
    assert bad == 0, "%s: %d of %d integer disparities differ" % (what, bad, d.numel())
    assert torch.equal(s, rs), "%s: scores differ, max |diff| %.3e" % (what, float((s - rs).abs().max()))


@pytest.mark.gpu
@pytest.mark.parametrize("bs", (3, 5, 7, 9))
def test_fast_path_is_the_volume_argmax(tx, bs):
    a, b = lcn_pair(2, 70, 300)
    assert_exact(tx, cu(a), cu(b), 64, bs, "lcn crop bs%d" % bs)
    rng = np.random.RandomState(bs)
    x = rng.randn(2, 1, 37, 133).astype(np.float32)
    y = (np.roll(x, 5, axis=3) + 0.5 * rng.randn(2, 1, 37, 133)).astype(np.float32)
    assert_exact(tx, cu(x), cu(y), 40, bs, "randn bs%d" % bs)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ("bs2", "bs4", "bs11", "C2", "f64"))
def test_generic_path_is_the_volume_argmax(tx, case):
    rng = np.random.RandomState(len(case))
    C = 2 if case == "C2" else 1
    bs = {"bs2": 2, "bs4": 4, "bs11": 11}.get(case, 9)
    x = rng.randn(2, C, 23, 50)
    y = np.roll(x, 4, axis=3) + 0.4 * rng.randn(2, C, 23, 50)
    dt = torch.float64 if case == "f64" else torch.float32
    assert_exact(tx, cu(x, dt), cu(y, dt), 19, bs, case)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 1, 30, 64, 1), (2, 1, 33, 90, 17), (1, 1, 25, 200, 128), (1, 1, 20, 40, 64),
                                   (2, 1, 31, 70, 24), (1, 1, 5, 60, 20)],
                         ids=["D1", "D17", "D128", "D_gt_W", "W_not_mult4", "H_lt_window"])
def test_shapes(tx, shape):
    B, C, H, W, D = shape
    a, b = lcn_pair(3, H, W)
    a, b = np.repeat(a[None], B, 0), np.repeat(np.roll(b, B, axis=1)[None], B, 0)
    for bs in (9, 5):
        assert_exact(tx, cu(a), cu(b), D, bs, "%s bs%d" % (shape, bs))


@pytest.mark.gpu
def test_misaligned_base_pointers(tx):
    a, b = lcn_pair(4, 40, 256)
    ba = torch.zeros(1 + a.size, device=DEV)
    bb = torch.zeros(3 + b.size, device=DEV)
    ta = ba[1:].view(a.shape).copy_(cu(a))           # 4-byte aligned, not 16
    tb = bb[3:].view(b.shape).copy_(cu(b))
    assert ta.data_ptr() % 16 and tb.data_ptr() % 16
    for bs in (9, 3):
        assert_exact(tx, ta[None], tb[None], 48, bs, "misaligned bs%d" % bs)


@pytest.mark.gpu
@pytest.mark.parametrize("bs", (9, 5))
def test_full_size_batch8(tx, bs):
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(8)
    assert_exact(tx, cu(d["ta"]), cu(d["pat_lcn"]), 128, bs, "480x640 batch 8 bs%d" % bs)


def ill_conditioned_inputs():
    """The inputs of test_xcorrvol_ill_conditioned_windows: raw intensities with a flat patch (block 9), and an exactly
    zero band (block 5)."""
    rng = np.random.RandomState(7)
    H, W = 40, 132
    a = (0.5 + 0.02 * rng.randn(1, 1, H, W)).astype(np.float32)
    b = (0.5 + 0.02 * rng.randn(1, 1, H, W)).astype(np.float32)
    a[0, 0, 5:25, 30:70] = 0.75
    b[0, 0, 10:30, 80:120] = rng.randn(20, 40)
    z = rng.randn(1, 1, H, W).astype(np.float32)
    z[0, 0, :, 40:90] = 0.0
    return [(a, b, 9), (z, np.roll(z, 2, axis=3), 5)]


@pytest.mark.gpu
def test_ill_conditioned_windows_and_overflow_fallback(tx):
    """Outputs the fix-up recomputes take no part in the fast-path maximum; their recomputed values are merged by the
    evaluation kernel, or by the overflow fallback kernel when the hit list is forced to size 0."""
    from connecting_the_dots_b200 import _lib
    for a, b, bs in ill_conditioned_inputs():
        a2, b2 = np.concatenate([a, a[..., ::-1]]), np.concatenate([b, b[..., ::-1]])
        ref = tx.disparity_from_volume(tx.xcorrvol(cu(a2), cu(b2), 21, bs), False)
        got = tx.xcorr_disparity(cu(a2), cu(b2), 21, bs, False)
        _lib.set_option("xcorr_hitcap", 0)
        try:
            fallback = tx.xcorr_disparity(cu(a2), cu(b2), 21, bs, False)
        finally:
            _lib.set_option("xcorr_hitcap", -1)
        for name, (d, s) in (("listed", got), ("overflow fallback", fallback)):
            assert torch.equal(d, ref[0]), "bs%d %s: disparities differ at %d pixels" % (bs, name, int((d != ref[0]).sum()))
            assert torch.equal(s, ref[1]), "bs%d %s: scores differ" % (bs, name)


@pytest.mark.gpu
@pytest.mark.parametrize("bs", (9, 5))
def test_subpixel_offset(tx, bs):
    """The fused path takes c-, c0, c+ in the centred form, within ~1e-5 of the volume's scores, so the parabola's vertex
    moves by at most ~4e-5 / |den|; the float32 disp adds at most half an ulp of d* (3.8e-6 at d* < 128)."""
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(2, 96, 320)
    a, b = cu(d["ta"]), cu(d["pat_lcn"])
    vol = tx.xcorrvol(a, b, 128, bs).double()
    di, _ = tx.xcorr_disparity(a, b, 128, bs, False)
    ds, _ = tx.xcorr_disparity(a, b, 128, bs, True)
    ref, _ = tx.disparity_from_volume(vol, True)
    rd, _ = tx.disparity_from_volume(vol, False)
    assert torch.equal(di.double(), rd)
    delta, ref_delta = ds.double() - di.double(), ref - rd
    assert float(delta.abs().max()) <= 0.5
    dd = di.long()
    D = vol.size(1)
    cm, c0, cp = (vol.gather(1, (dd + k).clamp(0, D - 1)) for k in (-1, 0, 1))
    den = (cm - 2 * c0 + cp).abs()
    sel = den >= 1e-3
    err = (delta - ref_delta).abs()[sel]
    assert sel.float().mean() > 0.5
    worst = float((err * den[sel]).max())
    assert worst <= 4e-5, "max |delta - delta_volume| * |den| = %.3e" % worst


@pytest.mark.gpu
def test_force_generic_is_the_generic_volume_argmax(tx):
    from connecting_the_dots_b200 import _lib
    a, b = lcn_pair(5, 30, 96)
    _lib.set_option("force_generic", 1)
    try:
        for sub in (False, True):
            (d, s), (rd, rs) = fused_and_volume(tx, cu(a)[None], cu(b)[None], 33, 9, sub)
            assert torch.equal(d, rd) and torch.equal(s, rs), "subpixel=%s" % sub
    finally:
        _lib.set_option("force_generic", 0)


@pytest.mark.gpu
def test_deterministic_streams_capture_and_serial(tx):
    from connecting_the_dots_b200 import _lib, synth
    d = synth.make_batch(2, 96, 256)
    a, b = cu(d["ta"]), cu(d["pat_lcn"])
    ref = tx.xcorr_disparity(a, b, 48, 9)
    again = tx.xcorr_disparity(a, b, 48, 9)
    assert torch.equal(ref[0], again[0]) and torch.equal(ref[1], again[1])
    _lib.set_option("xcorr_serial", 1)
    try:
        serial = tx.xcorr_disparity(a, b, 48, 9)
    finally:
        _lib.set_option("xcorr_serial", 0)
    assert torch.equal(serial[0], ref[0]) and torch.equal(serial[1], ref[1])
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        on_s = tx.xcorr_disparity(a, b, 48, 9)
    s.synchronize()
    assert torch.equal(on_s[0], ref[0]) and torch.equal(on_s[1], ref[1])
    disp, score = torch.zeros_like(ref[0]), torch.zeros_like(ref[1])
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _lib.call("ctd_xcorr_disparity_f32", a.data_ptr(), b.data_ptr(), disp.data_ptr(), score.data_ptr(), 2, 1, 96, 256, 48, 9, 1,
                  torch.cuda.current_stream().cuda_stream)
    for _ in range(3):
        disp.zero_()
        score.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(disp, ref[0]) and torch.equal(score, ref[1])
    # score is optional
    nd = torch.zeros_like(ref[0])
    _lib.call("ctd_xcorr_disparity_f32", a.data_ptr(), b.data_ptr(), nd.data_ptr(), None, 2, 1, 96, 256, 48, 9, 1,
              torch.cuda.current_stream().cuda_stream)
    assert torch.equal(nd, ref[0])


@pytest.mark.gpu
def test_errors_empty_3d_signature_and_module(tx):
    x = torch.rand(1, 1, 16, 20, device=DEV)
    with pytest.raises(RuntimeError):
        tx.xcorr_disparity(x, torch.rand(1, 1, 16, 21, device=DEV), 4, 3)
    with pytest.raises(RuntimeError):
        tx.xcorr_disparity(x, x.double(), 4, 3)
    with pytest.raises(RuntimeError):
        tx.xcorr_disparity(x.transpose(2, 3), x.transpose(2, 3), 4, 3)
    with pytest.raises(NotImplementedError):
        tx.xcorr_disparity(x.half(), x.half(), 4, 3)
    with pytest.raises(RuntimeError, match="n_disps"):
        tx.xcorr_disparity(x, x, 0, 3)
    e = torch.rand(0, 1, 16, 20, device=DEV)
    d, s = tx.xcorr_disparity(e, e, 0, 9)
    assert d.shape == (0, 1, 16, 20) and s.shape == (0, 1, 16, 20)
    a, b = lcn_pair(6, 32, 80)
    d4, s4 = tx.xcorr_disparity(cu(a)[None], cu(b)[None], 24, 9)
    d3, s3 = tx.xcorr_disparity(cu(a), cu(b), 24, 9)
    assert d3.shape == (1, 32, 80) and torch.equal(d3, d4[0]) and torch.equal(s3, s4[0])
    assert not d3.requires_grad and d3.dtype == torch.float32
    dm, sm = tx.XCorrDisparity(24, 9)(cu(a)[None], cu(b)[None])
    assert torch.equal(dm, d4) and torch.equal(sm, s4)


@pytest.mark.gpu
def test_end_to_end_against_ground_truth(tx):
    """synth.make_batch(2) at block 9, D = 128: the fraction of interior pixels (columns 140.. so that the true disparity
    is inside the search range) whose disparity is within 2 px of the ground truth.  Catches sign and offset errors in the
    d convention.  Measured on an NVIDIA B200: 0.660 (the CPU oracle's volume gave 0.76 on rows 200-247 of frame 0)."""
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(2)
    disp, score = tx.xcorr_disparity(cu(d["ta"]), cu(d["pat_lcn"]), 128, 9)
    gt = cu(d["disp"])
    inner = (slice(None), slice(None), slice(9, -9), slice(140, -9))
    frac = float(((disp - gt).abs() <= 2)[inner].float().mean())
    assert frac >= 0.6, frac
    assert float(score.max()) <= 1 + 1e-5
