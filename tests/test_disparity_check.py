"""Left-right consistency and uniqueness checks over a score volume (disparity_check.cu: ctd_disparity_check_*,
torchext.disparity_check / right_disparity_from_volume / disparity_check_pytorch / DisparityCheck).

The definition is disparity_check_pytorch with right_disparity_from_volume: the CPU tests pin both bit for bit to a pure-Python
loop over pixels and disparities.  The GPU tests hold the kernel bit for bit to the restatement run on the GPU, over synthetic
volumes with many ties and over the volumes of the library's three matchers.
"""
import itertools
import re
import subprocess

import numpy as np
import pytest
import torch

DEV = "cuda:0"


def _F():
    from connecting_the_dots_b200.torchext import functions
    return functions


def _wta(vals, subpixel, dtype):
    """First maximum of a list of Python floats and disparity_from_volume's fp64 offset: (disp, score, d*)."""
    n = len(vals)
    d = max(range(n), key=lambda i: (vals[i], -i))
    delta = 0.0
    if subpixel and 0 < d < n - 1:
        cm, c0, cp = vals[d - 1], vals[d], vals[d + 1]
        den = cm - 2.0 * c0 + cp
        if den < 0:
            delta = min(max((cm - cp) / (2.0 * den), -0.5), 0.5)
    return dtype(float(d) + delta), dtype(vals[d]), d


def check_brute(vol, max_diff, uniqueness, subpixel):
    """The definition one pixel at a time: vol [B,D,H,W] numpy -> disp, score, disp_right, score_right, valid [B,1,H,W]."""
    B, D, H, W = vol.shape
    dt = vol.dtype.type
    out = [np.zeros((B, 1, H, W), vol.dtype) for _ in range(4)] + [np.zeros((B, 1, H, W), bool)]
    for b, h in itertools.product(range(B), range(H)):
        dr = []
        for x in range(W):
            vals = [float(vol[b, d, h, x + d]) for d in range(min(D, W - x))]
            out[2][b, 0, h, x], out[3][b, 0, h, x], k = _wta(vals, subpixel, dt)
            dr.append(k)
        for w in range(W):
            vals = [float(vol[b, d, h, w]) for d in range(D)]
            out[0][b, 0, h, w], out[1][b, 0, h, w], k = _wta(vals, subpixel, dt)
            lr = max_diff < 0 or (w - k >= 0 and abs(k - dr[w - k]) <= max_diff)
            far = [vals[d] for d in range(D) if abs(d - k) >= 2]
            uq = uniqueness == 0 or not far or vals[k] - max(far) >= uniqueness
            out[4][b, 0, h, w] = lr and uq
    return out


def coarse(rng, shape, dtype):
    """Values on a grid of 1/4 in [-1, 1]: many exact ties, so the first-index rule and the uniqueness margin matter."""
    return (np.round(rng.rand(*shape) * 8) / 4 - 1).astype(dtype)


SHAPES = ((1, 1, 3, 6), (2, 2, 2, 5), (1, 3, 4, 7), (1, 5, 3, 9), (1, 5, 2, 3), (1, 3, 1, 1), (2, 5, 1, 8), (1, 7, 2, 4))


def cpu_volumes():
    rng = np.random.RandomState(3)
    for dtype in (np.float32, np.float64):
        for shape in SHAPES:
            yield "coarse %s %s" % (shape, dtype.__name__), coarse(rng, shape, dtype)
            yield "randn %s %s" % (shape, dtype.__name__), rng.randn(*shape).astype(dtype)


def test_restatement_matches_brute_force():
    F = _F()
    for name, v in cpu_volumes():
        t = torch.from_numpy(v)
        for subpixel in (True, False):
            rd, rs = F.right_disparity_from_volume(t, subpixel)
            ld, ls = F.disparity_from_volume(t, subpixel)
            for max_diff, u in itertools.product((-1, 0, 1, 3), (0.0, 0.25, 1.0)):
                ref = check_brute(v, max_diff, u, subpixel)
                d, s, ok = F.disparity_check_pytorch(t, max_diff, u, subpixel)
                assert ok.dtype == torch.bool and d.dtype == t.dtype and d.shape == ok.shape == (v.shape[0], 1) + v.shape[2:]
                msg = "%s sub %d max_diff %d u %g" % (name, subpixel, max_diff, u)
                assert np.array_equal(d.numpy(), ref[0]) and np.array_equal(s.numpy(), ref[1]), msg
                assert torch.equal(d, ld) and torch.equal(s, ls), msg
                assert np.array_equal(ok.numpy(), ref[4]), msg
            assert np.array_equal(rd.numpy(), ref[2]) and np.array_equal(rs.numpy(), ref[3]), "%s sub %d" % (name, subpixel)


def test_restatement_3d_and_checks_off():
    F = _F()
    v = torch.from_numpy(coarse(np.random.RandomState(1), (1, 6, 4, 9), np.float32))
    d, s, ok = F.disparity_check_pytorch(v[0], 1, 0.5)
    d4, s4, ok4 = F.disparity_check_pytorch(v, 1, 0.5)
    assert d.shape == (1, 4, 9) and torch.equal(d, d4[0]) and torch.equal(s, s4[0]) and torch.equal(ok, ok4[0])
    assert F.right_disparity_from_volume(v[0])[0].shape == (1, 4, 9)
    assert bool(F.disparity_check_pytorch(v, -1, 0.0)[2].all())
    # a pixel near the left edge whose left disparity points out of view fails the LR check whatever dR* is
    ok = F.disparity_check_pytorch(v, 100, 0.0)[2]
    dl = F.disparity_from_volume(v, False)[0].long()
    assert torch.equal(ok, torch.arange(9).view(1, 1, 1, 9) - dl >= 0)


def test_disparity_check_api_without_gpu(tx):
    from connecting_the_dots_b200 import _lib
    F = _F()
    v = torch.rand(1, 4, 6, 7)
    for fn in (lambda: tx.disparity_check(v), lambda: tx.DisparityCheck()(v)):
        with pytest.raises(RuntimeError, match="no CPU implementation"):
            fn()
    m = tx.DisparityCheck()
    assert (m.max_diff, m.uniqueness, m.subpixel) == (1, 0.0, True)
    for u in (-1.0, float("nan"), float("inf")):
        with pytest.raises(RuntimeError, match="uniqueness"):
            F.disparity_check_pytorch(v, 1, u)
    with pytest.raises(RuntimeError, match="D x H x W"):
        F.disparity_check_pytorch(v[0, 0], 1, 0.0)
    with pytest.raises(RuntimeError, match="no disparities"):
        F.right_disparity_from_volume(torch.rand(1, 0, 2, 3))
    # the C ABI checks its arguments before any device work (pointers here are never dereferenced)
    P, O1, O2 = 1 << 30, 1 << 34, 1 << 36
    n = 2 * 6 * 7
    f32 = lambda *a: _lib.call("ctd_disparity_check_f32", *a)  # noqa: E731
    f64 = lambda *a: _lib.call("ctd_disparity_check_f64", *a)  # noqa: E731
    for fn, args, msg in ((f32, (P, O1, None, None, None, None, 2, 4, -6, 7, 1, 0.0, 1, None), "negative size"),
                          (f32, (P, O1, None, None, None, None, -2, 4, 6, 7, 1, 0.0, 1, None), "negative size"),
                          (f32, (P, O1, None, None, None, None, 2, -4, 6, 7, 1, 0.0, 1, None), "negative size"),
                          (f32, (P, O1, None, None, None, None, 2, 4, 6, 7, 1, -0.5, 1, None), "uniqueness"),
                          (f64, (P, O1, None, None, None, None, 2, 4, 6, 7, 1, float("nan"), 1, None), "uniqueness"),
                          (f64, (P, O1, None, None, None, None, 2, 4, 6, 7, 1, float("inf"), 1, None), "uniqueness"),
                          (f32, (P, O1, None, None, None, None, 2, 0, 6, 7, 1, 0.0, 1, None), "D = 0"),
                          (f32, (None, O1, None, None, None, None, 2, 4, 6, 7, 1, 0.0, 1, None), "null pointer"),
                          (f32, (P, P + 4 * 4 * n - 4, None, None, None, None, 2, 4, 6, 7, 1, 0.0, 1, None), "overlaps vol"),
                          (f64, (P, None, None, None, None, P - n + 1, 2, 4, 6, 7, 1, 0.0, 1, None), "overlaps vol"),
                          (f32, (P, O1, O1 + 4 * n - 4, None, None, None, 2, 4, 6, 7, 1, 0.0, 1, None), "outputs overlap"),
                          (f32, (P, O1, None, None, O2, O2 + n - 1, 2, 4, 6, 7, 1, 0.0, 1, None), "outputs overlap"),
                          (f64, (P, None, O1, O1 - 8 * n + 8, None, None, 2, 4, 6, 7, 1, 0.0, 1, None), "outputs overlap")):
        with pytest.raises(_lib.CtdError, match=msg):
            fn(*args)
    # an empty batch is a no-op, with any D and null pointers
    f32(None, None, None, None, None, None, 0, 0, 6, 7, 1, 0.0, 1, None)
    f64(None, None, None, None, None, None, 2, 4, 0, 7, 1, 0.0, 1, None)
    f32(None, None, None, None, None, None, 2, 4, 6, 0, 1, 0.0, 1, None)


def test_disparity_check_kernels_have_no_atomics(tx):
    """The kernel owns every output element: no atomics at all."""
    from connecting_the_dots_b200 import _lib
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    atomics, kernels, kernel = [], set(), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            kernel = m.group(1) if "disparity_check_kernel" in m.group(1) else None
            if kernel:
                kernels.add(kernel)
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d+\s+)?((?:ATOM|RED)[A-Z0-9_.]*)", line)
        if m and kernel:
            atomics.append((kernel, m.group(1)))
    assert len(kernels) == 2, sorted(kernels)   # float, double
    assert not atomics, atomics


# ---------------------------------------------------------------- GPU
SETTINGS = ((1, 0.0), (0, 0.25), (3, 1.0), (-1, 0.25), (-1, 0.0), (2, 0.0))


def cu(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


def gpu_volumes(dtype):
    """(name, vol): the CPU shapes, D off multiples of 4 and 32, D > W, rows of several chunks (W > 1024, D > 1024)."""
    rng = np.random.RandomState(11)
    shapes = SHAPES + ((3, 37, 5, 61), (1, 33, 9, 130), (2, 128, 3, 640), (1, 250, 4, 97), (1, 1024, 2, 700),
                       (1, 1024, 3, 1000), (1, 70, 3, 1500), (1, 300, 2, 2049), (1, 1300, 2, 2600))
    for shape in shapes:
        yield "coarse %s" % (shape,), cu(coarse(rng, shape, np.float32), dtype)
        yield "randn %s" % (shape,), cu(rng.randn(*shape), dtype)


def assert_check_equal(got, ref, msg):
    names = ("disp", "score", "valid")
    for g, r, n in zip(got, ref, names):
        assert g.dtype == r.dtype and g.shape == r.shape, "%s: %s %s %s vs %s %s" % (msg, n, g.dtype, tuple(g.shape), r.dtype, tuple(r.shape))
        assert torch.equal(g, r), "%s: %d %s values differ" % (msg, int((g != r).sum()), n)


def call_abi(vol, outs, max_diff, u, subpixel, stream=None):
    """ctd_disparity_check_* over a [B,D,H,W] volume into outs = (disp, score, disp_right, score_right, valid) (None = NULL)."""
    from connecting_the_dots_b200 import _lib
    sfx = "_f32" if vol.dtype == torch.float32 else "_f64"
    st = torch.cuda.current_stream().cuda_stream if stream is None else stream
    _lib.call("ctd_disparity_check" + sfx, vol.data_ptr(), *[o.data_ptr() if o is not None else None for o in outs],
              *vol.shape, max_diff, u, int(subpixel), st)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_bit_exact_against_restatement(tx, dtype):
    for name, vol in gpu_volumes(dtype):
        for subpixel in (True, False):
            rd, rs = tx.right_disparity_from_volume(vol, subpixel)
            for max_diff, u in SETTINGS:
                msg = "%s sub %d max_diff %d u %g" % (name, subpixel, max_diff, u)
                ref = tx.disparity_check_pytorch(vol, max_diff, u, subpixel)
                assert_check_equal(tx.disparity_check(vol, max_diff, u, subpixel), ref, msg)
            outs = [torch.full_like(rd, 7.0) for _ in range(4)] + [torch.zeros(rd.shape, dtype=torch.uint8, device=DEV)]
            call_abi(vol, outs, 1, 0.25, subpixel)
            msg = "%s sub %d: C ABI" % (name, subpixel)
            assert torch.equal(outs[2], rd) and torch.equal(outs[3], rs), msg + ", right view"
            assert_check_equal((outs[0], outs[1], outs[4].bool()), tx.disparity_check_pytorch(vol, 1, 0.25, subpixel), msg)


@pytest.mark.gpu
def test_each_output_may_be_null(tx):
    vol = cu(coarse(np.random.RandomState(2), (2, 40, 7, 90), np.float32))
    ld, ls, ok = tx.disparity_check_pytorch(vol, 1, 0.5)
    rd, rs = tx.right_disparity_from_volume(vol)
    full = (ld, ls, rd, rs, ok.to(torch.uint8))
    for i in range(5):
        outs = [torch.full_like(t, 3) for t in full]
        outs[i] = None
        call_abi(vol, outs, 1, 0.5, True)
        for j in range(5):
            if j != i:
                assert torch.equal(outs[j], full[j]), "output %d with output %d NULL" % (j, i)
    call_abi(vol, [None] * 5, 1, 0.5, True)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_misaligned_views(tx, dtype):
    """Every pointer one element off a 16-byte boundary; W = 68 (rows aligned to each other) and W = 67 (not)."""
    rng = np.random.RandomState(4)
    for W in (68, 67):
        shape = (2, 24, 9, W)
        vol = cu(coarse(rng, shape, np.float32), dtype)
        n = 2 * 9 * W

        def view(count, dt=dtype, src=None):
            v = torch.zeros(1 + count, dtype=dt, device=DEV)[1:]
            if src is not None:
                v.copy_(src.reshape(-1))
            return v
        vv = view(vol.numel(), src=vol)
        assert vv.data_ptr() % 16
        outs = [view(n) for _ in range(4)] + [view(n, torch.uint8)]
        from connecting_the_dots_b200 import _lib
        _lib.call("ctd_disparity_check" + ("_f32" if dtype == torch.float32 else "_f64"), vv.data_ptr(),
                  *[o.data_ptr() for o in outs], *shape, 1, 0.25, 1, torch.cuda.current_stream().cuda_stream)
        ref = tx.disparity_check_pytorch(vol, 1, 0.25, True)
        rd, rs = tx.right_disparity_from_volume(vol, True)
        o = [t.view(2, 1, 9, W) for t in outs]
        assert_check_equal((o[0], o[1], o[4].bool()), ref, "W %d" % W)
        assert torch.equal(o[2], rd) and torch.equal(o[3], rs), "W %d: right view" % W


def bench_frames(B):
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(B)
    return cu(d["ta"]), cu(d["pat_lcn"]), d


@pytest.mark.gpu
def test_real_volumes_batch8(tx):
    """480x640, batch 8, D = 128: census_vol at block 1 and 9, xcorrvol at block 9, sgm_aggregate of the census volume."""
    a, b, _ = bench_frames(8)
    vols = (("census bs1", lambda: tx.census_vol(a, b, 128, (7, 9), 1), (1, 16.0)),
            ("census bs9", lambda: tx.census_vol(a, b, 128, (7, 9), 9), (1, 64.0)),
            ("xcorrvol bs9", lambda: tx.xcorrvol(a, b, 128, 9), (1, 0.05)),
            ("sgm census bs1", lambda: tx.sgm_aggregate(tx.census_vol(a, b, 128, (7, 9), 1), 6, 400, 8), (1, 100.0)))
    for name, make, (max_diff, u) in vols:
        vol = make()
        for md, uu, sub in ((max_diff, u, True), (0, 0.0, False), (-1, u, True)):
            ref = tx.disparity_check_pytorch(vol, md, uu, sub)
            got = tx.disparity_check(vol, md, uu, sub)
            assert_check_equal(got, ref, "%s max_diff %d u %g sub %d" % (name, md, uu, sub))
            del ref, got
        del vol


@pytest.mark.gpu
def test_past_2_31_elements(tx):
    """Batch 64 at 480x640, D = 128: 2.5e9 volume elements.  The last image equals the restatement on it alone."""
    a8, b8, _ = bench_frames(8)
    a = torch.cat([torch.roll(a8, k, dims=3) for k in range(8)])
    b = torch.cat([torch.roll(b8, k, dims=3) for k in range(8)])
    vol = tx.census_vol(a, b, 128, (7, 9), 9)
    assert vol.numel() > 2 ** 31
    got = tx.disparity_check(vol, 1, 16.0)
    ref = tx.disparity_check_pytorch(vol[-1:].clone(), 1, 16.0)
    assert_check_equal(tuple(t[-1:] for t in got), ref, "batch 64, last image")


@pytest.mark.gpu
def test_deterministic_streams_capture_3d_and_module(tx):
    vol = cu(coarse(np.random.RandomState(6), (3, 48, 20, 200), np.float32))
    ref = tx.disparity_check(vol, 1, 0.5)
    assert_check_equal(ref, tx.disparity_check_pytorch(vol, 1, 0.5), "eager")
    assert_check_equal(tx.disparity_check(vol, 1, 0.5), ref, "again")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        on_s = tx.disparity_check(vol, 1, 0.5)
    s.synchronize()
    assert_check_equal(on_s, ref, "side stream")
    outs = [torch.zeros_like(ref[0]), torch.zeros_like(ref[1]), None, None, torch.zeros(ref[2].shape, dtype=torch.uint8, device=DEV)]
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        call_abi(vol, outs, 1, 0.5, True)
    for _ in range(3):
        for o in outs:
            if o is not None:
                o.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert_check_equal((outs[0], outs[1], outs[4].bool()), ref, "graph replay")
    d3 = tx.disparity_check(vol[1], 1, 0.5)
    assert d3[0].shape == (1, 20, 200)
    assert_check_equal(d3, tuple(t[1] for t in ref), "[D,H,W] input")
    m = tx.DisparityCheck(1, 0.5)
    got = m(vol)
    assert_check_equal(got, ref, "module")
    assert not got[0].requires_grad and got[0].device == vol.device


@pytest.mark.gpu
def test_errors_and_empty(tx):
    from connecting_the_dots_b200 import _lib
    vol = torch.rand(1, 8, 16, 20, device=DEV)
    with pytest.raises(RuntimeError, match="uniqueness"):
        tx.disparity_check(vol, 1, -1.0)
    with pytest.raises(RuntimeError):
        tx.disparity_check(vol.transpose(2, 3))
    with pytest.raises(RuntimeError):
        tx.disparity_check(vol[0, 0])
    with pytest.raises(NotImplementedError):
        tx.disparity_check(vol.half())
    with pytest.raises(_lib.CtdError, match="D = 0"):
        tx.disparity_check(torch.rand(1, 0, 16, 20, device=DEV))
    with pytest.raises(_lib.CtdError, match="overlaps vol"):
        call_abi(vol, (vol, None, None, None, None), 1, 0.0, True)
    d, s, ok = tx.disparity_check(torch.rand(0, 8, 16, 20, device=DEV))
    assert d.shape == s.shape == ok.shape == (0, 1, 16, 20)
    assert tx.disparity_check(torch.rand(2, 0, 0, 20, device=DEV))[2].shape == (2, 1, 0, 20)


@pytest.mark.gpu
def test_end_to_end_against_ground_truth(tx):
    """synth.make_batch(2), census 7x9 at block 9, D = 128, ta against pat_lcn, interior rows and columns 9..-9.  A CPU probe of
    the definition gave: all pixels 0.614 within 2 px; max_diff = 1 keeps 0.633 of them at 0.822 within 2 px and rejects
    0.972 of the out-of-view pixels (w < round(gt)).  The GPU volume is bit-equal to the restatement, so these reproduce."""
    a, b, d = bench_frames(2)
    gt = cu(d["disp"])
    vol = tx.census_vol(a, b, 128, (7, 9), 9)
    disp, _, ok = tx.disparity_check(vol, 1, 0.0, subpixel=False)
    inner = (slice(None), slice(None), slice(9, -9), slice(9, -9))
    good = ((disp - gt).abs() <= 2)[inner]
    ok = ok[inner]
    out_of_view = (torch.arange(gt.shape[-1], device=DEV).view(1, 1, 1, -1) < gt.round())[inner]
    kept, acc_all, acc_kept = float(ok.float().mean()), float(good.float().mean()), float(good[ok].float().mean())
    rejected_oov = float((~ok)[out_of_view].float().mean())
    msg = "kept %.3f (probe 0.633), within 2 px: kept %.3f (0.822), all %.3f (0.614); out of view rejected %.3f (0.972)" % (
        kept, acc_kept, acc_all, rejected_oov)
    print(msg)
    assert kept >= 0.60 and acc_kept >= 0.80 and acc_all <= 0.65 and rejected_oov >= 0.95, msg
