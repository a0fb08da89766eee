"""Semi-global matching over a score volume (sgm.cu: ctd_sgm_*, torchext.sgm_aggregate / sgm_disparity).

The definition is sgm_aggregate_pytorch: the CPU tests pin it bit for bit to a pure-Python loop over pixels and paths doing
numpy scalar arithmetic in the volume's dtype.  The GPU tests hold the kernels bit for bit to the restatement run on the GPU,
and the fused winner-take-all to disparity_from_volume of the aggregated volume.
"""
import re
import subprocess

import numpy as np
import pytest
import torch

DEV = "cuda:0"
PATHS = {4: ((0, 1), (0, -1), (1, 0), (-1, 0)),
         8: ((0, 1), (0, -1), (1, 0), (-1, 0), (1, 1), (1, -1), (-1, 1), (-1, -1))}
SMALL_HW = ((1, 7), (6, 1), (5, 9), (9, 5))
PENALTIES = ((0.0, 0.0), (0.5, 0.5), (0.25, 1.5), (0.1, 0.7))


def _F():
    from connecting_the_dots_b200.torchext import functions
    return functions


def sgm_brute(vol, p1, p2, paths):
    """The definition, one pixel, one path and one disparity at a time: vol [D,H,W] -> A [D,H,W], in vol's dtype."""
    D, H, W = vol.shape
    t = vol.dtype.type
    p1, p2 = t(p1), t(p2)
    A = None
    for dy, dx in PATHS[paths]:
        L = np.zeros_like(vol)
        for h in (range(H) if dy >= 0 else range(H - 1, -1, -1)):
            for w in (range(W) if dx >= 0 else range(W - 1, -1, -1)):
                qh, qw = h - dy, w - dx
                if not (0 <= qh < H and 0 <= qw < W):
                    L[:, h, w] = vol[:, h, w]
                    continue
                lq = [L[d, qh, qw] for d in range(D)]
                M = max(lq)
                for d in range(D):
                    cand = [lq[d], M - p2] + ([lq[d - 1] - p1] if d > 0 else []) + ([lq[d + 1] - p1] if d < D - 1 else [])
                    L[d, h, w] = vol[d, h, w] + (max(cand) - M)
        A = L if A is None else A + L
    return A


def coarse(rng, shape, dtype):
    """Values on a grid of 1/4: many exact ties between disparities, neighbours and penalties."""
    return (np.round(rng.rand(*shape) * 8) / 4 - 1).astype(dtype)


# ---------------------------------------------------------------- CPU: the definition
@pytest.mark.parametrize("paths", (4, 8))
@pytest.mark.parametrize("dtype", (np.float32, np.float64))
def test_restatement_matches_brute_force(paths, dtype):
    F = _F()
    rng = np.random.RandomState(paths)
    for D in (1, 2, 5):
        for H, W in SMALL_HW:
            for p1, p2 in PENALTIES:
                for vol in (coarse(rng, (D, H, W), dtype), rng.randn(D, H, W).astype(dtype)):
                    ref = sgm_brute(vol, p1, p2, paths)
                    got = F.sgm_aggregate_pytorch(torch.from_numpy(vol), p1, p2, paths)
                    assert got.dtype == torch.from_numpy(vol).dtype and got.shape == vol.shape
                    assert np.array_equal(got.numpy(), ref), (D, H, W, p1, p2)
                    g4 = F.sgm_aggregate_pytorch(torch.from_numpy(np.stack([vol, vol[:, ::-1].copy()])), p1, p2, paths)
                    assert torch.equal(g4[0], got)


def test_sgm_api_without_gpu(tx):
    from connecting_the_dots_b200 import _lib
    F = _F()
    x = torch.rand(1, 4, 6, 7)
    for fn in (lambda: tx.sgm_aggregate(x, 0.1, 1.0), lambda: tx.sgm_disparity(x, 0.1, 1.0), lambda: tx.SGMDisparity()(x, x)):
        with pytest.raises(RuntimeError, match="no CPU implementation"):
            fn()
    m = tx.SGMDisparity()
    assert (m.n_disps, m.block_size, m.p1, m.p2, m.paths, m.subpixel) == (128, 9, 0.2, 2.0, 8, True)
    for args, msg in (((x, 0.1, 1.0, 6), "paths"), ((x, 0.5, 0.2), "penalties"), ((x, -0.1, 1.0), "penalties"),
                      ((x, 0.1, float("inf")), "penalties"), ((torch.rand(1, 0, 6, 7), 0.1, 1.0), "D >= 1")):
        with pytest.raises(RuntimeError, match=msg):
            F.sgm_aggregate_pytorch(*args)
    # the C ABI checks its arguments before any device work
    sgm = lambda *a: _lib.call("ctd_sgm_f32", *a)  # noqa: E731
    for args, msg in (((16, 1 << 20, None, None, 1, 4, 8, 8, 0.1, 1.0, 6, 1, None), "paths"),
                      ((16, 1 << 20, None, None, 1, 4, 8, 8, -0.1, 1.0, 4, 1, None), "penalties"),
                      ((16, 1 << 20, None, None, 1, 4, 8, 8, 0.5, 0.2, 4, 1, None), "penalties"),
                      ((16, 1 << 20, None, None, 1, 4, 8, 8, 0.1, float("nan"), 4, 1, None), "finite"),
                      ((16, 1 << 20, None, None, 1, 4, 8, 8, 0.1, 1e300, 4, 1, None), "finite"),
                      ((16, 1 << 20, None, None, 1, 0, 8, 8, 0.1, 1.0, 8, 1, None), "D = 0"),
                      ((16, 1 << 20, None, None, 1, 1025, 8, 8, 0.1, 1.0, 8, 1, None), "at most"),
                      ((16, 1 << 20, None, None, 1, 4, -8, 8, 0.1, 1.0, 8, 1, None), "negative size"),
                      ((16, None, None, None, 1, 4, 8, 8, 0.1, 1.0, 8, 1, None), "null pointer"),
                      ((4096, 4096 + 4 * 255, None, None, 1, 4, 8, 8, 0.1, 1.0, 8, 1, None), "overlaps")):
        with pytest.raises(_lib.CtdError, match=msg):
            sgm(*args)
    with pytest.raises(_lib.CtdError, match="paths"):
        _lib.call("ctd_sgm_f64", 16, 1 << 20, None, None, 1, 4, 8, 8, 0.1, 1.0, 2, 1, None)
    # an empty batch is a no-op, with any D
    _lib.call("ctd_sgm_f32", None, None, None, None, 0, 0, 8, 8, 0.1, 1.0, 8, 1, None)
    _lib.call("ctd_sgm_f64", None, None, None, None, 2, 4, 8, 0, 0.1, 1.0, 4, 0, None)


def test_sgm_kernels_have_no_floating_point_atomics(tx):
    """The SGM kernels own every output element (a line per lane group): no atomics at all."""
    from connecting_the_dots_b200 import _lib
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    atomics, kernels, kernel = [], set(), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            kernel = m.group(1) if re.search(r"sgm_(horizontal|lines)", m.group(1)) else None
            if kernel:
                kernels.add(kernel)
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d+\s+)?((?:ATOM|RED)[A-Z0-9_.]*)", line)
        if m and kernel:
            atomics.append((kernel, m.group(1)))
    assert len(kernels) == 2 * 6 * 3, sorted(kernels)   # {float, double} x K in {1..32} x {horizontal, lines, lines + WTA}
    assert not atomics, atomics


# ---------------------------------------------------------------- GPU
def cu(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


def gpu_volumes(dtype):
    """(name, [B,D,H,W] volume) pairs: the CPU test's shapes, odd sizes, W < D, D off multiples of 4 and 32, wide D."""
    rng = np.random.RandomState(11)
    out = []
    for D in (1, 2, 5):
        for H, W in SMALL_HW:
            out.append(("coarse D%d %dx%d" % (D, H, W), coarse(rng, (1, D, H, W), dtype)))
    for B, D, H, W in ((2, 7, 13, 37), (1, 40, 6, 11), (1, 33, 17, 29), (2, 130, 9, 21), (1, 300, 7, 5), (1, 1024, 3, 6),
                       (1, 128, 40, 70), (3, 64, 33, 1)):
        out.append(("randn %dx%dx%dx%d" % (B, D, H, W), rng.randn(B, D, H, W).astype(dtype)))
    out.append(("coarse 1x24x19x23", coarse(rng, (1, 24, 19, 23), dtype)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("paths", (4, 8))
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_aggregate_is_bit_exact(tx, paths, dtype):
    npdt = np.float32 if dtype == torch.float32 else np.float64
    for name, vol in gpu_volumes(npdt):
        v = cu(vol)
        for p1, p2 in ((0.2, 2.0), (0.0, 0.0), (0.5, 0.5)):
            got = tx.sgm_aggregate(v, p1, p2, paths)
            ref = tx.sgm_aggregate_pytorch(v, p1, p2, paths)
            assert got.dtype == dtype and got.shape == v.shape
            assert torch.equal(got, ref), "%s p1=%g p2=%g: %d values differ" % (name, p1, p2, int((got != ref).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_misaligned_base_pointers(tx, dtype):
    rng = np.random.RandomState(3)
    vol = cu(rng.randn(2, 37, 11, 29), dtype)
    buf = torch.zeros(1 + vol.numel(), dtype=dtype, device=DEV)
    v = buf[1:].view(vol.shape).copy_(vol)
    agg = torch.empty(1 + vol.numel(), dtype=dtype, device=DEV)[1:].view(vol.shape)
    disp = torch.empty(3 + 2 * 11 * 29, dtype=dtype, device=DEV)[3:].view(2, 1, 11, 29)
    assert v.data_ptr() % 16 and agg.data_ptr() % 16 and disp.data_ptr() % 16
    from connecting_the_dots_b200 import _lib
    _lib.call("ctd_sgm" + ("_f32" if dtype == torch.float32 else "_f64"), v.data_ptr(), agg.data_ptr(), disp.data_ptr(), None,
              2, 37, 11, 29, 0.2, 2.0, 8, 1, torch.cuda.current_stream().cuda_stream)
    ref = tx.sgm_aggregate_pytorch(vol, 0.2, 2.0, 8)
    assert torch.equal(agg, ref)
    assert torch.equal(disp, tx.disparity_from_volume(ref, True)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("subpixel", (True, False))
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_fused_wta_is_bit_exact(tx, subpixel, dtype):
    npdt = np.float32 if dtype == torch.float32 else np.float64
    for name, vol in gpu_volumes(npdt):
        v = cu(vol)
        for paths in (4, 8):
            d, s = tx.sgm_disparity(v, 0.2, 2.0, paths, subpixel)
            rd, rs = tx.disparity_from_volume(tx.sgm_aggregate(v, 0.2, 2.0, paths), subpixel)
            assert d.shape == rd.shape and d.dtype == dtype
            assert torch.equal(d, rd), "%s paths=%d: disparities differ at %d pixels" % (name, paths, int((d != rd).sum()))
            assert torch.equal(s, rs), "%s paths=%d: scores differ" % (name, paths)


def full_size_volume(tx, B):
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(B)
    return tx.xcorrvol(cu(d["ta"]), cu(d["pat_lcn"]), 128, 9), d


@pytest.mark.gpu
def test_full_size_batch8(tx):
    vol, _ = full_size_volume(tx, 8)
    for paths in (4, 8):
        agg = tx.sgm_aggregate(vol, 0.2, 2.0, paths)
        assert torch.equal(agg, tx.sgm_aggregate_pytorch(vol, 0.2, 2.0, paths)), "paths=%d" % paths
        d, s = tx.sgm_disparity(vol, 0.2, 2.0, paths)
        rd, rs = tx.disparity_from_volume(agg, True)
        assert torch.equal(d, rd) and torch.equal(s, rs), "paths=%d" % paths


@pytest.mark.gpu
def test_past_2_31_elements(tx):
    """Batch 64 at 480x640, D = 128: 2.5e9 elements (10 GB per volume).  The last image equals the restatement run on that
    image alone; the batch repeats the eight bench frames, shifted per copy so that the images differ."""
    vol8, _ = full_size_volume(tx, 8)
    vol = torch.cat([torch.roll(vol8, k, dims=3) for k in range(8)])
    del vol8
    assert vol.numel() > 2 ** 31
    d, s = tx.sgm_disparity(vol, 0.2, 2.0, 8)
    last = vol[-1:].clone()
    del vol
    ref = tx.sgm_aggregate_pytorch(last, 0.2, 2.0, 8)
    rd, rs = tx.disparity_from_volume(ref, True)
    assert torch.equal(d[-1:], rd) and torch.equal(s[-1:], rs)
    agg_last = tx.sgm_aggregate(last, 0.2, 2.0, 8)
    assert torch.equal(agg_last, ref)


@pytest.mark.gpu
def test_deterministic_streams_capture_null_outputs_3d_and_module(tx):
    from connecting_the_dots_b200 import _lib, synth
    d = synth.make_batch(2, 96, 256)
    a, b = cu(d["ta"]), cu(d["pat_lcn"])
    vol = tx.xcorrvol(a, b, 48, 9)
    ref = tx.sgm_disparity(vol, 0.2, 2.0)
    again = tx.sgm_disparity(vol, 0.2, 2.0)
    assert torch.equal(ref[0], again[0]) and torch.equal(ref[1], again[1])
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        on_s = tx.sgm_disparity(vol, 0.2, 2.0)
    s.synchronize()
    assert torch.equal(on_s[0], ref[0]) and torch.equal(on_s[1], ref[1])
    agg_ref = tx.sgm_aggregate(vol, 0.2, 2.0)
    agg, disp, score = torch.zeros_like(vol), torch.zeros_like(ref[0]), torch.zeros_like(ref[1])
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _lib.call("ctd_sgm_f32", vol.data_ptr(), agg.data_ptr(), disp.data_ptr(), score.data_ptr(), 2, 48, 96, 256, 0.2, 2.0, 8,
                  1, torch.cuda.current_stream().cuda_stream)
    for _ in range(3):
        agg.zero_()
        disp.zero_()
        score.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(agg, agg_ref) and torch.equal(disp, ref[0]) and torch.equal(score, ref[1])
    # disp and score are optional, each on its own
    st = torch.cuda.current_stream().cuda_stream
    nd, ns = torch.zeros_like(ref[0]), torch.zeros_like(ref[1])
    _lib.call("ctd_sgm_f32", vol.data_ptr(), agg.data_ptr(), nd.data_ptr(), None, 2, 48, 96, 256, 0.2, 2.0, 8, 1, st)
    _lib.call("ctd_sgm_f32", vol.data_ptr(), agg.data_ptr(), None, ns.data_ptr(), 2, 48, 96, 256, 0.2, 2.0, 8, 1, st)
    assert torch.equal(nd, ref[0]) and torch.equal(ns, ref[1])
    # [D,H,W] in, [1,H,W] out
    d3, s3 = tx.sgm_disparity(vol[1], 0.2, 2.0)
    assert d3.shape == (1, 96, 256) and torch.equal(d3, ref[0][1]) and torch.equal(s3, ref[1][1])
    assert torch.equal(tx.sgm_aggregate(vol[1], 0.2, 2.0), agg_ref[1])
    dm, sm = tx.SGMDisparity(48, 9)(a, b)
    assert torch.equal(dm, ref[0]) and torch.equal(sm, ref[1]) and not dm.requires_grad


@pytest.mark.gpu
def test_errors_and_empty(tx):
    from connecting_the_dots_b200 import _lib
    v = torch.rand(1, 8, 16, 20, device=DEV)
    with pytest.raises(RuntimeError, match="paths"):
        tx.sgm_aggregate(v, 0.1, 1.0, 6)
    with pytest.raises(RuntimeError, match="penalties"):
        tx.sgm_disparity(v, 1.0, 0.1)
    with pytest.raises(RuntimeError, match="penalties"):
        tx.sgm_disparity(v, -1.0, 0.1)
    with pytest.raises(RuntimeError):
        tx.sgm_aggregate(v.transpose(2, 3), 0.1, 1.0)
    with pytest.raises(RuntimeError):
        tx.sgm_aggregate(v[0, 0], 0.1, 1.0)
    with pytest.raises(NotImplementedError):
        tx.sgm_aggregate(v.half(), 0.1, 1.0)
    with pytest.raises(RuntimeError, match="D = 0"):
        tx.sgm_disparity(torch.rand(1, 0, 16, 20, device=DEV), 0.1, 1.0)
    with pytest.raises(_lib.CtdError, match="overlaps"):
        _lib.call("ctd_sgm_f32", v.data_ptr(), v.data_ptr() + 4, None, None, 1, 8, 16, 20, 0.1, 1.0, 8, 1,
                  torch.cuda.current_stream().cuda_stream)
    e = torch.rand(0, 0, 16, 20, device=DEV)
    d, s = tx.sgm_disparity(e, 0.1, 1.0)
    assert d.shape == (0, 1, 16, 20) and s.shape == (0, 1, 16, 20)
    assert tx.sgm_aggregate(torch.rand(2, 4, 0, 20, device=DEV), 0.1, 1.0).shape == (2, 4, 0, 20)


@pytest.mark.gpu
def test_end_to_end_against_ground_truth(tx):
    """synth.make_batch(2), block 9, D = 128: the fraction of interior pixels within 2 px of the ground truth, against the
    winner-take-all xcorr_disparity on the same frames.  A CPU probe of the definition on a float64 volume gave 0.842
    (8 paths) and 0.788 (4 paths) as the mean of the two frames; measured on an NVIDIA B200: see the asserts' messages."""
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(2)
    a, b, gt = cu(d["ta"]), cu(d["pat_lcn"]), cu(d["disp"])
    inner = (slice(None), slice(None), slice(9, -9), slice(140, -9))

    def frac(disp):
        return float(((disp - gt).abs() <= 2)[inner].float().mean())
    wta = frac(tx.xcorr_disparity(a, b, 128, 9)[0])
    vol = tx.xcorrvol(a, b, 128, 9)
    f8 = frac(tx.sgm_disparity(vol, 0.2, 2.0, 8)[0])
    f4 = frac(tx.sgm_disparity(vol, 0.2, 2.0, 4)[0])
    msg = "wta %.3f, 4 paths %.3f, 8 paths %.3f" % (wta, f4, f8)
    assert f8 >= 0.80 and f4 >= 0.75, msg
    assert f8 >= wta + 0.10 and f4 >= wta + 0.10, msg
