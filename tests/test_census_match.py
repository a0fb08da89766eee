"""Census-transform stereo matching (census_match.cu: ctd_census_*, torchext.census_transform / census_vol /
census_disparity).

The definitions are census_transform_pytorch and census_vol_pytorch: the CPU tests pin them bit for bit to pure-Python loops
over pixels and taps.  The GPU tests hold the kernels bit for bit to the restatements run on the GPU, and the fused
winner-take-all to disparity_from_volume of the restated volume, sub-pixel offset included (every cost is an integer).
"""
import re
import subprocess

import numpy as np
import pytest
import torch

DEV = "cuda:0"
WINDOWS = ((1, 3), (3, 1), (3, 3), (5, 5), (7, 9), (9, 7), (5, 13))


def _F():
    from connecting_the_dots_b200.torchext import functions
    return functions


def census_brute(x, wh, ww):
    """The transform one pixel and one tap at a time: x [C,H,W] -> list of Python ints (uint64 patterns) [C][H][W]."""
    C, H, W = x.shape
    rh, rw = wh // 2, ww // 2
    out = [[[0] * W for _ in range(H)] for _ in range(C)]
    for c in range(C):
        for h in range(H):
            for w in range(W):
                k, v = 0, 0
                for i in range(wh):
                    for j in range(ww):
                        if (i, j) == (rh, rw):
                            continue
                        n = x[c, min(max(h + i - rh, 0), H - 1), min(max(w + j - rw, 0), W - 1)]
                        if n < x[c, h, w]:
                            v |= 1 << k
                        k += 1
                out[c][h][w] = v
    return out


def as_unsigned(t):
    """int64 tensor -> numpy array of Python ints holding the uint64 patterns."""
    return np.vectorize(lambda v: int(v) & (2 ** 64 - 1), otypes=[object])(t.cpu().numpy())


def hamming_brute(x0, x1, D, wh, ww, bs):
    """S [D,H,W] of one image pair, one pixel, disparity and box tap at a time, from bin(a ^ b).count("1")."""
    C, H, W = x0.shape
    t0, t1 = census_brute(x0, wh, ww), census_brute(x1, wh, ww)
    hm = np.zeros((D, H, W), dtype=np.int64)
    for d in range(D):
        for h in range(H):
            for w in range(W):
                hm[d, h, w] = sum(bin(t0[c][h][w] ^ t1[c][h][max(w - d, 0)]).count("1") for c in range(C))
    r = bs // 2
    S = np.zeros_like(hm)
    for d in range(D):
        for h in range(H):
            for w in range(W):
                S[d, h, w] = sum(hm[d, min(max(h + i, 0), H - 1), min(max(w + j, 0), W - 1)]
                                 for i in range(-r, r + 1) for j in range(-r, r + 1))
    return S


def coarse(rng, shape, dtype=np.float32):
    """Values on a grid of 1/2 in [-1, 1]: many exact ties between a pixel and its taps, so < versus <= matters."""
    return (np.round(rng.rand(*shape) * 4) / 2 - 1).astype(dtype)


def box_replicate(v, bs):
    """Replicate-padded bs x bs box sum of [B,D,H,W], one tap at a time (the identity S(bs) = box(S(1)))."""
    r = bs // 2
    H, W = v.shape[-2:]
    out = torch.zeros_like(v)
    for i in range(-r, r + 1):
        for j in range(-r, r + 1):
            rows = (torch.arange(H) + i).clamp(0, H - 1)
            cols = (torch.arange(W) + j).clamp(0, W - 1)
            out += v[..., rows, :][..., cols]
    return out


# ---------------------------------------------------------------- CPU: the definition
@pytest.mark.parametrize("window", WINDOWS)
def test_transform_restatement_matches_brute_force(window):
    F = _F()
    rng = np.random.RandomState(sum(window))
    wh, ww = window
    cases = [rng.randn(1, 6, 11).astype(np.float32), coarse(rng, (3, 5, 8)), coarse(rng, (1, 2, 3)),   # H, W < window
             rng.randn(3, 4, 9)]  # float64
    nan = rng.randn(1, 5, 7).astype(np.float32)
    nan[0, 2, 3] = nan[0, 0, 0] = np.nan
    cases.append(nan)
    for x in cases:
        got = F.census_transform_pytorch(torch.from_numpy(x), window)
        assert got.dtype == torch.int64 and got.shape == x.shape
        assert (as_unsigned(got) == np.array(census_brute(x, wh, ww), dtype=object)).all(), (window, x.shape)
        assert torch.equal(F.census_transform_pytorch(torch.from_numpy(x[None]), window)[0], got)
    if wh * ww == 65:  # 64 bits: bit 63 is set for some pixel (the int64 is negative there)
        x = torch.from_numpy(rng.randn(1, 9, 20).astype(np.float32))
        assert bool((F.census_transform_pytorch(x, window) < 0).any())


def test_transform_nan_gives_zero_bits():
    F = _F()
    x = torch.randn(1, 1, 5, 5)
    x[0, 0, 2, 2] = float("nan")
    t = F.census_transform_pytorch(x, (3, 3))
    assert int(t[0, 0, 2, 2]) == 0                  # NaN centre: every comparison is false
    assert int(t[0, 0, 1, 1]) & (1 << 7) == 0       # NaN as the bottom-right tap of (1, 1)


@pytest.mark.parametrize("bs", (1, 3, 5))
def test_vol_restatement_matches_brute_force(bs):
    F = _F()
    rng = np.random.RandomState(bs)
    for C, H, W, window, D in ((1, 5, 7, (3, 3), 9), (3, 4, 6, (1, 3), 8), (1, 6, 5, (5, 5), 7), (2, 3, 9, (3, 5), 4)):
        rn = lambda: rng.randn(C, H, W).astype(np.float32)  # noqa: E731  (exact in both dtypes)
        for x0, x1 in ((rn(), rn()), (coarse(rng, (C, H, W)), coarse(rng, (C, H, W)))):
            ref = -hamming_brute(x0, x1, D, *window, bs)
            for dt in (torch.float32, torch.float64):
                got = F.census_vol_pytorch(torch.from_numpy(x0).to(dt), torch.from_numpy(x1).to(dt), D, window, bs)
                assert got.dtype == dt and got.shape == (D, H, W)
                assert np.array_equal(got.numpy(), ref.astype(got.numpy().dtype)), (C, H, W, window, D, bs)


def test_vol_box_identity():
    """census_vol_pytorch(bs) is the replicate-padded box filter of census_vol_pytorch(1)."""
    F = _F()
    rng = np.random.RandomState(7)
    a, b = torch.from_numpy(rng.randn(2, 2, 9, 13)), torch.from_numpy(rng.randn(2, 2, 9, 13))
    v1 = F.census_vol_pytorch(a, b, 16, (5, 5), 1)
    for bs in (3, 5, 9, 15):
        assert torch.equal(F.census_vol_pytorch(a, b, 16, (5, 5), bs), box_replicate(v1, bs)), bs


def test_census_api_without_gpu(tx):
    from connecting_the_dots_b200 import _lib
    F = _F()
    x = torch.rand(1, 1, 6, 7)
    for fn in (lambda: tx.census_transform(x), lambda: tx.census_vol(x, x, 4), lambda: tx.census_disparity(x, x, 4),
               lambda: tx.CensusDisparity()(x, x), lambda: tx.CensusSGMDisparity()(x, x)):
        with pytest.raises(RuntimeError, match="no CPU implementation"):
            fn()
    m = tx.CensusDisparity()
    assert (m.n_disps, m.window, m.block_size, m.subpixel) == (128, (7, 9), 9, True)
    m = tx.CensusSGMDisparity()
    assert (m.n_disps, m.window, m.block_size, m.paths, m.subpixel) == (128, (7, 9), 1, 8, True)
    for args, msg in ((((4, 9),), "odd"), (((7, 0),), "odd"), (((1, 1),), "2 to 65"), (((9, 9),), "2 to 65"),
                      (((7, 9), 4), "block_size"), (((7, 9), 17), "block_size"), (((7, 9), -1), "block_size")):
        with pytest.raises(RuntimeError, match=msg):
            F.census_vol_pytorch(x, x, 4, *args)
    with pytest.raises(RuntimeError, match="2 to 65"):
        F.census_transform_pytorch(x, (13, 7))
    with pytest.raises(RuntimeError, match="2\\^24"):
        F.census_vol_pytorch(torch.rand(1, 1300, 4, 4), torch.rand(1, 1300, 4, 4), 4, (7, 9), 15)
    with pytest.raises(RuntimeError, match="D = 0"):
        F.census_vol_pytorch(x, x, 0)
    with pytest.raises(RuntimeError, match="same shape"):
        F.census_vol_pytorch(x, torch.rand(1, 1, 6, 8), 4)
    assert F.census_vol_pytorch(torch.rand(0, 1, 6, 7), torch.rand(0, 1, 6, 7), 0).shape == (0, 0, 6, 7)
    # the C ABI checks its arguments before any device work (pointers here are never dereferenced)
    P, Q, O = 1 << 20, 1 << 30, 1 << 34
    vol = lambda *a: _lib.call("ctd_census_vol_f32", *a)  # noqa: E731
    dsp = lambda *a: _lib.call("ctd_census_disparity_f64", *a)  # noqa: E731
    tr = lambda *a: _lib.call("ctd_census_transform_f32", *a)  # noqa: E731
    for fn, args, msg in ((vol, (P, Q, O, 1, 1, 8, 8, 4, 4, 9, 1, None), "odd"),
                          (vol, (P, Q, O, 1, 1, 8, 8, 4, -7, 9, 1, None), "odd"),
                          (vol, (P, Q, O, 1, 1, 8, 8, 4, 1, 1, 1, None), "2 to 65"),
                          (vol, (P, Q, O, 1, 1, 8, 8, 4, 11, 7, 1, None), "2 to 65"),
                          (vol, (P, Q, O, 1, 1, 8, 8, 4, 7, 9, 2, None), "block_size"),
                          (vol, (P, Q, O, 1, 1, 8, 8, 4, 7, 9, 17, None), "block_size"),
                          (vol, (P, Q, O, 1, 1300, 8, 8, 4, 7, 9, 15, None), "2\\^24"),
                          (vol, (P, Q, O, 1, 1, 8, 8, 0, 7, 9, 1, None), "D = 0"),
                          (vol, (P, Q, O, 1, 1, -8, 8, 4, 7, 9, 1, None), "negative size"),
                          (vol, (P, None, O, 1, 1, 8, 8, 4, 7, 9, 1, None), "null pointer"),
                          (vol, (P, Q, None, 1, 1, 8, 8, 4, 7, 9, 1, None), "null pointer"),
                          (vol, (P, Q, P + 4 * 63, 1, 1, 8, 8, 4, 7, 9, 1, None), "overlaps"),
                          (vol, (P, Q, Q - 4 * 4 * 64 + 4, 1, 1, 8, 8, 4, 7, 9, 1, None), "overlaps"),
                          (dsp, (P, Q, O, None, 1, 1, 8, 8, 4, 7, 8, 9, 1, None), "odd"),
                          (dsp, (P, Q, O, None, 1, 1, 8, 8, 4, 7, 9, 16, 1, None), "block_size"),
                          (dsp, (P, Q, None, O, 1, 1, 8, 8, 4, 7, 9, 9, 1, None), "null pointer"),
                          (dsp, (P, Q, O, Q + 8, 1, 1, 8, 8, 4, 7, 9, 9, 1, None), "overlaps"),
                          (dsp, (P, Q, O, O + 8, 1, 1, 8, 8, 4, 7, 9, 9, 1, None), "overlaps"),
                          (tr, (P, O, 1, 1, 8, 8, 2, 3, None), "odd"),
                          (tr, (P, O, 1, 1, 8, 8, 5, 15, None), "2 to 65"),
                          (tr, (P, O, 1, -1, 8, 8, 7, 9, None), "negative size"),
                          (tr, (None, O, 1, 1, 8, 8, 7, 9, None), "null pointer"),
                          (tr, (P, P + 8, 1, 1, 8, 8, 7, 9, None), "overlaps")):
        with pytest.raises(_lib.CtdError, match=msg):
            fn(*args)
    # an empty batch is a no-op, with any D and null pointers
    _lib.call("ctd_census_vol_f32", None, None, None, 0, 1, 8, 8, 0, 7, 9, 1, None)
    _lib.call("ctd_census_disparity_f32", None, None, None, None, 2, 1, 0, 8, 0, 7, 9, 9, 1, None)
    _lib.call("ctd_census_transform_f64", None, None, 2, 1, 8, 0, 7, 9, None)


def test_census_kernels_have_no_atomics(tx):
    """The census kernels own every output element: no atomics at all."""
    from connecting_the_dots_b200 import _lib
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    atomics, kernels, kernel = [], set(), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            kernel = m.group(1) if re.search(r"census_(transform_kernel|match)I", m.group(1)) else None
            if kernel:
                kernels.add(kernel)
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d+\s+)?((?:ATOM|RED)[A-Z0-9_.]*)", line)
        if m and kernel:
            atomics.append((kernel, m.group(1)))
    assert len(kernels) == 2 * (1 + 8 * 2), sorted(kernels)   # {float, double} x (transform + R in 0..7 x {vol, WTA})
    assert not atomics, atomics


# ---------------------------------------------------------------- GPU
def cu(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


def gpu_pairs(dtype):
    """(name, in0, in1) of [B,C,H,W]: W off multiples of 4 and of 128, W < D, C = 1 and 3, coarse values and NaN."""
    rng = np.random.RandomState(5)
    out = []
    for B, C, H, W in ((1, 1, 1, 7), (2, 1, 13, 37), (1, 3, 9, 130), (1, 1, 17, 256), (3, 1, 11, 5), (1, 2, 20, 131)):
        out.append(("randn %dx%dx%dx%d" % (B, C, H, W), rng.randn(B, C, H, W), rng.randn(B, C, H, W)))
        out.append(("coarse %dx%dx%dx%d" % (B, C, H, W), coarse(rng, (B, C, H, W)), coarse(rng, (B, C, H, W))))
    nan0, nan1 = rng.randn(1, 1, 12, 40), rng.randn(1, 1, 12, 40)
    nan0[0, 0, 3, 5:9] = np.nan
    nan1[0, 0, 7, 20] = np.nan
    out.append(("nan 1x1x12x40", nan0, nan1))
    return [(n, cu(a, dtype), cu(b, dtype)) for n, a, b in out]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_transform_is_bit_exact(tx, dtype):
    for name, a, _ in gpu_pairs(dtype):
        for window in WINDOWS + ((13, 5), (1, 65), (65, 1)):
            got = tx.census_transform(a, window)
            assert got.dtype == torch.int64 and got.shape == a.shape and got.device == a.device
            assert torch.equal(got, tx.census_transform_pytorch(a, window)), "%s window %s" % (name, window)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_vol_and_disparity_are_bit_exact(tx, dtype):
    for name, a, b in gpu_pairs(dtype):
        W = a.shape[-1]
        for window, bs in (((7, 9), 1), ((7, 9), 9), ((3, 3), 3), ((5, 5), 15), ((1, 3), 5), ((9, 7), 7), ((5, 13), 1)):
            if a.shape[1] * (window[0] * window[1] - 1) * bs * bs > 1 << 24:
                continue
            for D in (1, 6, W + 5):
                ref = tx.census_vol_pytorch(a, b, D, window, bs)
                got = tx.census_vol(a, b, D, window, bs)
                assert got.dtype == dtype and got.shape == ref.shape
                assert torch.equal(got, ref), "%s %s bs %d D %d: %d values differ" % (name, window, bs, D, int((got != ref).sum()))
                for subpixel in (True, False):
                    d, s = tx.census_disparity(a, b, D, window, bs, subpixel)
                    rd, rs = tx.disparity_from_volume(ref, subpixel)
                    assert torch.equal(d, rd), "%s %s bs %d D %d sub %d: disparities differ" % (name, window, bs, D, subpixel)
                    assert torch.equal(s, rs), "%s %s bs %d D %d: scores differ" % (name, window, bs, D)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_misaligned_views(tx, dtype):
    """Every pointer one element off a 16-byte boundary, W a multiple of 4 (so only the pointers break alignment)."""
    from connecting_the_dots_b200 import _lib
    rng = np.random.RandomState(9)
    shape = (2, 1, 19, 68)
    n = int(np.prod(shape))

    def view(src, dt=dtype, count=n):
        buf = torch.zeros(1 + count, dtype=dt, device=DEV)
        v = buf[1:]
        if src is not None:
            v.copy_(src.reshape(-1))
        return v
    a, b = cu(rng.randn(*shape), dtype), cu(rng.randn(*shape), dtype)
    va, vb = view(a), view(b)
    assert va.data_ptr() % 16 and vb.data_ptr() % 16
    st = torch.cuda.current_stream().cuda_stream
    sfx = "_f32" if dtype == torch.float32 else "_f64"
    t = view(None, torch.int64)
    _lib.call("ctd_census_transform" + sfx, va.data_ptr(), t.data_ptr(), *shape, 7, 9, st)
    assert torch.equal(t.view(shape), tx.census_transform_pytorch(a, (7, 9)))
    for bs in (1, 9):
        D = 24
        out = view(None, dtype, 2 * D * 19 * 68)
        _lib.call("ctd_census_vol" + sfx, va.data_ptr(), vb.data_ptr(), out.data_ptr(), *shape, D, 7, 9, bs, st)
        ref = tx.census_vol_pytorch(a, b, D, (7, 9), bs)
        assert torch.equal(out.view(ref.shape), ref), bs
        dp, sc = view(None, dtype, 2 * 19 * 68), view(None, dtype, 2 * 19 * 68)
        _lib.call("ctd_census_disparity" + sfx, va.data_ptr(), vb.data_ptr(), dp.data_ptr(), sc.data_ptr(), *shape, D, 7, 9, bs, 1, st)
        rd, rs = tx.disparity_from_volume(ref, True)
        assert torch.equal(dp.view(rd.shape), rd) and torch.equal(sc.view(rs.shape), rs), bs


def bench_frames(B):
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(B)
    return cu(d["ta"]), cu(d["pat_lcn"]), d


@pytest.mark.gpu
def test_full_size_batch8(tx):
    a, b, _ = bench_frames(8)
    for bs in (1, 9):
        ref = tx.census_vol_pytorch(a, b, 128, (7, 9), bs)
        assert torch.equal(tx.census_vol(a, b, 128, (7, 9), bs), ref), bs
        d, s = tx.census_disparity(a, b, 128, (7, 9), bs)
        rd, rs = tx.disparity_from_volume(ref, True)
        del ref
        assert torch.equal(d, rd) and torch.equal(s, rs), bs


@pytest.mark.gpu
def test_past_2_31_elements(tx):
    """Batch 64 at 480x640, D = 128: 2.5e9 volume elements.  The last image equals the restatement run on it alone; the
    batch repeats the eight bench frames, shifted per copy so that the images differ."""
    a8, b8, _ = bench_frames(8)
    a = torch.cat([torch.roll(a8, k, dims=3) for k in range(8)])
    b = torch.cat([torch.roll(b8, k, dims=3) for k in range(8)])
    vol = tx.census_vol(a, b, 128, (7, 9), 1)
    assert vol.numel() > 2 ** 31
    last = vol[-1:].clone()
    del vol
    assert torch.equal(last, tx.census_vol_pytorch(a[-1:], b[-1:], 128, (7, 9), 1))
    d, s = tx.census_disparity(a, b, 128, (7, 9), 9)
    rd, rs = tx.disparity_from_volume(tx.census_vol_pytorch(a[-1:], b[-1:], 128, (7, 9), 9), True)
    assert torch.equal(d[-1:], rd) and torch.equal(s[-1:], rs)


@pytest.mark.gpu
def test_sgm_over_census_volume(tx):
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(2, 64, 160)
    a, b = cu(d["ta"]), cu(d["pat_lcn"])
    got = tx.sgm_disparity(tx.census_vol(a, b, 48, (7, 9), 1), 10, 120, 8)
    ref = tx.disparity_from_volume(tx.sgm_aggregate_pytorch(tx.census_vol_pytorch(a, b, 48, (7, 9), 1), 10, 120, 8))
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])


@pytest.mark.gpu
def test_deterministic_streams_capture_null_score_3d_and_modules(tx):
    from connecting_the_dots_b200 import _lib, synth
    d = synth.make_batch(2, 96, 256)
    a, b = cu(d["ta"]), cu(d["pat_lcn"])
    ref = tx.census_disparity(a, b, 48)
    again = tx.census_disparity(a, b, 48)
    assert torch.equal(ref[0], again[0]) and torch.equal(ref[1], again[1])
    vref = tx.census_vol(a, b, 48)
    assert torch.equal(vref, tx.census_vol(a, b, 48))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        on_s = tx.census_disparity(a, b, 48)
        von_s = tx.census_vol(a, b, 48)
    s.synchronize()
    assert torch.equal(on_s[0], ref[0]) and torch.equal(on_s[1], ref[1]) and torch.equal(von_s, vref)
    vol, disp, score = torch.zeros_like(vref), torch.zeros_like(ref[0]), torch.zeros_like(ref[1])
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        st = torch.cuda.current_stream().cuda_stream
        _lib.call("ctd_census_vol_f32", a.data_ptr(), b.data_ptr(), vol.data_ptr(), 2, 1, 96, 256, 48, 7, 9, 1, st)
        _lib.call("ctd_census_disparity_f32", a.data_ptr(), b.data_ptr(), disp.data_ptr(), score.data_ptr(), 2, 1, 96, 256, 48,
                  7, 9, 9, 1, st)
    for _ in range(3):
        vol.zero_()
        disp.zero_()
        score.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(vol, vref) and torch.equal(disp, ref[0]) and torch.equal(score, ref[1])
    # score is optional
    nd = torch.zeros_like(ref[0])
    _lib.call("ctd_census_disparity_f32", a.data_ptr(), b.data_ptr(), nd.data_ptr(), None, 2, 1, 96, 256, 48, 7, 9, 9, 1,
              torch.cuda.current_stream().cuda_stream)
    assert torch.equal(nd, ref[0])
    # [C,H,W] in, [1,H,W] / [D,H,W] / [C,H,W] out
    d3, s3 = tx.census_disparity(a[1], b[1], 48)
    assert d3.shape == (1, 96, 256) and torch.equal(d3, ref[0][1]) and torch.equal(s3, ref[1][1])
    assert torch.equal(tx.census_vol(a[1], b[1], 48), vref[1])
    assert torch.equal(tx.census_transform(a[1]), tx.census_transform(a)[1])
    dm, sm = tx.CensusDisparity(48)(a, b)
    assert torch.equal(dm, ref[0]) and torch.equal(sm, ref[1]) and not dm.requires_grad
    m = tx.CensusSGMDisparity(48)
    dm, sm = m(a, b)
    rd, rs = tx.sgm_disparity(vref, m.p1, m.p2, 8)
    assert torch.equal(dm, rd) and torch.equal(sm, rs)
    # outputs live on the inputs' device
    assert dm.device == a.device and tx.census_transform(a).device == a.device


@pytest.mark.gpu
def test_errors_and_empty(tx):
    from connecting_the_dots_b200 import _lib
    a = torch.rand(1, 1, 16, 20, device=DEV)
    with pytest.raises(RuntimeError, match="odd"):
        tx.census_vol(a, a, 8, (4, 9))
    with pytest.raises(RuntimeError, match="block_size"):
        tx.census_disparity(a, a, 8, (7, 9), 4)
    with pytest.raises(RuntimeError, match="2 to 65"):
        tx.census_transform(a, (9, 9))
    with pytest.raises(RuntimeError, match="D = 0"):
        tx.census_vol(a, a, 0)
    with pytest.raises(RuntimeError):
        tx.census_vol(a, a.double(), 8)
    with pytest.raises(RuntimeError):
        tx.census_vol(a, torch.rand(1, 1, 16, 21, device=DEV), 8)
    with pytest.raises(RuntimeError):
        tx.census_vol(a.transpose(2, 3), a.transpose(2, 3), 8)
    with pytest.raises(NotImplementedError):
        tx.census_vol(a.half(), a.half(), 8)
    with pytest.raises(NotImplementedError):
        tx.census_transform(a.half())
    with pytest.raises(_lib.CtdError, match="overlaps"):
        _lib.call("ctd_census_vol_f32", a.data_ptr(), a.data_ptr(), a.data_ptr() + 64, 1, 1, 16, 20, 1, 7, 9, 1,
                  torch.cuda.current_stream().cuda_stream)
    e = torch.rand(0, 1, 16, 20, device=DEV)
    d, s = tx.census_disparity(e, e, 8)
    assert d.shape == (0, 1, 16, 20) and s.shape == (0, 1, 16, 20)
    assert tx.census_vol(torch.rand(2, 1, 0, 20, device=DEV), torch.rand(2, 1, 0, 20, device=DEV), 4).shape == (2, 4, 0, 20)
    assert tx.census_transform(e).shape == e.shape


@pytest.mark.gpu
def test_end_to_end_against_ground_truth(tx):
    """synth.make_batch(2), 7x9 census, D = 128, the interior of the SGM test: the fraction of pixels within 2 px of the
    ground truth.  A CPU probe of the definition gave 0.681 for winner-take-all at block 9 and, for CensusSGMDisparity's
    defaults, p1 = 6, p2 = 400, 0.911 (8 paths) and 0.913 (4 paths); the GPU results are bit-equal to the definition."""
    a, b, d = bench_frames(2)
    gt = cu(d["disp"])
    inner = (slice(None), slice(None), slice(9, -9), slice(140, -9))

    def frac(disp):
        return float(((disp - gt).abs() <= 2)[inner].float().mean())
    wta = frac(tx.census_disparity(a, b, 128, (7, 9), 9)[0])
    f8 = frac(tx.CensusSGMDisparity(128)(a, b)[0])
    f4 = frac(tx.CensusSGMDisparity(128, paths=4)(a, b)[0])
    msg = "wta %.3f (probe 0.681), 8 paths %.3f (probe 0.911), 4 paths %.3f (probe 0.913)" % (wta, f8, f4)
    assert wta >= 0.66 and f8 >= 0.83 and f4 >= 0.77, msg
