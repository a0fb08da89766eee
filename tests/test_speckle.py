"""Speckle filter of disparity maps (speckle.cu: ctd_speckle_filter_*, torchext.speckle_filter / speckle_filter_pytorch).

The definition is speckle_filter_pytorch: the CPU tests pin it bit for bit to scipy's connected_components and to a
breadth-first search over pixels.  The GPU tests hold the kernels bit for bit to the restatement run on the GPU, over
synthetic maps built to stress the labelling (components across tile borders, a spiral and a snake that cover the image,
checkerboards, odd sizes) and over the disparities of the library's matchers.
"""
import collections
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


def edges(d, ok, max_diff):
    """The adjacency of the definition over one image d [H,W] (numpy): (src, dst) flat pixel indices."""
    H, W = d.shape
    idx = np.arange(H * W).reshape(H, W)
    d = d.astype(np.float64)
    src, dst = [], []
    for a, b in ((np.s_[:, :-1], np.s_[:, 1:]), (np.s_[:-1, :], np.s_[1:, :])):
        with np.errstate(invalid="ignore"):
            m = ok[a] & ok[b] & (np.abs(d[a] - d[b]) <= max_diff)
        src.append(idx[a][m])
        dst.append(idx[b][m])
    return np.concatenate(src), np.concatenate(dst)


def speckle_scipy(d, ok, max_size, max_diff):
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    H, W = d.shape
    n = H * W
    s, t = edges(d, ok, max_diff)
    _, lab = connected_components(coo_matrix((np.ones(len(s)), (s, t)), shape=(n, n)), directed=False)
    return ok & (np.bincount(lab)[lab].reshape(H, W) > max_size)


def speckle_bfs(d, ok, max_size, max_diff):
    """The definition one pixel at a time: breadth-first search from every unvisited valid pixel."""
    H, W = d.shape
    out = np.zeros((H, W), bool)
    seen = np.zeros((H, W), bool)
    for h0, w0 in itertools.product(range(H), range(W)):
        if seen[h0, w0] or not ok[h0, w0]:
            continue
        comp, queue = [], collections.deque([(h0, w0)])
        seen[h0, w0] = True
        while queue:
            h, w = queue.popleft()
            comp.append((h, w))
            for hh, ww in ((h + 1, w), (h - 1, w), (h, w + 1), (h, w - 1)):
                if 0 <= hh < H and 0 <= ww < W and not seen[hh, ww] and ok[hh, ww] and \
                        abs(float(d[h, w]) - float(d[hh, ww])) <= max_diff:
                    seen[hh, ww] = True
                    queue.append((hh, ww))
        for p in comp:
            out[p] = len(comp) > max_size
    return out


def random_map(rng, H, W, dtype, nan_frac=0.0):
    """Disparities on a grid of 1/2 in [0, 4]: many differences of exactly 0, 0.5 and 1, so the <= max_diff edge matters."""
    d = (np.round(rng.rand(H, W) * 8) / 2).astype(dtype)
    if nan_frac:
        d[rng.rand(H, W) < nan_frac] = np.nan
    return d


CPU_SHAPES = ((1, 1), (1, 12), (12, 1), (2, 3), (3, 7), (5, 5), (8, 11), (12, 12))
MAX_SIZES = (0, 1, 3, 1 << 40)


def test_restatement_matches_scipy_and_bfs():
    F = _F()
    rng = np.random.RandomState(5)
    for dtype, (H, W), density in itertools.product((np.float32, np.float64), CPU_SHAPES, (0.0, 0.3, 0.7, 1.0)):
        d = random_map(rng, H, W, dtype, nan_frac=0.1 if density == 0.7 else 0.0)
        ok = rng.rand(H, W) < density
        for max_diff in (0.0, 0.5, 1.0):
            for max_size in MAX_SIZES:
                msg = "%s %dx%d density %g max_diff %g max_size %d" % (dtype.__name__, H, W, density, max_diff, max_size)
                ref = speckle_scipy(d, ok, max_size, max_diff)
                assert np.array_equal(speckle_bfs(d, ok, max_size, max_diff), ref), msg
                got = F.speckle_filter_pytorch(torch.from_numpy(d)[None, None], torch.from_numpy(ok)[None, None],
                                               max_size, max_diff)
                assert got.dtype == torch.bool and got.shape == (1, 1, H, W), msg
                assert np.array_equal(got[0, 0].numpy(), ref), msg


def test_restatement_special_cases():
    F = _F()
    t = lambda a, dt=torch.float32: torch.tensor(a, dtype=dt).view(1, 1, 1, -1)  # noqa: E731
    # value chains: 0, 1, 2 with max_diff = 1 is one component of three, although |0 - 2| > 1
    assert F.speckle_filter_pytorch(t([0.0, 1.0, 2.0]), None, 2, 1.0).all()
    assert not F.speckle_filter_pytorch(t([0.0, 1.0, 2.5]), None, 2, 1.0).any()
    # differences exactly at max_diff join; the fp64 difference of float32 values decides
    assert F.speckle_filter_pytorch(t([0.5, 0.75]), None, 1, 0.25).all()
    a, b = np.float32(0.1), np.float32(0.2)
    assert float(np.float64(b) - np.float64(a)) > 0.1   # 0.10000000149...
    assert not F.speckle_filter_pytorch(t([a, b]), None, 1, 0.1).any()
    assert F.speckle_filter_pytorch(t([a, b]), None, 1, float(np.float64(b) - np.float64(a))).all()
    # NaN is adjacent to nothing, not even to NaN; inf - inf is NaN too
    assert torch.equal(F.speckle_filter_pytorch(t([np.nan, np.nan, 1.0, 1.0]), None, 1, 1.0), t([0, 0, 1, 1], torch.bool))
    assert not F.speckle_filter_pytorch(t([np.inf, np.inf]), None, 1, 1.0).any()
    # all invalid, all valid, valid=None, max_size = 0
    rng = np.random.RandomState(8)
    d = torch.from_numpy(random_map(rng, 3, 2 * 7, np.float64)).view(2, 1, 3, 7)
    assert not F.speckle_filter_pytorch(d, torch.zeros(d.shape, dtype=torch.bool), 0, 1.0).any()
    allv = torch.ones(d.shape, dtype=torch.bool)
    assert torch.equal(F.speckle_filter_pytorch(d, allv, 2, 0.5), F.speckle_filter_pytorch(d, None, 2, 0.5))
    assert F.speckle_filter_pytorch(d, None, 0, 0.0).all()
    assert F.speckle_filter_pytorch(d, allv, 3 * 7 - 1, 1e9).all() and not F.speckle_filter_pytorch(d, allv, 3 * 7, 1e9).any()
    ok = torch.from_numpy(rng.rand(2, 1, 3, 7) < 0.5)
    assert torch.equal(F.speckle_filter_pytorch(d, ok, 0, 0.5), ok)
    # images of a batch are separate; 3-D input
    for i in range(2):
        ref = speckle_scipy(d[i, 0].numpy(), ok[i, 0].numpy(), 2, 0.5)
        assert np.array_equal(F.speckle_filter_pytorch(d, ok, 2, 0.5)[i, 0].numpy(), ref)
        got3 = F.speckle_filter_pytorch(d[i], ok[i], 2, 0.5)
        assert got3.shape == (1, 3, 7) and np.array_equal(got3[0].numpy(), ref)


def test_speckle_api_without_gpu(tx):
    from connecting_the_dots_b200 import _lib
    F = _F()
    d = torch.rand(2, 1, 5, 6)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        tx.speckle_filter(d)
    for bad, exc, msg in (((torch.rand(2, 2, 5, 6),), RuntimeError, "1 x H x W"),
                          ((torch.rand(5, 6),), RuntimeError, "1 x H x W"),
                          ((d.half(),), NotImplementedError, "not implemented"),
                          ((d.int(),), NotImplementedError, "not implemented"),
                          ((d, torch.ones(2, 1, 5, 6)), RuntimeError, "bool"),
                          ((d, torch.ones(2, 1, 6, 5, dtype=torch.bool)), RuntimeError, "bool"),
                          ((d, None, -1), RuntimeError, "max_size"),
                          ((d, None, 2.5), RuntimeError, "max_size"),
                          ((d, None, 3, -0.5), RuntimeError, "max_diff"),
                          ((d, None, 3, float("nan")), RuntimeError, "max_diff"),
                          ((d, None, 3, float("inf")), RuntimeError, "max_diff")):
        with pytest.raises(exc, match=msg):
            F.speckle_filter_pytorch(*bad)
    # the C ABI checks its arguments before any device work (pointers here are never dereferenced)
    P, O = 1 << 30, 1 << 34
    n = 2 * 5 * 6
    f32 = lambda *a: _lib.call("ctd_speckle_filter_f32", *a)  # noqa: E731
    f64 = lambda *a: _lib.call("ctd_speckle_filter_f64", *a)  # noqa: E731
    for fn, args, msg in ((f32, (P, None, O, -2, 5, 6, 3, 1.0, None), "negative size"),
                          (f32, (P, None, O, 2, -5, 6, 3, 1.0, None), "negative size"),
                          (f64, (P, None, O, 2, 5, -6, 3, 1.0, None), "negative size"),
                          (f32, (P, None, O, 1, 1 << 16, 1 << 15, 3, 1.0, None), "INT32_MAX"),
                          (f32, (P, None, O, 1, 3, 1 << 31, 3, 1.0, None), "INT32_MAX"),
                          (f32, (P, None, O, 2, 5, 6, -1, 1.0, None), "max_size"),
                          (f64, (P, None, O, 2, 5, 6, 3, -1.0, None), "max_diff"),
                          (f64, (P, None, O, 2, 5, 6, 3, float("nan"), None), "max_diff"),
                          (f32, (P, None, O, 2, 5, 6, 3, float("inf"), None), "max_diff"),
                          (f32, (None, None, O, 2, 5, 6, 3, 1.0, None), "null pointer"),
                          (f32, (None, None, None, 2, 5, 6, 3, 1.0, None), "null pointer"),
                          (f32, (P, None, P + 4 * n - 1, 2, 5, 6, 3, 1.0, None), "overlaps disp"),
                          (f64, (P, None, P - n + 1, 2, 5, 6, 3, 1.0, None), "overlaps disp"),
                          (f32, (P, O, O + n - 1, 2, 5, 6, 3, 1.0, None), "overlaps valid"),
                          (f64, (P, O, O - n + 1, 2, 5, 6, 3, 1.0, None), "overlaps valid")):
        with pytest.raises(_lib.CtdError, match=msg):
            fn(*args)
    # an empty batch is a no-op with null pointers; valid_out = NULL is a no-op
    f32(None, None, None, 0, 5, 6, 3, 1.0, None)
    f64(None, None, None, 2, 0, 6, 3, 1.0, None)
    f32(None, None, None, 2, 5, 0, 3, 1.0, None)
    f32(P, O, None, 2, 5, 6, 3, 1.0, None)


def test_speckle_kernels_have_no_float_atomics(tx):
    """Unions and sizes use integer atomics (min and add on int32); no floating-point atomic anywhere in the kernels."""
    from connecting_the_dots_b200 import _lib
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    atomics, kernels, kernel = [], set(), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            kernel = m.group(1) if "speckle_" in m.group(1) else None
            if kernel:
                kernels.add(kernel)
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d+\s+)?((?:ATOM|RED)[A-Z0-9_.]*)", line)
        if m and kernel:
            atomics.append((kernel, m.group(1)))
    assert len(kernels) == 6, sorted(kernels)   # tiles and merge for float and double, sizes, mark
    assert atomics, "the unions are atomic"
    fp = [a for a in atomics if re.search(r"\.(BF16|F16|F32|F64|FTZ)", a[1])]
    assert not fp, fp


# ---------------------------------------------------------------- GPU
def cu(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


def assert_same(got, ref, msg):
    assert got.dtype == torch.bool and got.shape == ref.shape, "%s: %s %s vs %s" % (msg, got.dtype, tuple(got.shape), tuple(ref.shape))
    assert torch.equal(got, ref), "%s: %d of %d pixels differ" % (msg, int((got != ref).sum()), got.numel())


def check(tx, disp, valid, settings, msg):
    for max_size, max_diff in settings:
        ref = tx.speckle_filter_pytorch(disp, valid, max_size, max_diff)
        assert_same(tx.speckle_filter(disp, valid, max_size, max_diff), ref, "%s max_size %d max_diff %g" % (msg, max_size, max_diff))


def blocks_map(rng, B, H, W, cell):
    """Piecewise-constant disparities on cells of `cell` pixels with +-0.5 noise: components of many sizes and shapes that
    cross 32-pixel tile borders in both directions."""
    coarse = rng.randint(0, 6, size=(B, 1, -(-H // cell), -(-W // cell))).astype(np.float64)
    d = np.repeat(np.repeat(coarse, cell, axis=2), cell, axis=3)[:, :, :H, :W]
    return d + np.round(rng.rand(B, 1, H, W) * 2) / 4


SETTINGS = ((0, 1.0), (1, 0.0), (3, 0.25), (50, 0.5), (200, 1.0), (1 << 40, 1.0))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_bit_exact_on_synthetic_maps(tx, dtype):
    rng = np.random.RandomState(11)
    for (B, H, W), cell in itertools.product(((3, 100, 130), (2, 257, 300), (1, 64, 64)), (1, 5, 17, 40)):
        d = cu(blocks_map(rng, B, H, W, cell), dtype)
        for density in (1.0, 0.8, 0.3):
            ok = None if density == 1.0 else cu(rng.rand(B, 1, H, W) < density)
            check(tx, d, ok, SETTINGS, "%dx%dx%d cell %d density %g" % (B, H, W, cell, density))
    d = cu(blocks_map(rng, 2, 70, 90, 7), dtype)
    d[0, 0, rng.rand(70, 90) < 0.2] = float("nan")
    d[1, 0, :, 40] = float("inf")
    check(tx, d, None, SETTINGS, "NaN and inf")


def spiral(H, W):
    """A one-pixel-wide path (0) that spirals in from the border through one-pixel walls (10): ring r = min(h, w, H-1-h,
    W-1-w) is path for even r and wall for odd r; a gap in each wall ring leads to the next path ring, and a cut next to it
    turns each ring into one leg of a single spiral."""
    h, w = np.mgrid[:H, :W]
    r = np.minimum(np.minimum(h, w), np.minimum(H - 1 - h, W - 1 - w))
    d = np.where(r % 2 == 0, 0.0, 10.0)
    for k in range(0, min(H, W) // 2, 2):
        if k + 2 < H - 1 - k and k + 1 < W - 1 - k:
            d[k + 2, k + 1] = 0.0    # gap in wall ring k + 1
            d[k + 1, k] = 10.0       # cut in path ring k
    return d


def snake(H, W):
    """Even rows are path (0), odd rows walls (10) with one gap at alternating ends: one path through every even row."""
    d = np.where(np.arange(H)[:, None] % 2 == 0, 0.0, 10.0) * np.ones((1, W))
    d[1::4, W - 1] = 0.0
    d[3::4, 0] = 0.0
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_spiral_snake_and_checkerboard(tx, dtype):
    """The longest paths a 480x640 image holds (deep union-find trees, long find chains) and all-singleton components."""
    H, W = 480, 640
    maps = np.stack([spiral(H, W), snake(H, W), spiral(W, H).T])[:, None]
    d = cu(maps, dtype)
    path = tx.speckle_filter_pytorch(d, None, 10000, 0.5) & (d == 0)
    for i in range(3):   # each path is one component that covers about half of the image
        assert int(path[i].sum()) == int((d[i] == 0).sum()) > H * W // 3, "map %d is not one path" % i
    check(tx, d, None, ((0, 0.5), (10000, 0.5), (H * W // 2, 0.5), (H * W, 20.0), (H * W - 1, 20.0)), "spiral/snake")
    ok = cu(np.random.RandomState(1).rand(3, 1, H, W) < 0.999)
    check(tx, d, ok, ((100, 0.5),), "spiral/snake, a few pixels invalid")
    board = cu(((np.arange(H)[:, None] + np.arange(W)[None]) % 2 * 3.0)[None, None], dtype)
    for max_size, max_diff in ((0, 1.0), (1, 1.0), (1, 3.0)):
        got = tx.speckle_filter(board, None, max_size, max_diff)
        assert_same(got, tx.speckle_filter_pytorch(board, None, max_size, max_diff), "checkerboard %d %g" % (max_size, max_diff))
    assert tx.speckle_filter(board, None, 0, 1.0).all() and not tx.speckle_filter(board, None, 1, 1.0).any()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_odd_sizes(tx, dtype):
    """H and W of 1, 31, 33, 257 and 4097: partial tiles, one-row and one-column images."""
    rng = np.random.RandomState(2)
    sizes = (1, 31, 33, 257, 4097)
    for H, W in itertools.product(sizes, sizes):
        if H * W > 257 * 4097:
            continue
        B = 2 if H * W < 1 << 16 else 1
        d = cu(blocks_map(rng, B, H, W, 3), dtype)
        ok = cu(rng.rand(B, 1, H, W) < 0.9)
        check(tx, d, ok, ((0, 0.5), (2, 0.5), (40, 1.0)), "%dx%d" % (H, W))


def bench_frames(B):
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(B)
    return cu(d["ta"]), cu(d["pat_lcn"]), d


def pipeline_disparities(tx, a, b):
    """(name, disp, valid) of the matchers on the bench frames, D = 128, 7x9 census, integer disparities."""
    wta = tx.census_disparity(a, b, 128, (7, 9), 9, subpixel=False)[0]
    cd, _, cok = tx.disparity_check(tx.census_vol(a, b, 128, (7, 9), 9), 1, 0.0, subpixel=False)
    sgm = tx.sgm_disparity(tx.census_vol(a, b, 128, (7, 9), 1), 6, 400, 8, subpixel=False)[0]
    return (("census bs9 WTA", wta, None), ("census bs9 checked", cd, cok), ("census bs1 sgm", sgm, None))


@pytest.mark.gpu
def test_real_pipelines_batch8(tx):
    """480x640, batch 8: census block-9 WTA with and without disparity_check, census block 1 -> sgm_disparity."""
    a, b, _ = bench_frames(8)
    for name, disp, ok in pipeline_disparities(tx, a, b):
        check(tx, disp, ok, ((50, 1.0), (200, 1.0), (200, 0.0)), name)
    sub = tx.sgm_disparity(tx.census_vol(a, b, 128, (7, 9), 1), 6, 400, 8)[0]
    check(tx, sub, None, ((200, 1.0),), "census bs1 sgm, sub-pixel")
    check(tx, sub.double(), None, ((200, 0.5),), "census bs1 sgm, sub-pixel, float64")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_misaligned_views(tx, dtype):
    """disp, valid and valid_out one element off any alignment; W = 67 (rows not aligned to each other either)."""
    from connecting_the_dots_b200 import _lib
    rng = np.random.RandomState(4)
    B, H, W = 2, 45, 67
    d = cu(blocks_map(rng, B, H, W, 4), dtype)
    ok = cu(rng.rand(B, 1, H, W) < 0.85)
    n = B * H * W

    def view(src, dt):
        v = torch.zeros(1 + n, dtype=dt, device=DEV)[1:]
        if src is not None:
            v.copy_(src.reshape(-1))
        return v
    dv, okv, out = view(d, dtype), view(ok, torch.uint8), view(None, torch.uint8)
    assert dv.data_ptr() % 16 and okv.data_ptr() % 2 and out.data_ptr() % 2
    _lib.call("ctd_speckle_filter" + ("_f32" if dtype == torch.float32 else "_f64"), dv.data_ptr(), okv.data_ptr(),
              out.data_ptr(), B, H, W, 20, 0.5, torch.cuda.current_stream().cuda_stream)
    assert_same(out.view(B, 1, H, W).bool(), tx.speckle_filter_pytorch(d, ok, 20, 0.5), "misaligned views")


@pytest.mark.gpu
def test_past_2_31_pixels(tx):
    """2049 images of 1024x1024: 2.15e9 pixels.  The last image equals a call on it alone and the restatement."""
    B, H, W = 2049, 1024, 1024
    assert B * H * W > 2 ** 31
    g = torch.Generator(device=DEV).manual_seed(3)
    d = torch.randint(0, 3, (B, 1, H, W), device=DEV, generator=g, dtype=torch.float32)
    ok = torch.rand(B, 1, H, W, device=DEV, generator=g) < 0.9
    got = tx.speckle_filter(d, ok, 20, 0.0)
    last = tx.speckle_filter(d[-1:].clone(), ok[-1:].clone(), 20, 0.0)
    assert_same(got[-1:], last, "batch 2049, last image vs alone")
    assert_same(last, tx.speckle_filter_pytorch(d[-1:], ok[-1:], 20, 0.0), "last image vs restatement")


@pytest.mark.gpu
def test_deterministic_streams_capture_and_3d(tx):
    from connecting_the_dots_b200 import _lib
    rng = np.random.RandomState(6)
    d = cu(blocks_map(rng, 3, 200, 300, 6), torch.float32)
    ok = cu(rng.rand(3, 1, 200, 300) < 0.9)
    ref = tx.speckle_filter_pytorch(d, ok, 30, 0.5)
    for i in range(3):
        assert_same(tx.speckle_filter(d, ok, 30, 0.5), ref, "call %d" % i)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        on_s = tx.speckle_filter(d, ok, 30, 0.5)
    s.synchronize()
    assert_same(on_s, ref, "side stream")
    out = torch.zeros(d.shape, dtype=torch.uint8, device=DEV)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _lib.call("ctd_speckle_filter_f32", d.data_ptr(), ok.data_ptr(), out.data_ptr(), 3, 200, 300, 30, 0.5,
                  torch.cuda.current_stream().cuda_stream)
    for _ in range(3):
        out.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert_same(out.bool(), ref, "graph replay")
    got3 = tx.speckle_filter(d[1], ok[1], 30, 0.5)
    assert_same(got3, ref[1], "[1,H,W] input")
    assert_same(tx.speckle_filter(d, None, 30, 0.5), tx.speckle_filter_pytorch(d, None, 30, 0.5), "valid=None")
    assert_same(tx.speckle_filter(d, ok, 0, 0.5), ok, "max_size = 0")


@pytest.mark.gpu
def test_errors_empty_and_null_output(tx):
    from connecting_the_dots_b200 import _lib
    d = torch.rand(2, 1, 16, 20, device=DEV)
    ok = torch.ones(d.shape, dtype=torch.bool, device=DEV)
    for bad, exc in (((d.transpose(2, 3),), RuntimeError), ((d[:, :, :, :1].expand(2, 1, 16, 20),), RuntimeError),
                     ((d.half(),), NotImplementedError), ((d, ok.cpu()), RuntimeError), ((d, ok[:1]), RuntimeError),
                     ((d, None, -3), RuntimeError), ((d, None, 3, -1.0), RuntimeError)):
        with pytest.raises(exc):
            tx.speckle_filter(*bad)
    st = torch.cuda.current_stream().cuda_stream
    u8 = ok.to(torch.uint8)
    with pytest.raises(_lib.CtdError, match="overlaps disp"):
        _lib.call("ctd_speckle_filter_f32", d.data_ptr(), None, d.data_ptr() + 7, 2, 16, 20, 3, 1.0, st)
    with pytest.raises(_lib.CtdError, match="overlaps valid"):
        _lib.call("ctd_speckle_filter_f32", d.data_ptr(), u8.data_ptr(), u8.data_ptr(), 2, 16, 20, 3, 1.0, st)
    before = _lib.launch_count()
    _lib.call("ctd_speckle_filter_f32", d.data_ptr(), u8.data_ptr(), None, 2, 16, 20, 3, 1.0, st)
    e = tx.speckle_filter(torch.rand(0, 1, 16, 20, device=DEV))
    assert e.shape == (0, 1, 16, 20) and e.dtype == torch.bool
    assert tx.speckle_filter(torch.rand(2, 1, 0, 20, device=DEV)).shape == (2, 1, 0, 20)
    assert _lib.launch_count() == before, "an empty batch or a null valid_out launches nothing"
    tx.speckle_filter(d)
    assert _lib.launch_count() == before + 4


@pytest.mark.gpu
def test_end_to_end_against_ground_truth(tx):
    """synth.make_batch(2), census 7x9, D = 128, ta against pat_lcn, integer disparities, interior rows and columns 9..-9.
    A CPU probe of the definition gave, kept fraction / fraction of kept pixels within 2 px of the ground truth:
    block 9 WTA, disparity_check(1, 0) then speckle (200, 1): 0.462 / 0.938; block 1 -> sgm (p1 6, p2 400, 8 paths), speckle
    (200, 1) alone: 0.878 / 0.902.  The kernels are bit-equal to the definition, so these reproduce."""
    a, b, d = bench_frames(2)
    gt = cu(d["disp"])
    inner = (slice(None), slice(None), slice(9, -9), slice(9, -9))
    cd, _, cok = tx.disparity_check(tx.census_vol(a, b, 128, (7, 9), 9), 1, 0.0, subpixel=False)
    sgm = tx.sgm_disparity(tx.census_vol(a, b, 128, (7, 9), 1), 6, 400, 8, subpixel=False)[0]
    res = {}
    for name, disp, ok in (("bm check+speckle", cd, cok), ("sgm speckle", sgm, None)):
        keep = tx.speckle_filter(disp, ok, 200, 1.0)
        assert_same(keep, tx.speckle_filter_pytorch(disp, ok, 200, 1.0), name)
        good = ((disp - gt).abs() <= 2)[inner]
        # the probe averages the two images' fractions
        res[name] = tuple(float(np.mean([float(f(i)) for i in range(2)])) for f in (
            lambda i: keep[inner][i].float().mean(), lambda i: good[i][keep[inner][i]].float().mean()))
    msg = "check+speckle kept %.3f acc %.3f (probe 0.462 / 0.938); sgm speckle kept %.3f acc %.3f (0.878 / 0.902)" % (
        res["bm check+speckle"] + res["sgm speckle"])
    print(msg)
    (k1, a1), (k2, a2) = res["bm check+speckle"], res["sgm speckle"]
    assert abs(k1 - 0.462) <= 0.005 and abs(a1 - 0.938) <= 0.005, msg
    assert abs(k2 - 0.878) <= 0.005 and abs(a2 - 0.902) <= 0.005, msg
