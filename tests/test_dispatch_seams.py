"""GPU tests of the loss-path kernels at their dispatch seams (-m gpu).

On every call the host code of the photometric loss, LCN, the masked sums, the pattern warp, the fused pattern
similarity, the disparity loss and the depth-similarity loss picks one of several kernels from the width modulo 4, the
16-byte alignment of each pointer, minimum image sizes, the batch size and the total pixel count.  The other GPU tests
use aligned allocations at moderate batch sizes; these tests call the default dispatcher with contiguous but unaligned
views, batches either side of the chunk sizes (32768 images for the photometric loss, 65535 for the warp and LCN),
per-image patterns, the persistent grid of the disparity loss, the automatic pair-symmetric census forward and NULL
gradient pointers, and compare every result with a high-precision reference.

Each test also records the kernels its calls launched (torch.profiler; CUPTI sees the ctypes library's launches too) and
asserts that it ran the branch it was written for, so that a change of the dispatcher cannot quietly turn it into a
duplicate of another test.  Where the profiler's trace misses launches, only that assertion is skipped.
"""
import json
import os
import re
import tempfile

import numpy as np
import pytest
import torch

import oracle
from conftest import assert_close
from losses_torch import depth_similarity as _ref_depth_similarity, disparity_loss as _ref_disparity_loss
from test_gpu_ops import _grad_close, _lcn_reference_recipe, _reference_pattern_loss

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TYPES = ("mse", "sad", "census_mse", "census_sad")
CTD_ERR_INVALID = 1  # include/ctd_b200.h
PAD, FILL = 4096, -777.0


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _lib():
    from connecting_the_dots_b200 import _lib
    return _lib


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _invalid(msg):
    """pytest.raises for a call that the C ABI refuses with CTD_ERR_INVALID and `msg`."""
    return pytest.raises(_lib().CtdError, match=r"failed \(%d\): .*%s" % (CTD_ERR_INVALID, msg))


# ---------------------------------------------------------------- helpers
def _offset_view(shape, k, dtype=torch.float32):
    """(raw, view): a contiguous tensor of `shape` whose data_ptr() is k elements past a 16-byte boundary, inside an
    allocation whose margins hold a sentinel (k = 0: aligned, still guarded)."""
    n = int(np.prod(shape))
    raw = torch.full((n + 2 * PAD + k,), FILL, dtype=dtype, device=DEV)
    view = raw[PAD + k:PAD + k + n].view(*shape)
    assert view.is_contiguous() and view.data_ptr() % 16 == (k * raw.element_size()) % 16
    return raw, view


def _placed(src, k):
    """_offset_view holding a copy of `src` (numpy array or tensor)."""
    t = src if torch.is_tensor(src) else torch.from_numpy(np.ascontiguousarray(src))
    raw, view = _offset_view(tuple(t.shape), k, t.dtype)
    view.copy_(t)
    return raw, view


def _margins_intact(raw, view):
    start = (view.data_ptr() - raw.data_ptr()) // raw.element_size()
    return bool((raw[:start] == FILL).all()) and bool((raw[start + view.numel():] == FILL).all())


def _kernels(fn):
    """Run fn() under the profiler.  Returns (fn's result, [(kernel name, grid)] in launch order), or an empty list when
    the trace holds fewer of the library's kernels than the library counted launches (ctd_launch_count): a trace that
    misses launches cannot show which branch ran."""
    L = _lib()
    torch.cuda.synchronize()
    n0 = L.launch_count()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU, torch.profiler.ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    launched = L.launch_count() - n0
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f).get("traceEvents", [])
    ks = sorted((e.get("ts", 0), e.get("name", ""), tuple(e.get("args", {}).get("grid", ())))
                for e in events if str(e.get("cat", "")).lower() == "kernel")
    ks = [(n, g) for _, n, g in ks]
    ours = sum("ctd::" in n for n, _ in ks)
    if ours < launched:
        print("the trace holds %d of the %d kernels the library launched" % (ours, launched))
        return res, []
    return res, ks


def _grids(ks, name):
    """Grids of the launches of kernel `name` (a whole identifier of the demangled name: photo_fwd_box9 does not match
    photo_fwd_box9_tma)."""
    pat = re.compile(r"(?<!\w)%s(?!\w)" % re.escape(name))
    return [g for n, g in ks if pat.search(n)]


def _seen(ks, what):
    if not ks:
        print("%s: no complete kernel trace from the profiler on this machine; kernel-choice assertion skipped" % what)
    return bool(ks)


def _expect(ks, ran, among, what):
    """Of the kernels `among`, exactly those in `ran` were launched."""
    if _seen(ks, what):
        got = {k for k in among if _grids(ks, k)}
        assert got == set(ran), "%s: ran %s, expected %s (all kernels: %s)" % (what, sorted(got), sorted(ran), sorted({n for n, _ in ks}))


def _expect_chunks(ks, name, B, chunk, what, zper=1):
    """`name` ran once per chunk of at most `chunk` images, gridDim.z = the chunk's images x zper."""
    if _seen(ks, what):
        z = [g[2] for g in _grids(ks, name) if len(g) == 3]
        want = [min(chunk, B - b0) * zper for b0 in range(0, B, chunk)]
        assert z == want, "%s: %s grid.z per launch %s, expected %s" % (what, name, z, want)


# ---------------------------------------------------------------- 1. photometric loss, unaligned pointers
ENTRY_ARGS = {  # pointer arguments of each C entry point that take part in its dispatch (sums2 stays aligned)
    "fwd": ("es", "ta", "out"),
    "bwd": ("es", "ta", "grad_out", "grad_in"),
    "fwd_bwd": ("es", "ta", "grad_out", "out", "grad_in"),
    "fwd_bwd_masked": ("es", "ta", "grad_out", "mask", "out", "grad_in"),
}
BOX_KERNELS = ("photo_fwd_box9", "photo_bwd_box9", "photo_fwd_box9_tma", "photo_bwd_box9_tma", "photo_fwd_bwd_box9_tma", "masked_sums_kernel")
CENSUS_KERNELS = ("photo_fwd_census9", "photo_bwd_census9", "census_sym_kernel", "census_fwd_pairs", "masked_sums_kernel")


def _photometric_call(entry, p, B, C, H, W, ty, eps):
    L, st = _lib(), _stream()
    if entry == "fwd":
        L.call("ctd_photometric_fwd_f32", p["es"], p["ta"], p["out"], B, C, H, W, 9, ty, eps, st)
    elif entry == "bwd":
        L.call("ctd_photometric_bwd_f32", p["es"], p["ta"], p["grad_out"], p["grad_in"], B, C, H, W, 9, ty, eps, st)
    elif entry == "fwd_bwd":
        L.call("ctd_photometric_fwd_bwd_f32", p["es"], p["ta"], p["grad_out"], p["out"], p["grad_in"], B, C, H, W, 9, ty, eps, st)
    else:
        L.call("ctd_photometric_fwd_bwd_masked_f32", p["es"], p["ta"], p["grad_out"], p["mask"], p["out"], p["grad_in"], p["sums2"],
               B, C, H, W, 9, ty, eps, st)


def _box_kernels(entry, off):
    """What the mse / sad dispatcher runs at C = 1, W % 4 = 0 when the pointers named in `off` are unaligned: the TMA
    kernels need every pointer they touch aligned (photometric_tma.cu), else the shared-memory tile kernels run."""
    al = lambda names: not set(names) & set(off)
    fwd = "photo_fwd_box9_tma" if al(("es", "ta", "out")) else "photo_fwd_box9"
    bwd = "photo_bwd_box9_tma" if al(("es", "ta", "grad_out", "grad_in")) else "photo_bwd_box9"
    if entry == "fwd":
        return [fwd]
    if entry == "bwd":
        return [bwd]
    if entry == "fwd_bwd_masked" and al(ENTRY_ARGS[entry]):
        return ["photo_fwd_bwd_box9_tma"]
    ks = ["photo_fwd_bwd_box9_tma"] if al(ENTRY_ARGS["fwd_bwd"]) else [fwd, bwd]
    return ks + (["masked_sums_kernel"] if entry == "fwd_bwd_masked" else [])


@pytest.mark.parametrize("shape", [(2, 1, 40, 132), (1, 1, 96, 160)])
@pytest.mark.parametrize("ty", range(4))
def test_photometric_unaligned_pointers(tx, shape, ty):
    """Every entry point with each pointer argument one element past a 16-byte boundary on its own, then all of them
    (and all aligned, the TMA / vector control): loss map, gradient and masked sums against the oracle, outputs written
    inside their views only.  photometric.cu vec_ok, photometric_tma.cu accept / reject tests."""
    B, C, H, W = shape
    rng = np.random.RandomState(ty * 100 + W)
    es = rng.randn(B, C, H, W).astype(np.float32)
    data = {"es": es, "ta": (es + 0.7 * rng.randn(B, C, H, W)).astype(np.float32),
            "grad_out": rng.randn(B, 1, H, W).astype(np.float32), "mask": rng.rand(B, 1, H, W).astype(np.float32)}
    ref_out = oracle.photometric_loss_forward(data["es"], data["ta"], 9, ty, 0.5)
    ref_gi = oracle.photometric_loss_backward(data["es"], data["ta"], data["grad_out"], 9, ty, 0.5)
    m64 = data["mask"].astype(np.float64)
    ref_sums = ((m64 * ref_out).sum(), m64.sum())
    out_shape = {"out": (B, 1, H, W), "grad_in": (B, C, H, W)}
    for entry, names in ENTRY_ARGS.items():
        for off in [()] + [(n,) for n in names] + [names]:
            what = "%s %s offset %s" % (TYPES[ty], entry, off or "none")
            raws, views = {}, {}
            for n in names:
                k = 1 if n in off else 0
                raws[n], views[n] = _placed(data[n], k) if n in data else _offset_view(out_shape[n], k)
            sums2 = torch.full((2,), float("nan"), device=DEV)
            p = {n: v.data_ptr() for n, v in views.items()}
            p["sums2"] = sums2.data_ptr()
            _, ks = _kernels(lambda: _photometric_call(entry, p, B, C, H, W, ty, 0.5))
            if ty <= 1:
                _expect(ks, _box_kernels(entry, off), BOX_KERNELS, what)
            else:
                _expect(ks, ["photo_fwd_census9" if entry == "fwd" else "photo_bwd_census9"], CENSUS_KERNELS, what)
            if "out" in views:
                assert_close(views["out"].cpu().numpy(), ref_out, what=what + ": loss map")
            if "grad_in" in views:
                assert_close(views["grad_in"].cpu().numpy(), ref_gi, what=what + ": gradient")
            if entry == "fwd_bwd_masked":
                got = sums2.cpu().numpy().astype(np.float64)
                assert all(abs(g - r) <= 1e-5 * abs(r) for g, r in zip(got, ref_sums)), (what, got, ref_sums)
            for n in names:
                assert _margins_intact(raws[n], views[n]), "%s: %s written outside its view" % (what, n)


@pytest.mark.parametrize("ty", range(4))
def test_photometric_unaligned_batch_slices(tx, ty):
    """The realistic way to get unaligned tensors: es[1:], ta[1:], go[1:] of a batch of 61x83 images (odd H*W: every
    slice starts 12 bytes past a 16-byte boundary), through photometric_loss and weighted_photometric_loss with
    autograd."""
    rng = np.random.RandomState(61 + ty)
    es = rng.randn(3, 1, 61, 83).astype(np.float32)
    ta = (es + 0.7 * rng.randn(3, 1, 61, 83)).astype(np.float32)
    go = rng.randn(3, 1, 61, 83).astype(np.float32)
    mask = rng.rand(3, 1, 61, 83).astype(np.float32)
    E, T, G, M = (cu(a)[1:] for a in (es, ta, go, mask))
    assert all(t.is_contiguous() and t.data_ptr() % 16 == 12 for t in (E, T, G, M))
    es, ta, go, mask = es[1:], ta[1:], go[1:], mask[1:]
    ref_out = oracle.photometric_loss_forward(es, ta, 9, ty, 0.5)
    e = E.detach().requires_grad_(True)
    assert e.data_ptr() == E.data_ptr()
    out = tx.photometric_loss(e, T, 9, TYPES[ty], 0.5)
    (g,) = torch.autograd.grad(out, e, G)
    assert_close(out.detach().cpu().numpy(), ref_out, what="photometric_loss")
    assert_close(g.cpu().numpy(), oracle.photometric_loss_backward(es, ta, go, 9, ty, 0.5), what="photometric_loss gradient")
    val, loss_map = tx.weighted_photometric_loss(e, T, M, 9, TYPES[ty], 0.5)
    (g,) = torch.autograd.grad(2.0 * val, e)
    m64 = mask.astype(np.float64)
    ref_val = (m64 * ref_out).sum() / m64.sum()
    assert abs(val.item() - ref_val) <= 1e-5 * abs(ref_val)
    assert_close(loss_map.cpu().numpy(), ref_out, what="weighted loss map")
    ref_g = oracle.photometric_loss_backward(es, ta, mask, 9, ty, 0.5) * (2.0 / m64.sum())
    assert_close(g.cpu().numpy(), ref_g, what="weighted loss gradient")


# ---------------------------------------------------------------- 2. photometric loss, batch chunks
@pytest.mark.parametrize("ty,C,W", [(0, 2, 13), (1, 1, 13), (2, 1, 12), (3, 2, 12)])
def test_photometric_batch_chunks(tx, ty, C, W):
    """32768 and 32769 images: the tile kernels loop over the batch in chunks of 32768 (photometric.cu fwd, bwd and
    fwd_bwd loops) and fwd_bwd_masked takes the separate-calls path above 32768.  Sizes keep the chunked kernels in
    play: W = 13 keeps the TMA kernels out, H = 9 the pair-symmetric census kernel.  Every image against the oracle;
    C = 2 makes a chunk offset that forgets the channel count visible."""
    H, N = 9, 32769
    rng = np.random.RandomState(ty)
    es = rng.randn(N, C, H, W).astype(np.float32)
    ta = (es + 0.7 * rng.randn(N, C, H, W)).astype(np.float32)
    go = rng.randn(N, 1, H, W).astype(np.float32)
    mask = rng.rand(N, 1, H, W).astype(np.float32)
    ref_out = oracle.photometric_loss_forward(es, ta, 9, ty, 0.5)
    ref_gi = oracle.photometric_loss_backward(es, ta, go, 9, ty, 0.5)
    E, T, G, M = cu(es), cu(ta), cu(go), cu(mask)
    fk, bk = ("photo_fwd_box9", "photo_bwd_box9") if ty <= 1 else ("photo_fwd_census9", "photo_bwd_census9")
    X = tx.ext_cuda

    def check(what, B, out=None, gi=None):
        if out is not None:
            out = out.cpu().numpy()
            assert_close(out, ref_out[:B], what=what + " loss map")
            assert_close(out[32766:], ref_out[32766:B], what=what + " loss map, images from 32766")
        if gi is not None:
            gi = gi.cpu().numpy()
            assert_close(gi, ref_gi[:B], what=what + " gradient")
            assert_close(gi[32766:], ref_gi[32766:B], what=what + " gradient, images from 32766")

    for B in (32768, 32769):
        e, t, g, m = E[:B], T[:B], G[:B], M[:B]
        out, ks = _kernels(lambda: X.photometric_loss_forward(e, t, 9, ty, 0.5))
        _expect_chunks(ks, fk, B, 32768, "fwd B=%d" % B)
        check("fwd B=%d" % B, B, out=out)
        gi, ks = _kernels(lambda: X.photometric_loss_backward(e, t, g, 9, ty, 0.5))
        _expect_chunks(ks, bk, B, 32768, "bwd B=%d" % B)
        check("bwd B=%d" % B, B, gi=gi)
        (out, gi), ks = _kernels(lambda: X.photometric_loss_forward_backward(e, t, g, 9, ty, 0.5))
        if ty <= 1:
            _expect_chunks(ks, fk, B, 32768, "fwd_bwd B=%d" % B)
        _expect_chunks(ks, bk, B, 32768, "fwd_bwd B=%d" % B)
        check("fwd_bwd B=%d" % B, B, out=out, gi=gi)
        (out, gi, sums), ks = _kernels(lambda: X.photometric_loss_forward_backward_masked(e, t, g, m, 9, ty, 0.5))
        # census: one fused kernel (loss, gradient, sums) up to 32768 images, above that the chunked fused calls and the
        # separate masked sums; mse / sad (no TMA here): forward, backward and masked sums as separate kernels
        separate = ty <= 1 or B > 32768
        if _seen(ks, "fwd_bwd_masked B=%d" % B):
            assert bool(_grids(ks, "masked_sums_kernel")) == separate, "fwd_bwd_masked B=%d" % B
        _expect_chunks(ks, bk, B, 32768, "fwd_bwd_masked B=%d" % B)
        check("fwd_bwd_masked B=%d" % B, B, out=out, gi=gi)
        m64 = mask[:B].astype(np.float64)
        ref_sums = ((m64 * ref_out[:B]).sum(), m64.sum())
        got = sums.cpu().numpy().astype(np.float64)
        assert all(abs(a - r) <= 1e-5 * abs(r) for a, r in zip(got, ref_sums)), (B, got, ref_sums)


# ---------------------------------------------------------------- 3. LCN
def _lcn_forward_kernel(N, H, W):
    """lcn.cu lcn_impl at radius 5 with aligned pointers."""
    if W % 4 == 0 and H >= 32 and W >= 32:
        return "lcn_tma_kernel"
    return "lcn_generic_kernel" if N > 65535 else "lcn_strip_kernel"


@pytest.mark.parametrize("H,W", [(12, 13), (32, 32)])
def test_lcn_batch_chunks(tx, H, W):
    """65535 and 65537 images: above 65535 the forward takes lcn_generic_kernel unless the TMA kernel applies (12x13:
    W % 4 != 0 and H < 32; 32x32: TMA), and the backward loops its box kernel over chunks of 65535 images (it used to
    refuse them).  Forward against the oracle, backward against float64 autograd through the reference recipe, with
    both upstream gradients and with each one absent (NULL)."""
    N, r, eps = 65537, 5, 0.05
    g = torch.Generator(device="cpu").manual_seed(H * W)
    x = torch.rand(N, 1, H, W, generator=g)
    gl, gs = torch.randn(N, 1, H, W, generator=g), torch.randn(N, 1, H, W, generator=g)
    lo, so = oracle.lcn(x.numpy(), r, eps)
    X, GL, GS = x.to(DEV), gl.to(DEV), gs.to(DEV)
    xd = X.double().requires_grad_(True)
    l64, s64 = _lcn_reference_recipe(xd, r, eps)
    (ref_l,) = torch.autograd.grad(l64, xd, GL.double(), retain_graph=True)
    (ref_s,) = torch.autograd.grad(s64, xd, GS.double())
    ref_l, ref_s = ref_l.cpu().numpy(), ref_s.cpu().numpy()
    del xd, l64, s64
    for n in (65535, 65537):
        xn = X[:n].detach().requires_grad_(True)
        (l, s), ks = _kernels(lambda: tx.lcn(xn, r, eps))
        k = _lcn_forward_kernel(n, H, W)
        _expect(ks, [k], ("lcn_tma_kernel", "lcn_generic_kernel", "lcn_strip_kernel"), "lcn N=%d" % n)
        assert_close(l.detach().cpu().numpy(), lo[:n], what="lcn N=%d" % n)
        assert_close(s.detach().cpu().numpy(), so[:n], what="std N=%d" % n)
        (gx,), ks = _kernels(lambda: torch.autograd.grad((l * GL[:n]).sum() + (s * GS[:n]).sum(), xn))
        _expect_chunks(ks, "lcn_bwd_box_kernel", n, 65535, "lcn backward N=%d" % n)
        assert_close(gx.cpu().numpy(), (ref_l + ref_s)[:n], tol=2e-5, what="lcn backward N=%d" % n)
        l, s = l.detach(), s.detach()
        for gln, gsn, ref, what in ((GL[:n], None, ref_l, "grad_std NULL"), (None, GS[:n], ref_s, "grad_lcn NULL")):
            gx = tx.ext_cuda.lcn_backward(X[:n], l, s, gln, gsn, r, eps)
            assert_close(gx.cpu().numpy(), ref[:n], tol=2e-5, what="lcn backward N=%d, %s" % (n, what))


def test_lcn_unaligned_pointers(tx):
    """ctd_lcn_f32 and ctd_lcn_bwd_f32 with each pointer one to three elements past a 16-byte boundary, then all of
    them: the TMA kernel needs aligned x, lcn and std, else the strip kernel runs without its vector path (lcn.cu
    lcn_tma_launch, vec).  Results against the oracle and float64 autograd; outputs written inside their views only.
    Radius 9 is beyond the backward's limit (8) and is refused."""
    N, H, W, r, eps = 3, 40, 64, 5, 0.05
    L, st = _lib(), _stream()
    g = torch.Generator(device="cpu").manual_seed(7)
    x = torch.rand(N, 1, H, W, generator=g)
    gl, gs = torch.randn(N, 1, H, W, generator=g), torch.randn(N, 1, H, W, generator=g)
    lo, so = oracle.lcn(x.numpy(), r, eps)
    xd = x.double().requires_grad_(True)
    l64, s64 = _lcn_reference_recipe(xd, r, eps)
    (ref,) = torch.autograd.grad((l64 * gl.double()).sum() + (s64 * gs.double()).sum(), xd)
    names = ("x", "lcn", "std")
    for off in [()] + [(n,) for n in names] + [names]:
        what = "lcn offset %s" % ((off or "none"),)
        k = {n: (1 + i if n in off else 0) for i, n in enumerate(names)}
        (rx, vx), (rl, vl), (rs, vs) = _placed(x, k["x"]), _offset_view(x.shape, k["lcn"]), _offset_view(x.shape, k["std"])
        _, ks = _kernels(lambda: L.call("ctd_lcn_f32", vx.data_ptr(), vl.data_ptr(), vs.data_ptr(), N, H, W, r, eps, st))
        _expect(ks, ["lcn_strip_kernel" if off else "lcn_tma_kernel"], ("lcn_tma_kernel", "lcn_strip_kernel", "lcn_generic_kernel"), what)
        assert_close(vl.cpu().numpy(), lo, what=what)
        assert_close(vs.cpu().numpy(), so, what=what)
        assert _margins_intact(rx, vx) and _margins_intact(rl, vl) and _margins_intact(rs, vs), what
    l, s = tx.ext_cuda.lcn_forward(cu(x), r, eps)
    bnames = ("x", "lcn", "std", "grad_lcn", "grad_std", "grad_x")
    src = {"x": x, "lcn": l, "std": s, "grad_lcn": gl, "grad_std": gs}
    for off in [(n,) for n in bnames] + [bnames]:
        what = "lcn_bwd offset %s" % (off,)
        placed = {n: (_placed(src[n], 1 + i % 3 if n in off else 0) if n in src else _offset_view(x.shape, 1 + i % 3 if n in off else 0))
                  for i, n in enumerate(bnames)}
        p = {n: v.data_ptr() for n, (_, v) in placed.items()}
        L.call("ctd_lcn_bwd_f32", p["x"], p["lcn"], p["std"], p["grad_lcn"], p["grad_std"], p["grad_x"], N, H, W, r, eps, st)
        assert_close(placed["grad_x"][1].cpu().numpy(), ref.numpy(), tol=2e-5, what=what)
        assert all(_margins_intact(*rv) for rv in placed.values()), what
    with _invalid("radius 9 out of range"):
        tx.ext_cuda.lcn_backward(cu(x), l, s, cu(gl), None, 9, eps)


# ---------------------------------------------------------------- 4. warp and pattern similarity with per-image patterns
def test_warp_per_image_patterns(tx):
    """pattern [B,1,Hp,Wp] (Bp = B, warp.cu warp_fwd_kernel / warp_bwd_kernel): three distinct patterns of another size
    than the image against torch's CUDA grid_sample and its autograd; swapping two images' patterns (same disparity and
    upstream gradient for both) swaps their outputs bit for bit."""
    B, H, W, Hp, Wp = 3, 40, 70, 52, 90
    g = torch.Generator(device="cpu").manual_seed(11)
    pattern = torch.randn(B, 1, Hp, Wp, generator=g).to(DEV)
    disp = torch.rand(B, 1, H, W, generator=g) * (W * 0.4) - 4   # some samples leave the pattern
    go = torch.randn(B, 1, H, W, generator=g)
    disp[1], go[1] = disp[0], go[0]
    disp, go = disp.to(DEV).requires_grad_(True), go.to(DEV)
    ones = torch.ones(B, 1, H, W, device=DEV)
    _, proj_ref = _reference_pattern_loss(disp, pattern, ones, ones, "sad", 0.5, tx)
    (gref,) = torch.autograd.grad(proj_ref, disp, go)
    proj, ks = _kernels(lambda: tx.warp_pattern(pattern, disp))
    (gd,) = torch.autograd.grad(proj, disp, go)
    _expect_chunks(ks, "warp_fwd_kernel", B, 65535, "warp forward")
    assert_close(proj.detach().cpu().numpy(), proj_ref.detach().cpu().numpy(), what="warp forward")
    assert_close(gd.cpu().numpy(), gref.cpu().numpy(), what="warp backward")
    assert not torch.equal(proj[0], proj[1])
    swapped = pattern[[1, 0, 2]].contiguous()
    d = disp.detach()
    p2 = tx.ext_cuda.warp_pattern_forward(swapped, d)
    g2 = tx.ext_cuda.warp_pattern_backward(swapped, d, go)
    for a, b in ((0, 1), (1, 0), (2, 2)):
        assert torch.equal(p2[a], proj[b].detach()) and torch.equal(g2[a], gd[b]), (a, b)


@pytest.mark.parametrize("Bp", (1, 65536))
def test_warp_batch_chunks(tx, Bp):
    """65536 tiny images: the warp loops over chunks of 65535 images and moves the pattern pointer with each chunk when
    Bp = B (warp.cu).  Forward and backward against grid_sample."""
    B, H, W, Hp, Wp = 65536, 4, 5, 6, 7
    g = torch.Generator(device="cpu").manual_seed(Bp)
    pattern = torch.randn(Bp, 1, Hp, Wp, generator=g).to(DEV)
    disp = (torch.rand(B, 1, H, W, generator=g) * 3 - 1).to(DEV).requires_grad_(True)
    go = torch.randn(B, 1, H, W, generator=g).to(DEV)
    ones = torch.ones(B, 1, H, W, device=DEV)
    _, proj_ref = _reference_pattern_loss(disp, pattern, ones, ones, "sad", 0.5, tx)
    (gref,) = torch.autograd.grad(proj_ref, disp, go)
    proj, ks = _kernels(lambda: tx.warp_pattern(pattern, disp))
    _expect_chunks(ks, "warp_fwd_kernel", B, 65535, "warp forward")
    (gd,), ks = _kernels(lambda: torch.autograd.grad(proj, disp, go))
    _expect_chunks(ks, "warp_bwd_kernel", B, 65535, "warp backward")
    for a, b, what in ((proj.detach(), proj_ref.detach(), "warp forward"), (gd, gref, "warp backward")):
        a, b = a.cpu().numpy(), b.cpu().numpy()
        assert_close(a, b, what=what)
        assert_close(a[65534:], b[65534:], what=what + ", images from 65534")


@pytest.mark.parametrize("loss_type", ("census_sad", "census_mse"))
def test_pattern_similarity_per_image_patterns(tx, loss_type):
    """pattern_similarity_loss(fused=True) with Bp = B (photometric.cu fused tile loader) against the three-kernel
    composition (same bounds as the one-pattern test: pattern_proj bit for bit, value and gradient 1e-6) and against
    the reference recipe with grid_sample and the oracle (1e-5)."""
    B, H, W, Hp, Wp = 3, 60, 83, 72, 100
    g = torch.Generator(device="cpu").manual_seed(5)
    pattern = torch.randn(B, 1, Hp, Wp, generator=g).to(DEV)
    disp = (torch.rand(B, 1, H, W, generator=g) * (W * 0.3) - 6).to(DEV)
    im = torch.randn(B, 1, H, W, generator=g).to(DEV)
    std = (torch.rand(B, 1, H, W, generator=g) + 0.1).to(DEV)
    dr = disp.clone().requires_grad_(True)
    ref, proj_ref = _reference_pattern_loss(dr, pattern, im, std, loss_type, 0.5, tx)
    (gref,) = torch.autograd.grad(ref, dr)
    res = []
    for fused in (True, False):
        d = disp.clone().requires_grad_(True)
        (val, proj), ks = _kernels(lambda: tx.pattern_similarity_loss(d, pattern, im, std, loss_type, 0.5, fused=fused))
        _expect(ks, ["photo_bwd_census9"] + ([] if fused else ["warp_fwd_kernel"]), ("photo_bwd_census9", "warp_fwd_kernel"),
                "fused=%s" % fused)
        (gd,) = torch.autograd.grad(val, d)
        res.append((val.detach(), proj.detach(), gd))
        assert abs(val.item() - ref.item()) <= 1e-5 * abs(ref.item()), (fused, val.item(), ref.item())
        assert_close(proj.detach().cpu().numpy(), proj_ref.detach().cpu().numpy(), what="pattern_proj fused=%s" % fused)
        assert_close(gd.cpu().numpy(), gref.cpu().numpy(), what="d loss / d disp fused=%s" % fused)
    assert torch.equal(res[0][1], res[1][1]), "pattern_proj differs"
    assert abs(res[0][0].item() - res[1][0].item()) <= 1e-6 * abs(res[1][0].item())
    assert_close(res[0][2].cpu().numpy(), res[1][2].cpu().numpy(), tol=1e-6, what="d loss / d disp, fused vs three kernels")


def test_pattern_similarity_batch_limit(tx):
    """The fused kernel takes B <= 32768 (photometric.cu ctd_pattern_similarity_f32): 32768 images of 9x9 give the
    three-kernel composition's results, 32769 are refused with CTD_ERR_INVALID."""
    g = torch.Generator(device="cpu").manual_seed(9)
    pattern = torch.randn(1, 1, 12, 12, generator=g).to(DEV)
    for B in (32768, 32769):
        disp = (torch.rand(B, 1, 9, 9, generator=g) * 3).to(DEV)
        im = torch.randn(B, 1, 9, 9, generator=g).to(DEV)
        mask = (torch.rand(B, 1, 9, 9, generator=g) + 0.1).to(DEV)
        if B > 32768:
            with _invalid("size out of range"):
                tx.ext_cuda.pattern_similarity(pattern, disp, im, mask, mask, 3, 0.5)
            continue
        proj, out, gd, sums = tx.ext_cuda.pattern_similarity(pattern, disp, im, mask, mask, 3, 0.5)
        proj3 = tx.ext_cuda.warp_pattern_forward(pattern, disp)
        out3, gi3, sums3 = tx.ext_cuda.photometric_loss_forward_backward_masked(proj3, im, mask, mask, 9, 3, 0.5)
        gd3 = tx.ext_cuda.warp_pattern_backward(pattern, disp, gi3)
        assert torch.equal(proj, proj3)
        assert_close(out.cpu().numpy(), out3.cpu().numpy(), tol=1e-6, what="loss map")
        assert_close(gd.cpu().numpy(), gd3.cpu().numpy(), tol=1e-6, what="d loss / d disp")
        assert_close(sums.cpu().numpy(), sums3.cpu().numpy(), tol=1e-6, what="sums")


# ---------------------------------------------------------------- 5. disparity loss, persistent grid
def _disparity_inputs(B, H, W, seed):
    from connecting_the_dots_b200 import synth
    base = np.stack([synth.smooth_disparity(np.random.RandomState(seed + n % 64), H, W) for n in range(B)])[:, None]
    base = (base / 8.0 if H < 100 else base).astype(np.float32)
    edge = (1.0 / (1.0 + np.exp(-np.random.RandomState(seed).randn(B, 1, H, W) * 2))).astype(np.float32)
    return base, edge


@pytest.mark.parametrize("B,H,W", [(14, 480, 640), (5000, 20, 20)])
def test_disparity_loss_persistent_grid(tx, B, H, W):
    """More than MS_MAXBLK = 4096 tiles of 32x32 (14 x 300 and 5000 x 1): the kernel walks the tile list with 888
    persistent CTAs (disparity_loss.cu).  Value and both gradients against the torch restatement, with and without
    edge."""
    torch.backends.cudnn.allow_tf32 = False  # the restatement's two convolutions in fp32, not TF32
    base, edge = _disparity_inputs(B, H, W, 70)
    assert B * -(-H // 32) * -(-W // 32) > 4096
    for use_edge in (True, False):
        a, b = cu(base).requires_grad_(True), cu(base).requires_grad_(True)
        ea = cu(edge).requires_grad_(True) if use_edge else None
        eb = cu(edge).requires_grad_(True) if use_edge else None
        val, ks = _kernels(lambda: tx.disparity_loss(a, ea))
        if _seen(ks, "disparity_loss"):
            assert [g[0] for g in _grids(ks, "disparity_loss_kernel")] == [888], ks
        ref = _ref_disparity_loss(b, eb)
        (2.5 * val).backward()
        (2.5 * ref).backward()
        assert abs(float(val.detach()) - float(ref.detach())) <= 1e-5 * abs(float(ref.detach())), (float(val), float(ref))
        assert_close(a.grad.cpu().numpy(), b.grad.cpu().numpy(), tol=2e-5, what="grad disp edge=%s" % use_edge)
        if use_edge:
            assert_close(ea.grad.cpu().numpy(), eb.grad.cpu().numpy(), tol=2e-5, what="grad edge")


def test_disparity_loss_null_gradients(tx):
    """ctd_disparity_loss_f32 with grad_disp and / or grad_edge NULL, on the persistent grid (14 x 480x640): sums2 and
    every gradient still written are bit-equal to the full call's."""
    B, H, W = 14, 480, 640
    base, edge = _disparity_inputs(B, H, W, 80)
    disp, e = cu(base), cu(edge)
    L, st, scale = _lib(), _stream(), 1.0 / (B * H * W)

    def run(edge_on, gd_on, ge_on):
        sums = torch.full((2,), float("nan"), device=DEV)
        gd = torch.full_like(disp, float("nan")) if gd_on else None
        ge = torch.full_like(disp, float("nan")) if ge_on else None
        L.call("ctd_disparity_loss_f32", disp.data_ptr(), e.data_ptr() if edge_on else None, gd.data_ptr() if gd_on else None,
               ge.data_ptr() if ge_on else None, sums.data_ptr(), B, H, W, scale, st)
        return sums, gd, ge

    for edge_on in (True, False):
        sums, gd, ge = run(edge_on, True, edge_on)
        assert torch.isfinite(gd).all() and (ge is None or torch.isfinite(ge).all()) and torch.isfinite(sums).all()
        cases = ((False, True), (True, False), (False, False)) if edge_on else ((False, False),)
        for gd_on, ge_on in cases:
            s2, gd2, ge2 = run(edge_on, gd_on, ge_on)
            what = "edge=%s grad_disp=%s grad_edge=%s" % (edge_on, gd_on, ge_on)
            assert torch.equal(s2, sums), what
            assert gd2 is None or torch.equal(gd2, gd), what
            assert ge2 is None or torch.equal(ge2, ge), what
    with _invalid("grad_edge without edge"):
        L.call("ctd_disparity_loss_f32", disp.data_ptr(), None, disp.data_ptr(), disp.data_ptr(), cu(np.zeros(2, np.float32)).data_ptr(),
               B, H, W, scale, st)


# ---------------------------------------------------------------- 6. depth similarity
def _depth_args(d):
    return [cu(d[k]) for k in ("R0", "t0", "R1", "t1", "K")]


def test_depth_similarity_null_gradients(tx):
    """ctd_depth_similarity_f32 with grad_depthA and / or grad_depthB NULL (geometric.cu gA_img / gB_img): sums2 bit-equal
    to the full call, grad_depthA (plain stores) bit-equal, grad_depthB (atomics) within 1e-6."""
    from connecting_the_dots_b200 import synth
    B, H, W = 3, 48, 64
    d = synth.make_depth_pairs(B, H, W, seed=11)
    ray = tx.projection_rays(d["Ki"], H, W).to(DEV)
    d0, d1 = cu(d["depth0"]), cu(d["depth1"])
    R0, t0, R1, t1, K = _depth_args(d)
    L, st, scale = _lib(), _stream(), 1.0 / (B * H * W)

    def run(ga_on, gb_on):
        sums = torch.full((2,), float("nan"), device=DEV)
        ga = torch.full_like(d0, float("nan")) if ga_on else None
        gb = torch.zeros_like(d0) if gb_on else None
        L.call("ctd_depth_similarity_f32", d0.data_ptr(), d1.data_ptr(), ray.data_ptr(), K.data_ptr(), R0.data_ptr(), t0.data_ptr(),
               R1.data_ptr(), t1.data_ptr(), ga.data_ptr() if ga_on else None, gb.data_ptr() if gb_on else None, sums.data_ptr(),
               B, H, W, 0.1, scale, 0, st)
        return sums, ga, gb

    sums, ga, gb = run(True, True)
    assert torch.isfinite(ga).all() and torch.isfinite(sums).all() and float(gb.abs().max()) > 0
    for ga_on, gb_on in ((False, True), (True, False), (False, False)):
        s2, ga2, gb2 = run(ga_on, gb_on)
        what = "grad_depthA=%s grad_depthB=%s" % (ga_on, gb_on)
        assert torch.equal(s2, sums), what
        assert ga2 is None or torch.equal(ga2, ga), what
        if gb2 is not None:
            assert_close(gb2.cpu().numpy(), gb.cpu().numpy(), tol=1e-6, what=what)


def test_depth_similarity_batch_limit(tx):
    """One block per image at most MS_MAXBLK = 4096 blocks (geometric.cu): B = 4096 at 8x8 against the torch
    restatement, B = 4097 refused with CTD_ERR_INVALID."""
    from connecting_the_dots_b200 import synth
    torch.backends.cuda.matmul.allow_tf32 = False
    H, W = 8, 8
    d = synth.make_depth_pairs(4097, H, W, seed=12)
    ray = tx.projection_rays(d["Ki"], H, W).to(DEV)
    full = {k: cu(d[k]) for k in ("depth0", "depth1", "R0", "t0", "R1", "t1")}
    K = cu(d["K"])
    sl = lambda B: [full[k][:B] for k in ("R0", "t0", "R1", "t1")]
    B = 4096
    a0, a1 = full["depth0"][:B].clone().requires_grad_(True), full["depth1"][:B].clone().requires_grad_(True)
    b0, b1 = full["depth0"][:B].clone().requires_grad_(True), full["depth1"][:B].clone().requires_grad_(True)
    val, ks = _kernels(lambda: tx.projection_depth_similarity_loss(a0, a1, *sl(B), K, ray, 0.1))
    if _seen(ks, "depth_similarity B=4096"):
        assert [g[:2] for g in _grids(ks, "depth_similarity_kernel")] == [(1, 4096)] * 2, ks
    ref = _ref_depth_similarity(b0, b1, *sl(B), K, ray, 0.1)
    (3.0 * val).backward()
    (3.0 * ref).backward()
    assert abs(float(val) - float(ref)) <= 1e-5 * abs(float(ref)), (float(val), float(ref))
    _grad_close(a0.grad.cpu().numpy(), b0.grad.cpu().numpy(), "grad depth0")
    _grad_close(a1.grad.cpu().numpy(), b1.grad.cpu().numpy(), "grad depth1")
    with _invalid("batch too large for the reduction workspace"):
        tx.projection_depth_similarity_loss(full["depth0"], full["depth1"], *sl(4097), K, ray, 0.1)


# ---------------------------------------------------------------- 7. automatic pair-symmetric census forward
@pytest.mark.parametrize("ty", (2, 3))
def test_census_forward_automatic_pair_symmetric_dispatch(tx, ty):
    """The default dispatcher runs census_sym_kernel for forward-only calls from CS_MIN_PIXELS = 1.8 M pixels on
    (census_sym.cu): batch 6 at 480x640 (1.84 M) takes it, batch 5 (1.54 M) the gather kernel.  Both against the
    oracle."""
    rng = np.random.RandomState(ty)
    es = rng.randn(6, 1, 480, 640).astype(np.float32)
    ta = (es + 0.7 * rng.randn(6, 1, 480, 640)).astype(np.float32)
    ref = oracle.photometric_loss_forward(es, ta, 9, ty, 0.5)
    E, T = cu(es), cu(ta)
    for B in (6, 5):
        out, ks = _kernels(lambda: tx.photometric_loss(E[:B], T[:B], 9, TYPES[ty], 0.5))
        _expect(ks, ["census_sym_kernel" if B == 6 else "photo_fwd_census9"], CENSUS_KERNELS, "%s B=%d" % (TYPES[ty], B))
        assert_close(out.cpu().numpy(), ref[:B], what="%s B=%d" % (TYPES[ty], B))


# ---------------------------------------------------------------- 8. masked sums
@pytest.mark.parametrize("n", (1, 7, 2457600, 2457601, 2457602, 2457603))
def test_masked_sums_unaligned(tx, n):
    """masked_mean_terms with diff and / or mask unaligned (reduce.cu: the float4 path needs both aligned): float64 sums
    within 2e-6, run-to-run identical."""
    rng = np.random.RandomState(n % 1000)
    d = rng.rand(n).astype(np.float32)
    m = rng.rand(n).astype(np.float32)
    want = np.array([(m.astype(np.float64) * d).sum(), m.astype(np.float64).sum()])
    for kd, km in ((1, 0), (0, 2), (3, 3), (1, 2)):
        (rd, vd), (rm, vm) = _placed(d, kd), _placed(m, km)
        a, ks = _kernels(lambda: tx.masked_mean_terms(vd, vm))
        _expect(ks, ["masked_sums_kernel"], ("masked_sums_kernel",), "masked sums n=%d" % n)
        b = tx.masked_mean_terms(vd, vm)
        assert torch.equal(a, b), (n, kd, km)
        assert np.abs(a.cpu().numpy() - want).max() <= 2e-6 * want.max(), (n, kd, km, a.cpu().numpy(), want)
        assert _margins_intact(rd, vd) and _margins_intact(rm, vm)
