"""Correlation soft-argmax disparity (corr_softargmax.cu: ctd_corr_softargmax_fwd_* / _bwd_*, torchext.corr_softargmax /
corr_softargmax_pytorch / CorrSoftArgmax).

The definition is corr_softargmax_pytorch: the CPU tests pin it to a per-pixel numpy loop of the definition in fp64 and its
autograd gradients to finite differences.  The GPU tests hold the kernels to the restatement evaluated in fp64: the fp64
kernels to ~1e-10, the fp32 kernels to 1e-5 (forward) and 1e-4 (gradients) of the largest reference value.

Why 1e-4 for fp32 gradients: a gradient entry is a sum over up to D disparities of a_d times a feature, and a_d carries
the fp32 error of the recomputed score (a C-term dot product, relative error ~ sqrt(C) * 2^-24 of the score magnitude,
times |s|/tau in the exponent) and of the saved lse.  With |s|/tau of a few units that is ~1e-6 relative per term; summed
over D = 128 terms of mixed sign it stays well below 1e-4 of the largest entry.
"""
import re
import subprocess

import numpy as np
import pytest
import torch

from conftest import assert_close

DEV = "cuda:0"


def _F():
    from connecting_the_dots_b200.torchext import functions
    return functions


def corr_loop(f0, f1, D, tau):
    """The definition one pixel at a time in numpy fp64: (disp, lse), [B,1,H,W]."""
    f0, f1 = np.asarray(f0, np.float64), np.asarray(f1, np.float64)
    B, C, H, W = f0.shape
    disp, lse = np.zeros((B, 1, H, W)), np.zeros((B, 1, H, W))
    for b in range(B):
        for h in range(H):
            for w in range(W):
                s = np.array([np.dot(f0[b, :, h, w], f1[b, :, h, w - d]) / C for d in range(min(D, w + 1))])
                v = s / tau
                m = v.max()
                lse[b, 0, h, w] = m + np.log(np.exp(v - m).sum())
                p = np.exp(v - lse[b, 0, h, w])
                disp[b, 0, h, w] = (np.arange(len(p)) * p).sum()
    return disp, lse


def lse_pytorch(f0, f1, D, tau):
    """lse of the definition in plain torch, fp64, [B,1,H,W]."""
    a, b = f0.double(), f1.double()
    B, C, H, W = a.shape
    cols = [torch.nn.functional.pad((a[..., d:] * b[..., :W - d]).sum(1) / C, (d, 0), value=float("-inf"))
            for d in range(min(D, W))]
    return torch.logsumexp(torch.stack(cols, 1) / tau, 1, keepdim=True)


CPU_CASES = (  # B, C, H, W, D
    (1, 1, 1, 1, 1), (2, 3, 2, 1, 4), (1, 8, 2, 5, 9), (2, 1, 3, 7, 1), (1, 3, 2, 12, 5), (1, 8, 1, 20, 20), (2, 3, 2, 9, 3))


def test_restatement_matches_loop():
    F = _F()
    rng = np.random.RandomState(0)
    for (B, C, H, W, D) in CPU_CASES:
        for tau in (0.05, 1.0, 20.0):
            for scale in (1.0, 1e3):
                f0, f1 = rng.randn(B, C, H, W) * scale, rng.randn(B, C, H, W) * scale
                ref, ref_lse = corr_loop(f0, f1, D, tau)
                got = F.corr_softargmax_pytorch(torch.from_numpy(f0), torch.from_numpy(f1), D, tau)
                msg = "B%d C%d H%d W%d D%d tau %g scale %g" % (B, C, H, W, D, tau, scale)
                assert got.shape == (B, 1, H, W) and got.dtype == torch.float64, msg
                assert np.isfinite(got.numpy()).all(), msg
                np.testing.assert_allclose(got.numpy(), ref, rtol=1e-12, atol=1e-10, err_msg=msg)
                np.testing.assert_allclose(lse_pytorch(torch.from_numpy(f0), torch.from_numpy(f1), D, tau).numpy(), ref_lse,
                                           rtol=1e-12, err_msg=msg)
                assert (got[..., 0] == 0).all(), msg   # w = 0 has only d = 0
    f0 = torch.randn(3, 4, 6, dtype=torch.float64)
    f1 = torch.randn(3, 4, 6, dtype=torch.float64)
    assert torch.equal(F.corr_softargmax_pytorch(f0, f1, 5, 0.5), F.corr_softargmax_pytorch(f0[None], f1[None], 5, 0.5)[0])
    assert F.corr_softargmax_pytorch(f0[:, :0], f1[:, :0], 5).shape == (1, 0, 6)


def test_restatement_gradcheck():
    F = _F()
    torch.manual_seed(1)
    for (B, C, H, W, D), tau in (((1, 3, 2, 7, 4), 0.5), ((2, 2, 1, 9, 12), 1.0), ((1, 1, 2, 5, 1), 2.0)):
        f0 = torch.randn(B, C, H, W, dtype=torch.float64, requires_grad=True)
        f1 = torch.randn(B, C, H, W, dtype=torch.float64, requires_grad=True)
        assert torch.autograd.gradcheck(lambda a, b: F.corr_softargmax_pytorch(a, b, D, tau), (f0, f1))


def test_corr_softargmax_api_without_gpu(tx):
    from connecting_the_dots_b200 import _lib
    F = _F()
    f = torch.rand(2, 3, 5, 6)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        tx.corr_softargmax(f, f, 4)
    for bad, exc, msg in (((f, torch.rand(2, 3, 5, 7), 4), RuntimeError, "same shape"),
                          ((f, f.double(), 4), RuntimeError, "same shape and dtype"),
                          ((torch.rand(5, 6), torch.rand(5, 6), 4), RuntimeError, "C x H x W"),
                          ((f.half(), f.half(), 4), NotImplementedError, "not implemented"),
                          ((f, f, 0), RuntimeError, "n_disps"),
                          ((f, f, 2.5), RuntimeError, "n_disps"),
                          ((f[:, :0], f[:, :0], 4), RuntimeError, "C >= 1"),
                          ((f, f, 4, 0.0), RuntimeError, "temperature"),
                          ((f, f, 4, -1.0), RuntimeError, "temperature"),
                          ((f, f, 4, float("nan")), RuntimeError, "temperature"),
                          ((f, f, 4, float("inf")), RuntimeError, "temperature")):
        with pytest.raises(exc, match=msg):
            F.corr_softargmax_pytorch(*bad)
    # the C ABI checks its arguments before any device work (pointers here are never dereferenced)
    A, Bp, O, L, G = 1 << 30, 1 << 32, 1 << 34, 1 << 35, 1 << 36
    nf, nm = 2 * 3 * 5 * 6, 2 * 5 * 6
    fw32 = lambda *a: _lib.call("ctd_corr_softargmax_fwd_f32", *a)  # noqa: E731
    fw64 = lambda *a: _lib.call("ctd_corr_softargmax_fwd_f64", *a)  # noqa: E731
    bw32 = lambda *a: _lib.call("ctd_corr_softargmax_bwd_f32", *a)  # noqa: E731
    bw64 = lambda *a: _lib.call("ctd_corr_softargmax_bwd_f64", *a)  # noqa: E731
    dims = (2, 3, 5, 6, 4)
    for fn, args, msg in ((fw32, (A, Bp, O, L, -2, 3, 5, 6, 4, 1.0, None), "negative size"),
                          (fw64, (A, Bp, O, L, 2, 3, 5, 6, -4, 1.0, None), "negative size"),
                          (bw32, (A, Bp, O, L, G, A + (1 << 38), None, 2, 3, -5, 6, 4, 1.0, None), "negative size"),
                          (fw32, (A, Bp, O, L, 2, 0, 5, 6, 4, 1.0, None), "C must be"),
                          (fw32, (A, Bp, O, L, 2, 3, 5, 6, 0, 1.0, None), "n_disps"),
                          (bw64, (A, Bp, O, L, G, 1 << 38, None, 2, 3, 5, 6, 0, 1.0, None), "n_disps"),
                          (fw32, (A, Bp, O, L) + dims + (0.0, None), "temperature"),
                          (fw64, (A, Bp, O, L) + dims + (-1.0, None), "temperature"),
                          (fw32, (A, Bp, O, L) + dims + (float("nan"), None), "temperature"),
                          (bw32, (A, Bp, O, L, G, 1 << 38, None) + dims + (float("inf"), None), "temperature"),
                          (fw32, (A, Bp, O, L, 1, 1, 1, 1 << 30, 4, 1.0, None), "int32"),
                          (fw32, (None, Bp, O, L) + dims + (1.0, None), "null pointer"),
                          (fw32, (A, Bp, O, None) + dims + (1.0, None), "null pointer"),
                          (bw32, (A, Bp, O, L, None, 1 << 38, None) + dims + (1.0, None), "null pointer"),
                          (fw32, (A, Bp, A + 4 * nf - 4, L) + dims + (1.0, None), "disp overlaps an input"),
                          (fw64, (A, Bp, O, Bp - 8 * nm + 8) + dims + (1.0, None), "lse overlaps an input"),
                          (fw32, (A, Bp, O, O + 4 * nm - 4) + dims + (1.0, None), "disp overlaps lse"),
                          (bw32, (A, Bp, O, L, G, G + 4 * nm - 4, None) + dims + (1.0, None), "gradient overlaps"),
                          (bw64, (A, Bp, O, L, G, None, A + 8) + dims + (1.0, None), "gradient overlaps"),
                          (bw32, (A, Bp, O, L, G, 1 << 38, (1 << 38) + 4 * nf - 4) + dims + (1.0, None), "grad_f0 overlaps")):
        with pytest.raises(_lib.CtdError, match=msg):
            fn(*args)
    # an empty batch is a no-op with null pointers; both gradients NULL is a no-op
    fw32(None, None, None, None, 0, 3, 5, 6, 4, 1.0, None)
    fw64(None, None, None, None, 2, 0, 0, 6, 0, 1.0, None)
    bw32(None, None, None, None, None, None, None, 2, 3, 5, 0, 4, 1.0, None)
    bw64(A, Bp, O, L, G, None, None, *dims, 1.0, None)


def test_corr_softargmax_kernels_have_no_atomics(tx):
    from connecting_the_dots_b200 import _lib
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    atomics, kernels, kernel = [], set(), None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            kernel = m.group(1) if "corr_fwd" in m.group(1) or "corr_bwd" in m.group(1) else None
            if kernel:
                kernels.add(kernel)
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d+\s+)?((?:ATOM|RED)[A-Z0-9_.]*)", line)
        if m and kernel:
            atomics.append((kernel, m.group(1)))
    assert len(kernels) == 6, sorted(kernels)   # forward, grad_f0 and grad_f1 for float and double
    assert not atomics, atomics


# ---------------------------------------------------------------- GPU
def feats(g, shape, dtype=torch.float32):
    return torch.randn(shape, device=DEV, generator=g, dtype=torch.float64).to(dtype)


def reference(tx, f0, f1, D, tau, gd):
    """disp, lse, grad_f0, grad_f1 of the restatement in fp64 on the GPU."""
    a = f0.detach().double().requires_grad_(True)
    b = f1.detach().double().requires_grad_(True)
    disp = tx.corr_softargmax_pytorch(a, b, D, tau)
    disp.backward(gd.double())
    fb = (lambda t: t) if f0.dim() == 4 else (lambda t: t.unsqueeze(0))
    return disp.detach(), lse_pytorch(fb(a.detach()), fb(b.detach()), D, tau), a.grad, b.grad


def run_op(tx, f0, f1, D, tau, gd):
    a, b = f0.detach().clone().requires_grad_(True), f1.detach().clone().requires_grad_(True)
    disp = tx.corr_softargmax(a, b, D, tau)
    disp.backward(gd)
    return disp.detach(), a.grad, b.grad


def compare(tx, f0, f1, D, tau, gd, msg, tol_f=None, tol_g=None):
    fp64 = f0.dtype == torch.float64
    tol_f = tol_f or (1e-10 if fp64 else 1e-5)
    tol_g = tol_g or (1e-10 if fp64 else 1e-4)
    rd, _, r0, r1 = reference(tx, f0, f1, D, tau, gd)
    d, g0, g1 = run_op(tx, f0, f1, D, tau, gd)
    assert d.dtype == f0.dtype and d.shape == rd.shape, msg
    e = [assert_close(d.cpu(), rd.cpu(), tol_f, msg + " disp"), assert_close(g0.cpu(), r0.cpu(), tol_g, msg + " grad_f0"),
         assert_close(g1.cpu(), r1.cpu(), tol_g, msg + " grad_f1")]
    return e


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_against_restatement_sizes(tx, dtype):
    """C across one and several channel slabs (32 float / 16 double per slab), D across one and several disparity groups
    and past W, H and W around the 128-pixel chunks."""
    g = torch.Generator(device=DEV).manual_seed(0)
    cases = [(2, C, 5, 33, D) for C in (1, 8, 32, 64, 200) for D in (1, 17)]
    cases += [(2, 8, 3, W, D) for W in (1, 31, 33, 257) for D in (1, 17, 128, 300)]
    cases += [(1, 32, 2, 4097, 128), (1, 3, 1, 4097, 300), (1, 200, 1, 257, 128), (1, 64, 2, 300, 300), (1, 5, 31, 129, 64),
              (1, 1, 257, 31, 17)]
    worst = {}
    for (B, C, H, W, D) in cases:
        for tau in (0.3, 1.0):
            f0, f1 = feats(g, (B, C, H, W), dtype), feats(g, (B, C, H, W), dtype)
            gd = feats(g, (B, 1, H, W), dtype)
            e = compare(tx, f0, f1, D, tau, gd, "B%d C%d H%d W%d D%d tau %g %s" % (B, C, H, W, D, tau, dtype))
            worst = {k: max(worst.get(k, 0), v) for k, v in zip(("disp", "g0", "g1"), e)}
    print("worst relative errors", dtype, worst)


@pytest.mark.gpu
def test_lse_and_large_features(tx):
    """The saved lse against the fp64 definition; features scaled by 1e3 (a naive exp overflows) in fp64."""
    from connecting_the_dots_b200 import _lib
    g = torch.Generator(device=DEV).manual_seed(1)
    for dtype, tol in ((torch.float32, 1e-6), (torch.float64, 1e-12)):
        f0, f1 = feats(g, (2, 16, 3, 200), dtype), feats(g, (2, 16, 3, 200), dtype)
        disp, lse = torch.empty(2, 1, 3, 200, dtype=dtype, device=DEV), torch.empty(2, 1, 3, 200, dtype=dtype, device=DEV)
        _lib.call("ctd_corr_softargmax_fwd" + ("_f32" if dtype == torch.float32 else "_f64"), f0.data_ptr(), f1.data_ptr(),
                  disp.data_ptr(), lse.data_ptr(), 2, 16, 3, 200, 90, 0.7, torch.cuda.current_stream().cuda_stream)
        assert_close(lse.cpu(), lse_pytorch(f0, f1, 90, 0.7).cpu(), tol, "lse %s" % dtype)
    f0, f1 = feats(g, (1, 8, 2, 150), torch.float64) * 1e3, feats(g, (1, 8, 2, 150), torch.float64) * 1e3
    for tau in (0.05, 20.0):
        compare(tx, f0, f1, 64, tau, feats(g, (1, 1, 2, 150), torch.float64), "features x 1e3, tau %g" % tau)


@pytest.mark.gpu
def test_gradcheck_cuda_fp64(tx):
    g = torch.Generator(device=DEV).manual_seed(2)
    f0 = feats(g, (1, 3, 2, 11), torch.float64).requires_grad_(True)
    f1 = feats(g, (1, 3, 2, 11), torch.float64).requires_grad_(True)
    assert torch.autograd.gradcheck(lambda a, b: tx.corr_softargmax(a, b, 6, 0.5), (f0, f1))


def bench_frames(B):
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(B)
    return torch.from_numpy(d["ta"]).to(DEV), torch.from_numpy(d["pat_lcn"]).to(DEV)


@pytest.mark.gpu
def test_bench_frames_batch8(tx):
    """480x640, batch 8, D = 128: the LCN'd IR image against the pattern (C = 1) and random C = 32 features."""
    ta, pat = bench_frames(8)
    g = torch.Generator(device=DEV).manual_seed(3)
    gd = feats(g, (8, 1, 480, 640))
    e1 = compare(tx, ta, pat, 128, 1.0, gd, "bench frames C1")
    f0, f1 = feats(g, (8, 32, 480, 640)), feats(g, (8, 32, 480, 640))
    e32 = compare(tx, f0, f1, 128, 0.5, gd, "random C32")
    print("bench frames C1 rel err", e1, "random C32", e32)


@pytest.mark.gpu
def test_one_input_and_special_grad_disp(tx):
    g = torch.Generator(device=DEV).manual_seed(4)
    f0, f1 = feats(g, (2, 6, 4, 90)), feats(g, (2, 6, 4, 90))
    gd = feats(g, (2, 1, 4, 90))
    _, _, r0, r1 = reference(tx, f0, f1, 40, 1.0, gd)
    for which in (0, 1):
        a = f0.clone().requires_grad_(which == 0)
        b = f1.clone().requires_grad_(which == 1)
        tx.corr_softargmax(a, b, 40, 1.0).backward(gd)
        got, other = (a, b) if which == 0 else (b, a)
        assert other.grad is None
        assert_close(got.grad.cpu(), (r0 if which == 0 else r1).cpu(), 1e-4, "only f%d requires grad" % which)
    a, b = f0.clone().requires_grad_(True), f1.clone().requires_grad_(True)
    tx.corr_softargmax(a, b, 40, 1.0).backward(torch.zeros_like(gd))
    assert not a.grad.any() and not b.grad.any(), "zero grad_disp"
    mixed = torch.where(torch.rand(gd.shape, device=DEV, generator=g) < 0.5, -1.0, 1.0) * (torch.rand(gd.shape, device=DEV, generator=g) < 0.7)
    compare(tx, f0, f1, 40, 1.0, mixed, "mixed-sign grad_disp with zeros")
    with torch.no_grad():
        assert not tx.corr_softargmax(f0, f1, 40).requires_grad
    m = tx.CorrSoftArgmax(40, 1.0)
    assert torch.equal(m(f0, f1), tx.corr_softargmax(f0, f1, 40, 1.0))


@pytest.mark.gpu
def test_deterministic_streams_capture_and_3d(tx):
    from connecting_the_dots_b200 import _lib
    g = torch.Generator(device=DEV).manual_seed(5)
    B, C, H, W, D = 2, 40, 6, 300, 96
    f0, f1, gd = feats(g, (B, C, H, W)), feats(g, (B, C, H, W)), feats(g, (B, 1, H, W))
    ref = run_op(tx, f0, f1, D, 0.8, gd)
    for i in range(3):
        for x, y, n in zip(run_op(tx, f0, f1, D, 0.8, gd), ref, ("disp", "grad_f0", "grad_f1")):
            assert torch.equal(x, y), "call %d: %s differs" % (i, n)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        on_s = run_op(tx, f0, f1, D, 0.8, gd)
    s.synchronize()
    assert all(torch.equal(x, y) for x, y in zip(on_s, ref)), "side stream"
    disp, lse = torch.zeros(B, 1, H, W, device=DEV), torch.zeros(B, 1, H, W, device=DEV)
    g0, g1 = torch.zeros_like(f0), torch.zeros_like(f1)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        st = torch.cuda.current_stream().cuda_stream
        _lib.call("ctd_corr_softargmax_fwd_f32", f0.data_ptr(), f1.data_ptr(), disp.data_ptr(), lse.data_ptr(), B, C, H, W, D,
                  0.8, st)
        _lib.call("ctd_corr_softargmax_bwd_f32", f0.data_ptr(), f1.data_ptr(), disp.data_ptr(), lse.data_ptr(), gd.data_ptr(),
                  g0.data_ptr(), g1.data_ptr(), B, C, H, W, D, 0.8, st)
    for _ in range(2):
        for t in (disp, lse, g0, g1):
            t.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(disp, ref[0]) and torch.equal(g0, ref[1]) and torch.equal(g1, ref[2]), "graph replay"
    d3, a3, b3 = run_op(tx, f0[1], f1[1], D, 0.8, gd[1])
    assert d3.shape == (1, H, W)
    assert torch.equal(d3, ref[0][1]) and torch.equal(a3, ref[1][1]) and torch.equal(b3, ref[2][1]), "[C,H,W] input"


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", (torch.float32, torch.float64))
def test_misaligned_views(tx, dtype):
    """Every C-ABI pointer one element off any alignment; W = 67 (rows not aligned to each other either)."""
    from connecting_the_dots_b200 import _lib
    g = torch.Generator(device=DEV).manual_seed(6)
    B, C, H, W, D = 2, 5, 7, 67, 30
    f0, f1, gd = feats(g, (B, C, H, W), dtype), feats(g, (B, C, H, W), dtype), feats(g, (B, 1, H, W), dtype)
    rd, rl, r0, r1 = reference(tx, f0, f1, D, 1.0, gd)

    def view(src, n):
        v = torch.zeros(1 + n, dtype=dtype, device=DEV)[1:]
        if src is not None:
            v.copy_(src.reshape(-1))
        return v
    nf, nm = B * C * H * W, B * H * W
    a, b, gv = view(f0, nf), view(f1, nf), view(gd, nm)
    disp, lse, g0, g1 = view(None, nm), view(None, nm), view(None, nf), view(None, nf)
    assert a.data_ptr() % 16 and disp.data_ptr() % 16
    sfx, st = "_f32" if dtype == torch.float32 else "_f64", torch.cuda.current_stream().cuda_stream
    _lib.call("ctd_corr_softargmax_fwd" + sfx, a.data_ptr(), b.data_ptr(), disp.data_ptr(), lse.data_ptr(), B, C, H, W, D, 1.0, st)
    _lib.call("ctd_corr_softargmax_bwd" + sfx, a.data_ptr(), b.data_ptr(), disp.data_ptr(), lse.data_ptr(), gv.data_ptr(),
              g0.data_ptr(), g1.data_ptr(), B, C, H, W, D, 1.0, st)
    tol_f, tol_g = (1e-5, 1e-4) if dtype == torch.float32 else (1e-10, 1e-10)
    assert_close(disp.view(B, 1, H, W).cpu(), rd.cpu(), tol_f, "disp")
    assert_close(lse.view(B, 1, H, W).cpu(), rl.cpu(), tol_f, "lse")
    assert_close(g0.view(B, C, H, W).cpu(), r0.cpu(), tol_g, "grad_f0")
    assert_close(g1.view(B, C, H, W).cpu(), r1.cpu(), tol_g, "grad_f1")


@pytest.mark.gpu
def test_errors_and_empty(tx):
    from connecting_the_dots_b200 import _lib
    f = torch.rand(2, 3, 16, 20, device=DEV)
    for bad, exc in (((f.transpose(2, 3), f.transpose(2, 3), 4), RuntimeError), ((f, f.double(), 4), RuntimeError),
                     ((f, f.cpu(), 4), RuntimeError), ((f.half(), f.half(), 4), NotImplementedError),
                     ((f, f, 0), RuntimeError), ((f, f, 4, 0.0), RuntimeError), ((f, f[:, :2], 4), RuntimeError)):
        with pytest.raises(exc):
            tx.corr_softargmax(*bad)
    st = torch.cuda.current_stream().cuda_stream
    disp, lse = torch.empty(2, 1, 16, 20, device=DEV), torch.empty(2, 1, 16, 20, device=DEV)
    with pytest.raises(_lib.CtdError, match="disp overlaps an input"):
        _lib.call("ctd_corr_softargmax_fwd_f32", f.data_ptr(), f.data_ptr(), f.data_ptr() + 4, lse.data_ptr(), 2, 3, 16, 20, 4, 1.0, st)
    with pytest.raises(_lib.CtdError, match="gradient overlaps"):
        _lib.call("ctd_corr_softargmax_bwd_f32", f.data_ptr(), f.data_ptr(), disp.data_ptr(), lse.data_ptr(), disp.data_ptr(),
                  lse.data_ptr(), None, 2, 3, 16, 20, 4, 1.0, st)
    before = _lib.launch_count()
    e0 = torch.rand(0, 3, 16, 20, device=DEV, requires_grad=True)
    out = tx.corr_softargmax(e0, e0.detach(), 4)
    assert out.shape == (0, 1, 16, 20)
    out.sum().backward()
    assert e0.grad.shape == e0.shape
    assert tx.corr_softargmax(torch.rand(2, 3, 0, 20, device=DEV), torch.rand(2, 3, 0, 20, device=DEV), 4).shape == (2, 1, 0, 20)
    _lib.call("ctd_corr_softargmax_bwd_f32", f.data_ptr(), f.data_ptr(), disp.data_ptr(), lse.data_ptr(), disp.data_ptr(),
              None, None, 2, 3, 16, 20, 4, 1.0, st)
    assert _lib.launch_count() == before, "an empty batch or two null gradients launch nothing"
    a = f.clone().requires_grad_(True)
    tx.corr_softargmax(a, f, 4).sum().backward()
    assert _lib.launch_count() == before + 2, "one forward and one gradient launch"


@pytest.mark.gpu
def test_past_2_31_elements(tx):
    """2049 images of 2 x 512 x 1024: 2.15e9 elements per feature map.  The last image equals a call on it alone."""
    B, C, H, W, D = 2049, 2, 512, 1024, 17
    assert B * C * H * W > 2 ** 31
    g = torch.Generator(device=DEV).manual_seed(7)
    f0, f1 = torch.randn(B, C, H, W, device=DEV, generator=g), torch.randn(B, C, H, W, device=DEV, generator=g)
    gd = torch.randn(B, 1, H, W, device=DEV, generator=g)
    a, b = f0.requires_grad_(True), f1.requires_grad_(True)
    disp = tx.corr_softargmax(a, b, D, 1.0)
    disp.backward(gd)
    last = run_op(tx, f0[-1:].detach().clone(), f1[-1:].detach().clone(), D, 1.0, gd[-1:].clone())
    assert torch.equal(disp[-1:].detach(), last[0]), "disp of the last image"
    assert torch.equal(a.grad[-1:], last[1]) and torch.equal(b.grad[-1:], last[2]), "gradients of the last image"
    ref = reference(tx, f0[-1:, :, :64].detach(), f1[-1:, :, :64].detach(), D, 1.0, gd[-1:, :, :64])
    assert_close(last[0][:, :, :64].cpu(), ref[0].cpu(), 1e-5, "last image vs restatement")
