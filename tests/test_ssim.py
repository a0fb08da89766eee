"""SSIM photometric loss (ssim.cu, torchext.ssim_loss / weighted_ssim_loss).

The reference has no SSIM op, so the oracle is the definition itself, written down twice: a brute-force numpy loop over
pixels and clamped taps, and the float64 torch restatement ssim_loss_pytorch (autograd gives its gradient).  The CPU
tests pin the restatement and the closed-form gradient to the definition; the GPU tests hold the kernels to the
restatement with the repo comparator (max |got - ref| <= tol * max |ref|).
"""
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from conftest import assert_close

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
C1, C2 = 0.01 ** 2, 0.03 ** 2


def _F():
    from connecting_the_dots_b200.torchext import functions
    return functions


def ssim_brute(es, ta, bs, c1=C1, c2=C2):
    """The definition, one pixel and one tap at a time (float64)."""
    B, C, H, W = es.shape
    out = np.zeros((B, 1, H, W))
    n = bs * bs
    for b in range(B):
        for c in range(C):
            for h in range(H):
                for w in range(W):
                    xs, ys = [], []
                    for i in range(bs):
                        for j in range(bs):
                            hh = min(max(h + i - bs // 2, 0), H - 1)
                            ww = min(max(w + j - bs // 2, 0), W - 1)
                            xs.append(float(es[b, c, hh, ww]))
                            ys.append(float(ta[b, c, hh, ww]))
                    mx, my = sum(xs) / n, sum(ys) / n
                    vxx = sum((x - mx) ** 2 for x in xs) / n
                    vyy = sum((y - my) ** 2 for y in ys) / n
                    vxy = sum((x - mx) * (y - my) for x, y in zip(xs, ys)) / n
                    s = (2 * mx * my + c1) * (2 * vxy + c2) / ((mx * mx + my * my + c1) * (vxx + vyy + c2))
                    out[b, 0, h, w] += (1 - s) / 2
    return out


def ssim_grad_closed_form(es, ta, go, bs, c1=C1, c2=C2):
    """grad_es[p] = -1/2 sum_w m(w,p) go[w] (a_w + beta_w (x_p - mx_w) + gamma_w (y_p - my_w)), the multiplicity m coming
    from visiting every clamped tap of every window (float64)."""
    B, C, H, W = es.shape
    n = bs * bs
    lo = bs // 2
    hh = np.clip(np.arange(H)[:, None] + np.arange(bs)[None, :] - lo, 0, H - 1)  # [H, bs]
    ww = np.clip(np.arange(W)[:, None] + np.arange(bs)[None, :] - lo, 0, W - 1)  # [W, bs]
    grad = np.zeros_like(es, dtype=np.float64)
    for b in range(B):
        for c in range(C):
            x, y, g = es[b, c].astype(np.float64), ta[b, c].astype(np.float64), go[b, 0].astype(np.float64)
            tx_ = [x[hh[:, i]][:, ww[:, j]] for i in range(bs) for j in range(bs)]
            ty_ = [y[hh[:, i]][:, ww[:, j]] for i in range(bs) for j in range(bs)]
            mx, my = sum(tx_) / n, sum(ty_) / n
            vxx = sum((t - mx) ** 2 for t in tx_) / n
            vyy = sum((t - my) ** 2 for t in ty_) / n
            vxy = sum((p - mx) * (q - my) for p, q in zip(tx_, ty_)) / n
            A1, A2 = 2 * mx * my + c1, 2 * vxy + c2
            B1, B2 = mx * mx + my * my + c1, vxx + vyy + c2
            S = A1 * A2 / (B1 * B2)
            a = 2 * (my * A2 / B2 - mx * S) / (n * B1)
            beta = -2 * S / (n * B2)
            gamma = 2 * A1 / (n * B1 * B2)
            for i in range(bs):
                for j in range(bs):
                    rows, cols = hh[:, i][:, None], ww[:, j][None, :]
                    xp, yp = x[rows, cols], y[rows, cols]
                    term = -0.5 * g * (a + beta * (xp - mx) + gamma * (yp - my))
                    np.add.at(grad[b, c], (np.broadcast_to(rows, term.shape), np.broadcast_to(cols, term.shape)), term)
    return grad


# ---------------------------------------------------------------- CPU: the oracle and the API surface
@pytest.mark.parametrize("bs", (1, 2, 3, 4, 9))
@pytest.mark.parametrize("C", (1, 3))
def test_restatement_matches_brute_force_definition(bs, C):
    rng = np.random.RandomState(bs * 10 + C)
    es = rng.rand(2, C, 5, 7)
    ta = np.clip(es + 0.2 * rng.randn(2, C, 5, 7), 0, 1)
    got = _F().ssim_loss_pytorch(torch.from_numpy(es), torch.from_numpy(ta), bs).numpy()
    assert got.shape == (2, 1, 5, 7)
    assert_close(got, ssim_brute(es, ta, bs), tol=1e-12, what="restatement vs definition")


def test_restatement_known_answers():
    F = _F()
    rng = np.random.RandomState(3)
    x = torch.from_numpy(rng.rand(1, 2, 9, 11))
    assert float(F.ssim_loss_pytorch(x, x, 5).abs().max()) <= 1e-15          # identical images: S = 1
    a, b, C = 0.3, 0.7, 3
    got = F.ssim_loss_pytorch(torch.full((1, C, 6, 8), a, dtype=torch.float64), torch.full((1, C, 6, 8), b, dtype=torch.float64), 3)
    want = C * (1 - (2 * a * b + C1) / (a * a + b * b + C1)) / 2                # constant planes: only the luminance term
    assert np.allclose(got.numpy(), want, rtol=1e-14, atol=0)
    es, ta = rng.rand(1, 1, 2, 3), rng.rand(1, 1, 2, 3)                         # image smaller than the window
    small = F.ssim_loss_pytorch(torch.from_numpy(es), torch.from_numpy(ta), 9).numpy()
    assert_close(small, ssim_brute(es, ta, 9), tol=1e-12, what="image smaller than the window")


def test_restatement_gradcheck_and_closed_form_gradient():
    F = _F()
    rng = np.random.RandomState(5)
    es = torch.from_numpy(rng.rand(1, 2, 5, 6)).requires_grad_(True)
    ta = torch.from_numpy(rng.rand(1, 2, 5, 6))
    assert torch.autograd.gradcheck(lambda e: F.ssim_loss_pytorch(e, ta, 3), (es,))
    for bs, shape in ((3, (2, 2, 7, 9)), (4, (1, 2, 6, 8)), (9, (1, 2, 11, 12)), (9, (1, 1, 3, 4))):
        e = rng.rand(*shape)
        t = np.clip(e + 0.3 * rng.randn(*shape), 0, 1)
        go = rng.randn(shape[0], 1, shape[2], shape[3])
        et = torch.from_numpy(e).requires_grad_(True)
        (g,) = torch.autograd.grad(F.ssim_loss_pytorch(et, torch.from_numpy(t), bs), et, torch.from_numpy(go))
        assert_close(ssim_grad_closed_form(e, t, go, bs), g.numpy(), tol=1e-12, what="closed form bs %d" % bs)


def test_ssim_api_surface_and_no_cpu_fallback(tx):
    x = torch.rand(1, 1, 12, 12)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        tx.ssim_loss(x, x, 3)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        tx.weighted_ssim_loss(x, x, torch.ones_like(x), 3)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        tx.SSIMLoss(9)(x, x)
    with pytest.raises(Exception, match="invalid loss type"):       # photometric_loss keeps its reference contract
        tx.photometric_loss(x, x, 9, "ssim")
    assert "ssim" not in tx.LOSS_TYPES


def test_ssim_argument_validation_without_gpu(tx):
    from connecting_the_dots_b200 import _lib
    with pytest.raises(_lib.CtdError, match="block_size"):
        _lib.call("ctd_ssim_fwd_f32", 16, 16, 16, 1, 1, 8, 8, 0, C1, C2, None)
    with pytest.raises(_lib.CtdError, match="c1 and c2"):
        _lib.call("ctd_ssim_bwd_f32", 16, 16, 16, 16, 1, 1, 8, 8, 3, C1, 0.0, None)
    with pytest.raises(_lib.CtdError, match="c1 and c2"):
        _lib.call("ctd_ssim_fwd_f64", 16, 16, 16, 1, 1, 8, 8, 3, -1.0, C2, None)
    with pytest.raises(_lib.CtdError, match="null pointer"):
        _lib.call("ctd_ssim_fwd_f32", None, None, None, 1, 1, 8, 8, 3, C1, C2, None)
    with pytest.raises(_lib.CtdError, match="null pointer"):
        _lib.call("ctd_ssim_fwd_bwd_masked_f32", 16, 16, 16, 16, 16, 16, None, 1, 1, 8, 8, 3, C1, C2, None)
    # an empty batch is a no-op
    _lib.call("ctd_ssim_fwd_f32", None, None, None, 0, 1, 8, 8, 3, C1, C2, None)
    _lib.call("ctd_ssim_bwd_f64", None, None, None, None, 0, 1, 8, 8, 3, C1, C2, None)


def test_ssim_kernels_have_no_floating_point_atomics(tx):
    """The only atomics in ssim.cu are the integer ticket of finish_masked_sums, one per masked kernel."""
    from connecting_the_dots_b200 import _lib
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    atomics, kernel = [], None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            kernel = m.group(1)
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,6}\*/\s+(?:@!?U?P\d+\s+)?((?:ATOM|RED)[A-Z0-9_.]*)", line)
        if m and kernel and "ssim" in kernel:
            atomics.append((kernel, m.group(1)))
    assert atomics, "no ssim kernel found in the library"
    for k, op in atomics:
        assert "ssim_bwd_tile" in k and not re.search(r"F16|F32|F64|BF16", op), (k, op)


# ---------------------------------------------------------------- GPU: kernels against the restatement
def cu(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


def ref64(es, ta, go, bs, c1=C1, c2=C2):
    """float64 restatement on the GPU: loss map and autograd gradient w.r.t. es."""
    e = cu(es, torch.float64).requires_grad_(True)
    out = _F().ssim_loss_pytorch(e, cu(ta, torch.float64), bs, c1, c2)
    (g,) = torch.autograd.grad(out, e, cu(go, torch.float64))
    return out.detach().cpu().numpy(), g.cpu().numpy()


def kernels(tx, es, ta, go, bs, dtype=torch.float32, c1=C1, c2=C2):
    e = cu(es, dtype).requires_grad_(True)
    out = tx.ssim_loss(e, cu(ta, dtype), bs, c1, c2)
    out.backward(cu(go, dtype))
    return out.detach().cpu().numpy(), e.grad.cpu().numpy()


def pair(rng, B, C, H, W):
    es = rng.rand(B, C, H, W).astype(np.float32)
    ta = np.clip(es + 0.15 * rng.randn(B, C, H, W), 0, 1).astype(np.float32)
    go = rng.randn(B, 1, H, W).astype(np.float32)
    return es, ta, go


# B, H, W: ragged widths (scalar path), multi-tile with W % 4 == 0 (128-bit path), H < bs, W < bs, W % 4 == 2
SHAPES = [(2, 37, 45), (1, 70, 132), (1, 5, 40), (1, 40, 6), (3, 33, 66)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("C", (1, 3))
@pytest.mark.parametrize("bs", (1, 2, 3, 4, 5, 7, 9, 11))
def test_ssim_f32_vs_restatement(tx, bs, C, shape):
    B, H, W = shape
    es, ta, go = pair(np.random.RandomState(bs * 1000 + C * 100 + W), B, C, H, W)
    fwd, bwd = kernels(tx, es, ta, go, bs)
    rf, rb = ref64(es, ta, go, bs)
    assert_close(fwd, rf, what="fwd")
    assert_close(bwd, rb, what="bwd")


@pytest.mark.gpu
@pytest.mark.parametrize("bs", (3, 9))
def test_ssim_f32_full_size_batch(tx, bs):
    es, ta, go = pair(np.random.RandomState(bs), 2, 1, 480, 640)
    fwd, bwd = kernels(tx, es, ta, go, bs)
    rf, rb = ref64(es, ta, go, bs)
    assert_close(fwd, rf, what="fwd")
    assert_close(bwd, rb, what="bwd")


@pytest.mark.gpu
@pytest.mark.parametrize("bs", (3, 9))
@pytest.mark.parametrize("data", ("ir", "lcn"))
def test_ssim_f32_on_synthetic_frames(tx, bs, data):
    """Raw IR frames in [0, 1] (clipped flat regions: window variance ~0, the case the centred moments are for) and the
    LCN'd estimate / target pair of the trainer."""
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(2)
    if data == "ir":
        es, ta = d["im"], np.ascontiguousarray(np.roll(d["im"], 2, axis=3))
    else:
        es, ta = d["es"], d["ta"]
    fwd, bwd = kernels(tx, es, ta, d["go"], bs)
    rf, rb = ref64(es, ta, d["go"], bs)
    assert_close(fwd, rf, what="fwd")
    assert_close(bwd, rb, what="bwd")


@pytest.mark.gpu
@pytest.mark.parametrize("bs", (2, 3, 9))
@pytest.mark.parametrize("C", (1, 3))
def test_ssim_f64_vs_restatement(tx, bs, C):
    rng = np.random.RandomState(bs + C)
    es = rng.rand(2, C, 23, 30)
    ta = np.clip(es + 0.2 * rng.randn(2, C, 23, 30), 0, 1)
    go = rng.randn(2, 1, 23, 30)
    fwd, bwd = kernels(tx, es, ta, go, bs, torch.float64)
    rf, rb = ref64(es, ta, go, bs)
    assert_close(fwd, rf, tol=1e-10, what="fwd64")
    assert_close(bwd, rb, tol=1e-10, what="bwd64")


@pytest.mark.gpu
@pytest.mark.parametrize("bs", (3, 9, 11))
def test_ssim_force_generic_agrees(tx, bs):
    from connecting_the_dots_b200 import _lib
    es, ta, go = pair(np.random.RandomState(bs), 2, 2, 45, 70)
    mask = np.random.RandomState(1).rand(2, 1, 45, 70).astype(np.float32)
    args = (cu(es), cu(ta), cu(go), cu(mask), bs, C1, C2)
    fast = (tx.ext_cuda.ssim_forward(*args[:2], bs, C1, C2), tx.ext_cuda.ssim_backward(*args[:3], bs, C1, C2),
            *tx.ext_cuda.ssim_forward_backward_masked(*args))
    _lib.set_option("force_generic", 1)
    try:
        slow = (tx.ext_cuda.ssim_forward(*args[:2], bs, C1, C2), tx.ext_cuda.ssim_backward(*args[:3], bs, C1, C2),
                *tx.ext_cuda.ssim_forward_backward_masked(*args))
    finally:
        _lib.set_option("force_generic", 0)
    for name, a, b in zip(("fwd", "bwd", "fused fwd", "fused bwd", "fused sums"), fast, slow):
        assert_close(a.cpu().numpy(), b.cpu().numpy(), tol=1e-6, what="tile vs generic " + name)


@pytest.mark.gpu
@pytest.mark.parametrize("bs", (3, 9))
def test_ssim_fused_masked_matches_separate_calls(tx, bs):
    from connecting_the_dots_b200 import _lib
    es, ta, go = pair(np.random.RandomState(20 + bs), 3, 1, 96, 160)
    mask = np.random.RandomState(2).rand(3, 1, 96, 160).astype(np.float32)
    e, t, g, m = cu(es), cu(ta), cu(go), cu(mask)
    out0 = tx.ext_cuda.ssim_forward(e, t, bs, C1, C2)
    gi0 = tx.ext_cuda.ssim_backward(e, t, g, bs, C1, C2)
    sums0 = tx.masked_mean_terms(out0, m)
    runs = [tx.ext_cuda.ssim_forward_backward_masked(e, t, g, m, bs, C1, C2) for _ in range(2)]
    out, gi, sums = runs[0]
    assert_close(out.cpu().numpy(), out0.cpu().numpy(), tol=1e-6, what="fused loss map")
    assert torch.equal(gi, gi0), "the fused kernel's gradient is the stand-alone backward's"
    assert_close(sums.cpu().numpy(), sums0.cpu().numpy(), tol=1e-6, what="sums")
    for a, b in zip(runs[0], runs[1]):
        assert torch.equal(a, b), "two calls differ"
    # capture into a CUDA graph, replay on a non-default stream: the same bits
    o2, g2, s2 = torch.empty_like(out), torch.empty_like(gi), torch.empty_like(sums)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _lib.call("ctd_ssim_fwd_bwd_masked_f32", e.data_ptr(), t.data_ptr(), g.data_ptr(), m.data_ptr(), o2.data_ptr(), g2.data_ptr(),
                  s2.data_ptr(), 3, 1, 96, 160, bs, C1, C2, torch.cuda.current_stream().cuda_stream)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    for _ in range(2):
        for x in (o2, g2, s2):
            x.zero_()
        torch.cuda.synchronize()
        with torch.cuda.stream(s):
            graph.replay()
        s.synchronize()
        assert torch.equal(o2, out) and torch.equal(g2, gi) and torch.equal(s2, sums)


@pytest.mark.gpu
@pytest.mark.parametrize("bs", (3, 9))
def test_weighted_ssim_loss_matches_composition(tx, bs):
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(2, 96, 160)
    es = cu(d["im"]).requires_grad_(True)
    ta, mask = cu(np.roll(d["im"], 3, axis=3)), cu(d["std"])
    e64 = cu(d["im"], torch.float64).requires_grad_(True)
    ref = (mask.double() * _F().ssim_loss_pytorch(e64, ta.double(), bs)).sum() / mask.double().sum()
    (gref,) = torch.autograd.grad(3.0 * ref, e64)
    val, loss_map = tx.weighted_ssim_loss(es, ta, mask, bs)
    (g,) = torch.autograd.grad(3.0 * val, es)
    assert abs(val.item() - ref.item()) <= 1e-5 * abs(ref.item())
    assert_close(g.cpu().numpy(), gref.cpu().numpy(), what="weighted loss gradient")
    assert_close(loss_map.cpu().numpy(), tx.ssim_loss(es.detach(), ta, bs).cpu().numpy(), tol=1e-6, what="loss map")


@pytest.mark.gpu
def test_ssim_errors_and_empty(tx):
    x = torch.rand(1, 1, 16, 16, device=DEV)
    with pytest.raises(RuntimeError):
        tx.ssim_loss(x, x[:, :, :8].contiguous(), 3)                  # shape mismatch
    with pytest.raises(RuntimeError):
        tx.ssim_loss(x.transpose(2, 3), x, 3)                         # non-contiguous
    with pytest.raises(NotImplementedError):
        tx.ssim_loss(x.half(), x.half(), 3)
    with pytest.raises(RuntimeError, match="block_size"):
        tx.ssim_loss(x, x, 0)
    with pytest.raises(RuntimeError, match="c1 and c2"):
        tx.ssim_loss(x, x, 3, C1, 0.0)
    with pytest.raises(RuntimeError):
        tx.ext_cuda.ssim_forward_backward_masked(x.double(), x.double(), x.double(), x.double(), 3, C1, C2)  # fp32 only
    e = torch.zeros(0, 2, 16, 16, device=DEV, requires_grad=True)
    out = tx.ssim_loss(e, e.detach(), 9)
    assert out.shape == (0, 1, 16, 16)
    out.sum().backward()
    assert e.grad.shape == e.shape
    z = torch.zeros(0, 1, 16, 16, device=DEV)
    o, g, s = tx.ext_cuda.ssim_forward_backward_masked(z, z, z, z, 9, C1, C2)
    assert o.shape == z.shape and g.shape == z.shape and s.tolist() == [0.0, 0.0]
    assert tx.ssim_loss(x, x, 9).abs().max().item() <= 1e-6                # identical images
    assert tx.SSIMLoss(9)(x, x).shape == (1, 1, 16, 16)
