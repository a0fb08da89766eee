"""GPU parity suite (-m gpu): every op of the drop-in torchext package, called through the C ABI of
libctd_b200.so, against the CPU oracle (oracle/ctd_oracle.c, pinned to the reference by
tests/test_oracle.py) and the committed golden vectors of the unmodified reference.

Tolerances: bit-exact for CrossCheck masks and NN / ProjNN indices; 1e-5 relative for loss maps,
gradients, cost volumes and LCN, with the comparator tests/conftest.py:assert_close
(max |got - ref| <= 1e-5 * max |ref|).
"""
import ctypes

import numpy as np
import pytest
import torch

import oracle
from conftest import assert_close

pytestmark = pytest.mark.gpu
TYPES = ("mse", "sad", "census_mse", "census_sad")
DEV = "cuda:0"


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def photometric_both(tx, es, ta, go, bs, ty, eps):
    e = cu(es).requires_grad_(True)
    out = tx.photometric_loss(e, cu(ta), bs, TYPES[ty], eps)
    out.backward(cu(go))
    return out.detach().cpu().numpy(), e.grad.cpu().numpy()


# ---------------------------------------------------------------- photometric loss
@pytest.mark.parametrize("C", (1, 2))
@pytest.mark.parametrize("bs", (2, 3, 9))
@pytest.mark.parametrize("ty", range(4))
def test_photometric_golden(tx, golden, C, bs, ty):
    g = golden("photometric")
    es, ta, go = g[f"f32_C{C}_es"], g[f"f32_C{C}_ta"], g[f"f32_C{C}_go"]
    eps = 0.5 if ty == 3 else 0.1
    fwd, bwd = photometric_both(tx, es, ta, go, bs, ty, eps)
    assert_close(fwd, g[f"f32_C{C}_bs{bs}_t{ty}_fwd"], what="fwd")
    assert_close(bwd, g[f"f32_C{C}_bs{bs}_t{ty}_bwd"], what="bwd")


@pytest.mark.parametrize("ty", range(4))
def test_photometric_golden_f64(tx, golden, ty):
    g = golden("photometric")
    for C in (1, 2):
        es, ta, go = g[f"f64_C{C}_es"], g[f"f64_C{C}_ta"], g[f"f64_C{C}_go"]
        eps = 0.5 if ty == 3 else 0.1
        fwd, bwd = photometric_both(tx, es, ta, go, 9, ty, eps)
        assert fwd.dtype == np.float64
        assert_close(fwd, g[f"f64_C{C}_bs9_t{ty}_fwd"], tol=1e-12, what="fwd64")
        assert_close(bwd, g[f"f64_C{C}_bs9_t{ty}_bwd"], tol=1e-12, what="bwd64")


SHAPES = [  # B, C, H, W, bs -- ragged widths (scalar path), multi-tile, tiny (generic path), block sizes
    (2, 1, 33, 132, 9), (1, 1, 40, 67, 9), (1, 2, 64, 256, 9), (1, 1, 9, 9, 9), (3, 1, 70, 200, 9),
    (1, 3, 17, 23, 9), (1, 1, 5, 6, 9), (1, 1, 3, 3, 9), (2, 1, 20, 31, 5), (1, 2, 16, 16, 4), (1, 1, 12, 40, 1),
    (1, 1, 8, 300, 9), (1, 1, 300, 12, 9),
    # more census widths and heights: 120, 160 and 44 columns, 16 x 16
    (1, 1, 48, 120, 9), (2, 1, 40, 160, 9), (3, 1, 100, 44, 9), (1, 1, 16, 16, 9),
]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("ty", range(4))
def test_photometric_vs_oracle(tx, shape, ty):
    B, C, H, W, bs = shape
    rng = np.random.RandomState(hash(shape) % 2**31)
    es = rng.randn(B, C, H, W).astype(np.float32)
    ta = (es + 0.7 * rng.randn(B, C, H, W)).astype(np.float32)
    es[0, 0, H // 2, W // 2] = ta[0, 0, H // 2, W // 2]
    go = rng.rand(B, 1, H, W).astype(np.float32)
    eps = 0.5
    fwd, bwd = photometric_both(tx, es, ta, go, bs, ty, eps)
    assert_close(fwd, oracle.photometric_loss_forward(es, ta, bs, ty, eps), what="fwd")
    assert_close(bwd, oracle.photometric_loss_backward(es, ta, go, bs, ty, eps), what="bwd")


@pytest.mark.parametrize("ty", range(4))
def test_photometric_generic_kernels_agree(tx, ty):
    """force_generic routes block-size-9 fp32 through the generic kernels as well."""
    from connecting_the_dots_b200 import _lib
    rng = np.random.RandomState(5)
    es = rng.randn(2, 2, 30, 44).astype(np.float32)
    ta = rng.randn(2, 2, 30, 44).astype(np.float32)
    go = rng.randn(2, 1, 30, 44).astype(np.float32)  # signed upstream gradient
    _lib.set_option("force_generic", 1)
    try:
        fwd, bwd = photometric_both(tx, es, ta, go, 9, ty, 0.3)
    finally:
        _lib.set_option("force_generic", 0)
    assert_close(fwd, oracle.photometric_loss_forward(es, ta, 9, ty, 0.3), what="fwd")
    assert_close(bwd, oracle.photometric_loss_backward(es, ta, go, 9, ty, 0.3), what="bwd")
    fwd2, bwd2 = photometric_both(tx, es, ta, go, 9, ty, 0.3)
    assert_close(fwd2, fwd, what="fast vs generic fwd")
    assert_close(bwd2, bwd, what="fast vs generic bwd")


SYM_SHAPES = [(1, 16, 16), (2, 33, 132), (1, 40, 67), (1, 130, 200), (1, 250, 48), (3, 128, 36), (1, 129, 150), (2, 61, 301)]


def _census_all_entry_points(tx, es, ta, go, mask, ty, eps=0.5):
    """forward, backward, fused forward+backward and the fused masked call of one census mode -> dict of numpy arrays"""
    from connecting_the_dots_b200 import _lib
    B, _, H, W = es.shape
    e, t, g, m = cu(es), cu(ta), cu(go), cu(mask)
    r = {"fwd": tx.ext_cuda.photometric_loss_forward(e, t, 9, ty, eps), "bwd": tx.ext_cuda.photometric_loss_backward(e, t, g, 9, ty, eps)}
    r["f_fwd"], r["f_bwd"] = tx.ext_cuda.photometric_loss_forward_backward(e, t, g, 9, ty, eps)
    out, gi, sums = torch.empty_like(e), torch.empty_like(e), torch.zeros(2, device=DEV)
    _lib.call("ctd_photometric_fwd_bwd_masked_f32", e.data_ptr(), t.data_ptr(), g.data_ptr(), m.data_ptr(), out.data_ptr(), gi.data_ptr(),
              sums.data_ptr(), B, 1, H, W, 9, ty, eps, torch.cuda.current_stream().cuda_stream)
    r["m_fwd"], r["m_bwd"], r["sums"] = out, gi, sums
    return {k: v.cpu().numpy() for k, v in r.items()}


@pytest.mark.parametrize("shape", SYM_SHAPES)
@pytest.mark.parametrize("ty", (2, 3))
def test_census_pair_symmetric_kernel_vs_oracle(tx, shape, ty):
    """census_sym.cu (every pixel pair evaluated once) through all four entry points against the oracle: one and several
    strips (120 useful rows each), one and several column tiles, widths that are / are not multiples of four (128-bit
    and scalar staging), rows below the last strip, the clamped border band."""
    B, H, W = shape
    rng = np.random.RandomState(H * 1000 + W + ty)
    es = rng.randn(B, 1, H, W).astype(np.float32)
    ta = (es + 0.6 * rng.randn(B, 1, H, W)).astype(np.float32)
    go = rng.randn(B, 1, H, W).astype(np.float32)
    mask = (rng.rand(B, 1, H, W) + 0.5).astype(np.float32)
    from connecting_the_dots_b200 import _lib
    _lib.set_option("census_sym", 1)   # every entry point through the pair-symmetric kernel (default: forward only)
    try:
        r = _census_all_entry_points(tx, es, ta, go, mask, ty)
    finally:
        _lib.set_option("census_sym", 2)
    of, ob = oracle.photometric_loss_forward(es, ta, 9, ty, 0.5), oracle.photometric_loss_backward(es, ta, go, 9, ty, 0.5)
    for k in ("fwd", "f_fwd", "m_fwd"):
        assert_close(r[k], of, what=k)
    for k in ("bwd", "f_bwd", "m_bwd"):
        assert_close(r[k], ob, what=k)
    want = np.array([(mask.astype(np.float64) * of).sum(), mask.astype(np.float64).sum()])
    assert np.abs(r["sums"] - want).max() <= 1e-5 * np.abs(want).max()


@pytest.mark.parametrize("ty", (2, 3))
def test_census_pair_symmetric_kernel_matches_gather_kernels(tx, ty):
    """A/B inside the library at the bench size: pair-symmetric kernel (census_sym = 1) against the gather kernels."""
    from connecting_the_dots_b200 import _lib, synth
    d = synth.make_batch(3)
    _lib.set_option("census_sym", 1)
    try:
        a = _census_all_entry_points(tx, d["es"], d["ta"], d["go"], d["std"], ty)
        again = _census_all_entry_points(tx, d["es"], d["ta"], d["go"], d["std"], ty)
        _lib.set_option("census_sym", 0)
        b = _census_all_entry_points(tx, d["es"], d["ta"], d["go"], d["std"], ty)
    finally:
        _lib.set_option("census_sym", 2)
    for k in a:
        if k == "sums":
            assert np.abs(a[k] - b[k]).max() <= 1e-5 * np.abs(b[k]).max()
        else:
            assert_close(a[k], b[k], what=k)
    for k in a:
        assert np.array_equal(a[k], again[k]), "run-to-run difference in " + k


def test_census_pair_symmetric_kernel_exact_sign_decisions(tx):
    """census_sad's sign(): images quantised to a few levels make many window terms EXACTLY zero (sign 0 in the reference)
    or equal up to rounding; every such pixel has to come out of the exact pass like ext_cpu's.  Also a constant image
    (every pair a tie) and a pair of images that differ in one pixel."""
    rng = np.random.RandomState(5)
    B, H, W = 2, 70, 120
    es = rng.randint(0, 3, (B, 1, H, W)).astype(np.float32)
    ta = rng.randint(0, 3, (B, 1, H, W)).astype(np.float32)
    go = rng.rand(B, 1, H, W).astype(np.float32)
    cases = [(es, ta), (es, es.copy()), (np.full_like(es, 0.25), np.full_like(es, 0.75))]
    one = es.copy()
    one[0, 0, 30, 50] += 1.0
    cases.append((one, es))
    from connecting_the_dots_b200 import _lib
    for mode in (1, 2):   # the pair-symmetric kernel's exact pass, then the default dispatch (gather kernel's exact pass)
        _lib.set_option("census_sym", mode)
        try:
            for e, t in cases:
                fwd, bwd = photometric_both(tx, e, t, go, 9, 3, 0.5)
                assert_close(fwd, oracle.photometric_loss_forward(e, t, 9, 3, 0.5), what="quantised fwd")
                ob = oracle.photometric_loss_backward(e, t, go, 9, 3, 0.5)
                scale = max(float(np.abs(ob).max()), 1e-30)
                assert float(np.abs(bwd - ob).max()) <= 1e-5 * scale + 1e-12, "quantised bwd"
        finally:
            _lib.set_option("census_sym", 2)


TILE_SHAPES = [(1, 9, 12), (2, 16, 64), (1, 10, 72), (3, 21, 132), (1, 130, 200), (2, 61, 300), (1, 250, 48), (5, 40, 68),
               (2, 150, 280)]


@pytest.mark.parametrize("shape", TILE_SHAPES)
@pytest.mark.parametrize("ty", (2, 3))
def test_census_tile_kernel_vs_oracle(tx, shape, ty):
    """The census tile kernels of photometric.cu (census_sym = 0: every call) through all four entry points against the
    oracle, one launch each: images smaller than a 64 x 16 tile, ragged last tile column (width not a multiple of 64)
    and last tile row (height not a multiple of 16), widths that are / are not multiples of four, several images,
    every pixel of the smallest image ON the border."""
    B, H, W = shape
    rng = np.random.RandomState(H * 1000 + W + ty)
    es = rng.randn(B, 1, H, W).astype(np.float32)
    ta = (es + 0.6 * rng.randn(B, 1, H, W)).astype(np.float32)
    go = rng.randn(B, 1, H, W).astype(np.float32)
    mask = (rng.rand(B, 1, H, W) + 0.5).astype(np.float32)
    from connecting_the_dots_b200 import _lib
    _lib.set_option("census_sym", 0)
    try:
        n0 = _lib.launch_count()
        r = _census_all_entry_points(tx, es, ta, go, mask, ty)
        assert _lib.launch_count() - n0 == 4, "one kernel per entry point"
    finally:
        _lib.set_option("census_sym", 2)
    of, ob = oracle.photometric_loss_forward(es, ta, 9, ty, 0.5), oracle.photometric_loss_backward(es, ta, go, 9, ty, 0.5)
    for k in ("fwd", "f_fwd", "m_fwd"):
        assert_close(r[k], of, what=k)
    for k in ("bwd", "f_bwd", "m_bwd"):
        assert_close(r[k], ob, what=k)
    want = np.array([(mask.astype(np.float64) * of).sum(), mask.astype(np.float64).sum()])
    assert np.abs(r["sums"] - want).max() <= 1e-5 * np.abs(want).max()


def test_census_tile_kernel_exact_sign_decisions_and_determinism(tx):
    """The census tile kernels (census_sym = 0) on quantised images (many window terms exactly zero or equal up to
    rounding), a constant image (every pair a tie) and the bench frames, whose flat regions tie exactly: census_sad's
    sign() decisions have to be the reference's, and two runs have to agree bit for bit."""
    from connecting_the_dots_b200 import _lib, synth
    rng = np.random.RandomState(11)
    B, H, W = 2, 70, 120
    es = rng.randint(0, 3, (B, 1, H, W)).astype(np.float32)
    ta = rng.randint(0, 3, (B, 1, H, W)).astype(np.float32)
    go = rng.rand(B, 1, H, W).astype(np.float32)
    d = synth.make_batch(1, 96, 128)
    cases = [(es, ta, go), (es, es.copy(), go), (np.full_like(es, 0.25), np.full_like(es, 0.75), go), (d["es"], d["ta"], d["go"])]
    _lib.set_option("census_sym", 0)
    try:
        for e, t, g in cases:
            fwd, bwd = photometric_both(tx, e, t, g, 9, 3, 0.5)
            _, again = photometric_both(tx, e, t, g, 9, 3, 0.5)
            assert np.array_equal(bwd, again)
            ob = oracle.photometric_loss_backward(e, t, g, 9, 3, 0.5)
            scale = max(float(np.abs(ob).max()), 1e-30)
            assert float(np.abs(bwd - ob).max()) <= 1e-5 * scale + 1e-12, "quantised bwd"
    finally:
        _lib.set_option("census_sym", 2)


@pytest.mark.parametrize("shape", [(2, 1, 40, 72), (1, 2, 33, 50), (1, 1, 96, 160), (1, 1, 7, 9)])
@pytest.mark.parametrize("ty", range(4))
def test_photometric_fused_forward_backward(tx, shape, ty):
    """ctd_photometric_fwd_bwd_f32 (one fused kernel for the census modes) against the oracle's two passes."""
    B, C, H, W = shape
    rng = np.random.RandomState(B * 100 + W)
    es = rng.randn(B, C, H, W).astype(np.float32)
    ta = (es + 0.6 * rng.randn(B, C, H, W)).astype(np.float32)
    go = rng.randn(B, 1, H, W).astype(np.float32)
    out, gi = tx.ext_cuda.photometric_loss_forward_backward(cu(es), cu(ta), cu(go), 9, ty, 0.5)
    assert_close(out.cpu().numpy(), oracle.photometric_loss_forward(es, ta, 9, ty, 0.5), what="fused fwd")
    assert_close(gi.cpu().numpy(), oracle.photometric_loss_backward(es, ta, go, 9, ty, 0.5), what="fused bwd")


@pytest.mark.parametrize("shape", [(2, 1, 40, 72), (1, 2, 33, 50), (3, 1, 96, 160)])
@pytest.mark.parametrize("ty", range(4))
def test_photometric_fused_masked_sums(tx, shape, ty):
    """ctd_photometric_fwd_bwd_masked_f32: loss map, gradient and the masked-mean terms of one pass; run twice to
    check that the ticket counter resets and the sums are run-to-run identical."""
    B, C, H, W = shape
    rng = np.random.RandomState(B * 10 + ty)
    es = rng.randn(B, C, H, W).astype(np.float32)
    ta = (es + 0.6 * rng.randn(B, C, H, W)).astype(np.float32)
    go = rng.randn(B, 1, H, W).astype(np.float32)
    mask = rng.rand(B, 1, H, W).astype(np.float32)
    ref_out = oracle.photometric_loss_forward(es, ta, 9, ty, 0.5)
    res = [tx.ext_cuda.photometric_loss_forward_backward_masked(cu(es), cu(ta), cu(go), cu(mask), 9, ty, 0.5) for _ in range(2)]
    out, gi, sums = res[0]
    assert_close(out.cpu().numpy(), ref_out, what="fused fwd")
    assert_close(gi.cpu().numpy(), oracle.photometric_loss_backward(es, ta, go, 9, ty, 0.5), what="fused bwd")
    num, den = float((mask.astype(np.float64) * ref_out).sum()), float(mask.astype(np.float64).sum())
    assert abs(float(sums[0]) - num) <= 1e-5 * abs(num) and abs(float(sums[1]) - den) <= 1e-5 * den
    assert torch.equal(res[0][2], res[1][2])


@pytest.mark.parametrize("ty", (1, 3))
def test_weighted_photometric_loss_matches_composition(tx, ty):
    """The fused masked-mean op equals photometric_loss -> (mask*d).sum()/mask.sum() with autograd, value and gradient."""
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(2, 96, 160)
    es = cu(d["es"]).requires_grad_(True)
    ta, mask = cu(d["ta"]), cu(d["std"])
    ref = (mask * tx.photometric_loss(es, ta, 9, TYPES[ty], 0.5)).sum() / mask.sum()
    (gref,) = torch.autograd.grad(3.0 * ref, es)
    val, loss_map = tx.weighted_photometric_loss(es, ta, mask, 9, TYPES[ty], 0.5)
    (g,) = torch.autograd.grad(3.0 * val, es)
    assert abs(val.item() - ref.item()) <= 1e-5 * abs(ref.item())
    assert_close(g.cpu().numpy(), gref.cpu().numpy(), what="weighted loss gradient")
    assert_close(loss_map.cpu().numpy(), oracle.photometric_loss_forward(d["es"], d["ta"], 9, ty, 0.5), what="loss map")


@pytest.mark.parametrize("ty", (1, 3))
def test_photometric_full_size_synthetic(tx, ty):
    """BASELINE config 1/2 data: 480x640 LCN'd dot-pattern pairs, grad_out = std / sum(std)."""
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(2)
    eps = 0.5
    fwd, bwd = photometric_both(tx, d["es"], d["ta"], d["go"], 9, ty, eps)
    assert_close(fwd, oracle.photometric_loss_forward(d["es"], d["ta"], 9, ty, eps), what="fwd")
    assert_close(bwd, oracle.photometric_loss_backward(d["es"], d["ta"], d["go"], 9, ty, eps), what="bwd")


def test_photometric_backward_is_deterministic_and_linear(tx):
    """No atomics: two runs are bit-identical; the backward is linear in grad_out (size-independent
    property checked at the bench size, batch 8)."""
    torch.manual_seed(0)
    es = torch.randn(8, 1, 480, 640, device=DEV)
    ta = torch.randn(8, 1, 480, 640, device=DEV)
    g1 = torch.rand(8, 1, 480, 640, device=DEV)
    g2 = torch.rand(8, 1, 480, 640, device=DEV)
    for ty in (1, 3):
        a = tx.ext_cuda.photometric_loss_backward(es, ta, g1, 9, ty, 0.5)
        b = tx.ext_cuda.photometric_loss_backward(es, ta, g1, 9, ty, 0.5)
        assert torch.equal(a, b)
        c = tx.ext_cuda.photometric_loss_backward(es, ta, g2, 9, ty, 0.5)
        s = tx.ext_cuda.photometric_loss_backward(es, ta, g1 + g2, 9, ty, 0.5)
        assert_close((a + c).cpu().numpy(), s.cpu().numpy(), tol=2e-5, what="linearity")


@pytest.mark.parametrize("ty", range(4))
def test_photometric_matches_torch_restatement_and_autograd(tx, ty):
    """photometric_loss_pytorch (functions.py:120-147 counterpart) in fp64 with autograd is an
    independent second implementation of forward AND backward."""
    rng = np.random.RandomState(8)
    es = torch.from_numpy(rng.randn(1, 2, 21, 37)).to(DEV).requires_grad_(True)
    ta = torch.from_numpy(rng.randn(1, 2, 21, 37)).to(DEV)
    go = torch.from_numpy(rng.randn(1, 1, 21, 37)).to(DEV)
    ref = tx.photometric_loss_pytorch(es, ta, 9, TYPES[ty], 0.5)
    (gref,) = torch.autograd.grad(ref, es, go)
    out = tx.photometric_loss(es, ta, 9, TYPES[ty], 0.5)
    (g,) = torch.autograd.grad(out, es, go)
    assert_close(out.detach().cpu().numpy(), ref.detach().cpu().numpy(), tol=1e-10, what="fwd")
    assert_close(g.cpu().numpy(), gref.cpu().numpy(), tol=1e-9, what="bwd")


def test_photometric_empty_and_errors(tx):
    e = torch.zeros(0, 1, 16, 16, device=DEV)
    assert tx.photometric_loss(e, e, 9, "sad").shape == (0, 1, 16, 16)
    x = torch.randn(1, 1, 16, 16, device=DEV)
    with pytest.raises(Exception, match="invalid loss type"):
        tx.photometric_loss(x, x, 9, "ssim")
    with pytest.raises(RuntimeError):
        tx.photometric_loss(x.transpose(2, 3), x, 9, "sad")          # non-contiguous
    with pytest.raises(NotImplementedError):
        tx.photometric_loss(x.half(), x.half(), 9, "sad")
    with pytest.raises(RuntimeError):
        tx.photometric_loss(x.cpu(), x.cpu(), 9, "sad")              # no CPU path
    with pytest.raises(RuntimeError):
        tx.photometric_loss(x, x[:, :, :8].contiguous(), 9, "sad")   # shape mismatch
    assert tx.photometric_loss(x, x, 9, "MSE").abs().max().item() == 0  # case-insensitive type


# ---------------------------------------------------------------- LCN
@pytest.mark.parametrize("r,e", ((5, 0.05), (2, 0.1)))
def test_lcn_golden(tx, golden, r, e):
    """vs the reference torch module: same bound as the oracle's own test (the reference's fp32 conv
    summation order is unspecified and var cancels on flat regions)."""
    g = golden("lcn")
    l, s = tx.lcn(cu(g["x"]), r, e)
    l, s = l.cpu().numpy(), s.cpu().numpy()
    assert np.abs(s - g[f"r{r}_std"]).max() <= 2e-4 * np.abs(g[f"r{r}_std"]).max()
    assert np.abs(l - g[f"r{r}_lcn"]).max() <= 2e-4 * np.abs(g[f"r{r}_lcn"]).max()
    lo, so = oracle.lcn(g["x"], r, e)
    assert_close(l, lo, what="lcn vs oracle")
    assert_close(s, so, what="std vs oracle")


@pytest.mark.parametrize("shape", [(1, 480, 640, 5), (3, 37, 130, 5), (2, 16, 12, 3), (1, 61, 259, 7), (1, 40, 40, 17),
                                   (1, 6, 6, 5), (2, 100, 128, 0), (1, 9, 1000, 2), (1, 20, 32, 5), (2, 20, 132, 5)])
def test_lcn_vs_oracle(tx, shape):
    N, H, W, r = shape
    rng = np.random.RandomState(N * 7 + H)
    x = rng.rand(N, 1, H, W).astype(np.float32)
    x[0, 0, : H // 2, : W // 2] = 0.5   # flat region: var collapses to the 1e-6 floor
    l, s = tx.lcn(cu(x), r, 0.05)
    lo, so = oracle.lcn(x, r, 0.05)
    assert_close(l.cpu().numpy(), lo, what="lcn")
    assert_close(s.cpu().numpy(), so, what="std")
    mod = tx.LCN(r, 0.05)
    l2, s2 = mod(cu(x))
    assert torch.equal(l2, l) and torch.equal(s2, s)


def _lcn_reference_recipe(x, r, e):
    """model/networks.py:523-533 restated with the same torch ops (on whatever device x lives)."""
    k = 2 * r + 1
    w = torch.ones(1, 1, k, k, device=x.device, dtype=x.dtype)
    pad = torch.nn.functional.pad(x, (r,) * 4, mode="reflect")
    box, box2 = torch.nn.functional.conv2d(pad, w), torch.nn.functional.conv2d(pad * pad, w)
    avg = box / k ** 2
    std = torch.sqrt(box2 / k ** 2 - avg ** 2 + 1e-6) + e
    return (x - avg) / std, std


def test_lcn_vs_reference_recipe_on_baseline_frames(tx):
    """The kernel against the reference's own LCN recipe (networks.py:523-533) evaluated by torch on the CPU and on this
    GPU (TF32 off), and all three against the same recipe in float64, on 8 BASELINE synthetic frames (480x640).
    Measured (recorded by the print below): the two fp32 reference evaluations differ from each other by ~3e-5 and from
    the float64 value by ~1e-4 in `std`, all of it on the ~2 % of windows that are flat (image clipped at 0 / 1), where
    var = E[x^2] - avg^2 cancels to fp32 rounding noise above the 1e-6 floor.  Asserted:
      * on every window with raw std > 0.02 (97.7 % of the pixels) the kernel matches BOTH reference evaluations to the
        north-star 1e-5, lcn and std;
      * everywhere, the kernel is closer to the float64 value than either fp32 reference evaluation is (exact box sums),
        and within 2e-4 of both (the bound the formula allows, test_lcn_golden)."""
    from connecting_the_dots_b200 import synth
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    x = torch.from_numpy(synth.make_batch(8)["im"])
    lc, sc = _lcn_reference_recipe(x, 5, 0.05)
    lg, sg = (t.cpu() for t in _lcn_reference_recipe(x.to(DEV), 5, 0.05))
    l64, s64 = _lcn_reference_recipe(x.double(), 5, 0.05)
    l, s = (t.cpu() for t in tx.lcn(x.to(DEV), 5, 0.05))
    textured = (s64 - 0.05) > 0.02

    def rel(a, b, where=None):
        d = (a.double() - b.double()).abs()
        if where is not None:
            d = d[where]
        return float(d.max() / b.double().abs().max())

    rows = {"ref cpu-vs-cuda": (rel(lg, lc), rel(sg, sc)), "ref cpu vs f64": (rel(lc, l64), rel(sc, s64)),
            "ref cuda vs f64": (rel(lg, l64), rel(sg, s64)), "kernel vs f64": (rel(l, l64), rel(s, s64)),
            "kernel vs ref cpu": (rel(l, lc), rel(s, sc)), "kernel vs ref cuda": (rel(l, lg), rel(s, sg)),
            "kernel vs ref cpu, textured": (rel(l, lc, textured), rel(s, sc, textured)),
            "kernel vs ref cuda, textured": (rel(l, lg, textured), rel(s, sg, textured))}
    print("LCN on BASELINE frames (lcn, std), textured fraction %.4f: " % float(textured.float().mean())
          + "; ".join("%s %.2e %.2e" % (k, *v) for k, v in rows.items()))
    assert float(textured.float().mean()) > 0.95
    for k in ("kernel vs ref cpu, textured", "kernel vs ref cuda, textured"):
        assert max(rows[k]) <= 1e-5, (k, rows[k])
    for q in (0, 1):
        assert rows["kernel vs f64"][q] <= 1.2 * min(rows["ref cpu vs f64"][q], rows["ref cuda vs f64"][q]) + 1e-6, rows
        assert max(rows["kernel vs ref cpu"][q], rows["kernel vs ref cuda"][q]) <= 2e-4, rows


def test_lcn_reference_disagrees_with_itself_on_flat_fixture(tx, golden):
    """The 2e-4 bound of test_lcn_golden is the reference's own: on the golden fixture (which contains an exactly flat
    region, var = 1e-6 floor after cancellation) torch-on-CPU and torch-on-CUDA evaluations of networks.py:523-533 are
    compared with each other; the kernel must be no further from either than 2e-4 and the fixture's two reference
    evaluations are reported."""
    torch.backends.cudnn.allow_tf32 = False
    g = golden("lcn")
    x = torch.from_numpy(g["x"])
    lc, sc = _lcn_reference_recipe(x, 5, 0.05)
    lg, sg = _lcn_reference_recipe(x.to(DEV), 5, 0.05)
    rel = lambda a, b: float((a.double().cpu() - b.double().cpu()).abs().max() / b.double().abs().max())
    print("LCN golden fixture: reference cpu-vs-cuda lcn %.2e std %.2e" % (rel(lg, lc), rel(sg, sc)))
    l, s = tx.lcn(x.to(DEV), 5, 0.05)
    for ref_l, ref_s in ((lc, sc), (lg, sg)):
        assert rel(l, ref_l) <= 2e-4 and rel(s, ref_s) <= 2e-4
    # the committed golden came from the reference's own class on CPU torch: same numbers as the recipe above
    assert rel(lc, torch.from_numpy(g["r5_lcn"])) <= 1e-6


def test_lcn_normalize_matches_reference_cython_build(tx, golden):
    """torchext.lcn_normalize = data/lcn/lcn.pyx normalize (the data generator's offline LCN): bit-identical to the
    reference's Cython build on the golden inputs, and to the oracle on a 480x640 frame, single and batched."""
    g = golden("lcn_cython")
    for n in "abcde":
        ks, eps = g[n + "_args"]
        l, s = tx.lcn_normalize(cu(g[n + "_x"]), int(ks), float(eps))
        assert np.array_equal(l.cpu().numpy(), g[n + "_lcn"]) and np.array_equal(s.cpu().numpy(), g[n + "_std"]), n
    from connecting_the_dots_b200 import synth
    im = synth.make_batch(2)["im"][:, 0]
    l, s = tx.lcn_normalize(cu(im), 5, 0.1)          # create_syn_data.py:182 arguments
    for b in range(2):
        lo, so = oracle.lcn_cython(im[b], 5, 0.1)
        assert np.array_equal(l[b].cpu().numpy(), lo) and np.array_equal(s[b].cpu().numpy(), so)
    with pytest.raises(RuntimeError):
        tx.lcn_normalize(torch.rand(8, 8), 2, 0.1)   # no CPU path


@pytest.mark.parametrize("shape", [(2, 40, 70, 5), (1, 16, 16, 5), (1, 33, 45, 2), (1, 480, 640, 5), (2, 12, 9, 8)])
def test_lcn_backward_matches_autograd_of_reference_recipe(tx, shape):
    """d loss / d x of networks.LCN for upstream gradients of BOTH outputs, against torch autograd through the reference's
    own recipe (networks.py:523-533) in float64; reflection-padded borders, mirrored windows from both sides on small images."""
    N, H, W, r = shape
    g = torch.Generator(device="cpu").manual_seed(H * W)
    x = torch.rand(N, 1, H, W, generator=g)
    gl, gs = torch.randn(N, 1, H, W, generator=g), torch.randn(N, 1, H, W, generator=g)
    xd = x.double().requires_grad_(True)
    l64, s64 = _lcn_reference_recipe(xd, r, 0.05)
    (ref,) = torch.autograd.grad((l64 * gl.double()).sum() + (s64 * gs.double()).sum(), xd)
    xg = x.to(DEV).requires_grad_(True)
    l, s = tx.lcn(xg, r, 0.05)
    (got,) = torch.autograd.grad((l * gl.to(DEV)).sum() + (s * gs.to(DEV)).sum(), xg)
    assert_close(got.cpu().numpy(), ref.numpy(), tol=2e-5, what="lcn backward")
    (got_l,) = torch.autograd.grad(tx.lcn(xg, r, 0.05)[0].mul(gl.to(DEV)).sum(), xg)     # only one output used
    (ref_l,) = torch.autograd.grad((_lcn_reference_recipe(xd, r, 0.05)[0] * gl.double()).sum(), xd)
    assert_close(got_l.cpu().numpy(), ref_l.numpy(), tol=2e-5, what="lcn backward, lcn output only")


def test_lcn_f64_and_errors(tx):
    rng = np.random.RandomState(2)
    x = rng.rand(2, 1, 30, 50)
    l, s = tx.lcn(cu(x), 5, 0.05)
    lo, so = oracle.lcn(x, 5, 0.05)
    assert_close(l.cpu().numpy(), lo, tol=1e-12)
    assert_close(s.cpu().numpy(), so, tol=1e-12)
    with pytest.raises(RuntimeError):
        tx.lcn(torch.rand(1, 1, 4, 40, device=DEV), 5, 0.05)   # radius >= height: ReflectionPad2d refuses too
    with pytest.raises(RuntimeError):
        tx.lcn(torch.rand(1, 2, 40, 40, device=DEV), 5, 0.05)  # single channel only (networks.py:514)


# ---------------------------------------------------------------- xcorrvol
def test_xcorrvol_golden(tx, golden):
    g = golden("xcorrvol")
    for k in [k[:-4] for k in g.files if k.endswith("_in0")]:
        D = int(k.split("_D")[1].split("_")[0])
        bs = int(k.split("_bs")[1])
        got = tx.xcorrvol(cu(g[k + "_in0"]), cu(g[k + "_in1"]), D, bs)
        assert_close(got.cpu().numpy(), g[k + "_out"], what=k)
    flat = np.full((1, 6, 8), 0.25, np.float32)
    assert_close(tx.xcorrvol(cu(flat), cu(flat), 3, 3).cpu().numpy() + 1, g["flat_out"] + 1, what="flat")
    assert_close(tx.xcorrvol(cu(g["self_in"]), cu(g["self_in"]), 1, 3).cpu().numpy(), g["self_out"], what="self")


@pytest.mark.parametrize("shape", [(1, 1, 40, 150, 32, 9), (2, 1, 24, 70, 17, 9), (1, 2, 20, 40, 8, 5), (1, 1, 9, 33, 40, 9),
                                   (1, 1, 30, 64, 5, 3), (1, 3, 12, 20, 4, 2)])
def test_xcorrvol_vs_oracle(tx, shape):
    B, C, H, W, D, bs = shape
    rng = np.random.RandomState(D)
    a = rng.randn(B, C, H, W).astype(np.float32)
    b = (np.roll(a, 3, axis=3) + 0.3 * rng.randn(B, C, H, W)).astype(np.float32)
    got = tx.xcorrvol(cu(a), cu(b), D, bs).cpu().numpy()
    assert got.shape == (B, D, H, W)
    for i in range(B):
        assert_close(got[i], oracle.xcorrvol(a[i], b[i], D, bs), what="batched image %d" % i)
    one = tx.xcorrvol(cu(a[0]), cu(b[0]), D, bs).cpu().numpy()  # the reference's 3-D signature
    assert one.shape == (D, H, W)
    assert np.array_equal(one, got[0])


def test_xcorrvol_ill_conditioned_windows(tx):
    """Windows whose mean dominates their spread (raw intensities, constant patches, one flat image): the
    separable kernel must hand them to its centred two-pass path and still match ext_cpu's arithmetic."""
    rng = np.random.RandomState(7)
    H, W, D = 40, 132, 21
    a = (0.5 + 0.02 * rng.randn(1, 1, H, W)).astype(np.float32)
    b = (0.5 + 0.02 * rng.randn(1, 1, H, W)).astype(np.float32)
    a[0, 0, 5:25, 30:70] = 0.75                      # flat patch inside a textured image
    b[0, 0, 10:30, 80:120] = rng.randn(20, 40)       # well-conditioned island in a dim image
    got = tx.xcorrvol(cu(a), cu(b), D, 9).cpu().numpy()
    assert_close(got[0], oracle.xcorrvol(a[0], b[0], D, 9), what="raw intensities + flat patch")
    z = rng.randn(1, 1, H, W).astype(np.float32)
    z[0, 0, :, 40:90] = 0.0                          # exactly zero band: sigma = 0, norm = 1e-8
    got = tx.xcorrvol(cu(z), cu(np.roll(z, 2, axis=3)), D, 5).cpu().numpy()
    assert_close(got[0], oracle.xcorrvol(z[0], np.roll(z, 2, axis=3)[0], D, 5), what="zero band")


def test_xcorrvol_fixup_overflow_path(tx):
    """The fix-up lists untrusted outputs in a bounded hit list; with the list forced to size 0 the in-place
    fallback kernel must produce exactly the same volume."""
    from connecting_the_dots_b200 import _lib
    rng = np.random.RandomState(11)
    H, W, D = 40, 132, 21
    a = (0.5 + 0.02 * rng.randn(2, 1, H, W)).astype(np.float32)
    b = (0.5 + 0.02 * rng.randn(2, 1, H, W)).astype(np.float32)
    a[1, 0, 5:25, 30:70] = 0.75
    listed = tx.xcorrvol(cu(a), cu(b), D, 9)
    _lib.set_option("xcorr_hitcap", 0)
    try:
        inplace = tx.xcorrvol(cu(a), cu(b), D, 9)
    finally:
        _lib.set_option("xcorr_hitcap", -1)
    assert torch.equal(listed, inplace)
    for n in range(2):
        assert_close(listed[n].cpu().numpy(), oracle.xcorrvol(a[n], b[n], D, 9), what="raw intensities image %d" % n)


def test_xcorrvol_separable_matches_direct(tx):
    """A/B: the separable kernel against the direct centred kernel of the same library on LCN'd data."""
    from connecting_the_dots_b200 import _lib, synth
    d = synth.make_pair(1, 64, 320)
    a, b = cu(d["ta"][None]), cu(d["pat_lcn"][None])
    fast = tx.xcorrvol(a, b, 128, 9)
    _lib.set_option("xcorr_direct", 1)
    try:
        direct = tx.xcorrvol(a, b, 128, 9)
    finally:
        _lib.set_option("xcorr_direct", 0)
    assert_close(fast.cpu().numpy(), direct.cpu().numpy(), what="separable vs direct")


def test_xcorrvol_full_size_properties(tx):
    """BASELINE config 3 size (480x640, D=128, block 9), checked through size-independent properties: the volume is a
    correlation coefficient (|.| <= 1), an image against itself scores 1 at d = 0, against a copy shifted by s pixels
    it scores 1 at d = s, and batching does not change any image's result."""
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(2)
    a = cu(d["ta"])
    s = 37
    b = torch.roll(a, -s, dims=3)  # b[x] = a[x + s]  ->  b[w - s] = a[w]
    vol = tx.xcorrvol(a, b, 128, 9)
    assert vol.shape == (2, 128, 480, 640)
    assert float(vol.abs().max()) <= 1 + 1e-5
    assert float((vol[:, s, :, s + 8:640 - s - 8] - 1).abs().max()) <= 1e-5
    self_vol = tx.xcorrvol(a, a, 4, 9)
    assert float((self_vol[:, 0] - 1).abs().max()) <= 1e-5
    one = tx.xcorrvol(a[1], b[1], 128, 9)
    assert torch.equal(one, vol[1])


@pytest.mark.parametrize("bs", (9, 5))
def test_xcorrvol_full_size_golden(tx, golden, bs):
    """BASELINE configs[2] at its own size against the UNMODIFIED reference: 480x640, D = 128, the batched B = 8 call;
    image 0 is compared with the rows and columns of the reference's volume kept in tests/golden/xcorrvol_full.npz
    (tests/golden/make_golden_full.py: oracle/_ref xcorrvol_cpu on the same synthetic LCN'd pair)."""
    from connecting_the_dots_b200 import synth
    g = golden("xcorrvol_full")
    d = synth.make_batch(8)
    in0, in1 = d["ta"], d["pat_lcn"]
    # the fixture was made from the same seeded inputs
    assert np.array_equal(in0[0, 0, 240], g["in0_row240"]) and np.array_equal(in1[0, 0, 240], g["in1_row240"])
    assert float(in0[0].astype(np.float64).sum()) == float(g["in0_sum"])
    vol = tx.xcorrvol(cu(in0), cu(in1), 128, bs)
    assert vol.shape == (8, 128, 480, 640)
    rows, cols = torch.from_numpy(g["rows"]).to(DEV), torch.from_numpy(g["cols"]).to(DEV)
    got = vol[0].index_select(1, rows).index_select(2, cols).cpu().numpy()
    assert_close(got, g["bs%d" % bs], what="xcorrvol 480x640 D128 bs%d vs reference" % bs)
    one = tx.xcorrvol(cu(in0[0]), cu(in1[0]), 128, bs)   # the reference's unbatched 3-D signature, same result
    assert torch.equal(one, vol[0])


def test_xcorrvol_fork_join_matches_serial_and_is_capturable(tx):
    """The call forks inside (the two statistics passes side by side, the sweep beside the main kernel) and joins before
    the hits are evaluated: same volume as with every kernel on the caller's stream, on a non-default stream, and when
    the call is captured into a CUDA graph and replayed."""
    from connecting_the_dots_b200 import _lib, synth
    d = synth.make_batch(2, 96, 256)
    a, b = cu(d["ta"]), cu(d["pat_lcn"])
    _lib.set_option("xcorr_serial", 1)
    try:
        ref = tx.xcorrvol(a, b, 48, 9)
    finally:
        _lib.set_option("xcorr_serial", 0)
    assert torch.equal(tx.xcorrvol(a, b, 48, 9), ref)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        on_s = tx.xcorrvol(a, b, 48, 9)
    s.synchronize()
    assert torch.equal(on_s, ref)
    out = torch.zeros_like(ref)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _lib.call("ctd_xcorrvol_f32", a.data_ptr(), b.data_ptr(), out.data_ptr(), 2, 1, 96, 256, 48, 9, torch.cuda.current_stream().cuda_stream)
    for _ in range(3):
        out.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, ref)


def test_xcorrvol_synthetic_lcn_data(tx):
    """LCN'd dot-pattern rows (the BASELINE config 3 data) on a crop the oracle finishes quickly."""
    from connecting_the_dots_b200 import synth
    d = synth.make_pair(0, 96, 256)
    a, b = d["ta"][None], d["pat_lcn"][None]
    got = tx.xcorrvol(cu(a), cu(b), 48, 9).cpu().numpy()
    assert_close(got, oracle.xcorrvol(a, b, 48, 9), what="lcn crop")


# ---------------------------------------------------------------- proj_nn / nn / crosscheck: bit-exact
@pytest.mark.parametrize("ps", (1, 2, 3, 5, 9))
def test_proj_nn_golden(tx, golden, ps):
    g = golden("proj_nn")
    got = tx.proj_nn(cu(g["xyz0"]), cu(g["xyz1"]), cu(g["K"]), ps)
    assert got.dtype == torch.int64
    assert np.array_equal(got.cpu().numpy(), g[f"ps{ps}"])


@pytest.mark.parametrize("dt", (np.float32, np.float64))
def test_proj_nn_vs_oracle(tx, dt):
    from connecting_the_dots_b200 import synth
    xyz, K, poses = synth.make_clouds(3, 120, 160, seed=3)
    K = K.astype(dt)
    for ps in (3, 5):
        for i, j in ((0, 1), (1, 2), (2, 0)):
            x0 = synth.transform(xyz[i], poses[j]).astype(dt)[None]
            x1 = xyz[j].astype(dt)[None]
            x0[0, 0, :4] = [[1, 1, 0], [0, 0, 0], [np.nan, 1, 1], [1e30, 1, 1e-8]]
            got = tx.proj_nn(cu(x0), cu(x1), cu(K), ps).cpu().numpy()
            want = oracle.proj_nn(x0, x1, K, ps)
            assert np.array_equal(got, want)
            assert (want >= 0).mean() > 0.5
    xb = np.stack([xyz[0], xyz[1]]).astype(dt)
    got = tx.proj_nn(cu(xb), cu(xb[::-1].copy()), cu(K), 3).cpu().numpy()   # batch offset in the flat index
    assert np.array_equal(got, oracle.proj_nn(xb, xb[::-1].copy(), K, 3))


@pytest.mark.parametrize("ps", (1, 2, 3, 5, 7, 9))
def test_proj_nn_fixed_kernel_vs_oracle(tx, ps):
    """The fixed-patch row kernel against the oracle on a ragged image size: smooth geometry, wild geometry (projections
    all over the image, NaN, zero depth, points behind the camera) and queries that all miss the image."""
    from connecting_the_dots_b200 import synth
    xyz, K, poses = synth.make_clouds(2, 61, 83, seed=3)
    cases = [(synth.transform(xyz[0], poses[1])[None], xyz[1][None], K)]
    rng = np.random.RandomState(ps)
    wild0 = (xyz[0] * rng.uniform(0.2, 3.0, xyz[0].shape)).astype(np.float32)[None]      # projections scattered
    wild0[0, 5, 7] = [np.nan, 1, 1]
    wild0[0, 6, 7] = [1, 1, 0]
    wild0[0, 40:, :40] *= np.float32(-1.0)                                                # behind the camera: still valid indices
    cases.append((wild0, xyz[1][None], K))
    far = (xyz[0] + np.float32([5.0, 0, 0]))[None]                                        # everything projects outside
    cases.append((far.astype(np.float32), xyz[1][None], K))
    for x0, x1, K_ in cases:
        got = tx.proj_nn(cu(x0), cu(x1), cu(K_), ps).cpu().numpy()
        assert np.array_equal(got, oracle.proj_nn(x0, x1, K_, ps))


def test_nn_golden_and_split(tx, golden):
    g = golden("nn")
    assert np.array_equal(tx.nn(cu(g["p0"]), cu(g["p1"])).cpu().numpy(), g["idx"])
    assert np.array_equal(tx.nn(cu(g["p0"][:5]), cu(g["p1"][:0].reshape(0, 3))).cpu().numpy(), g["idx_empty"])
    rng = np.random.RandomState(21)
    for n0, n1, dt in ((1000, 5000, np.float32), (777, 4099, np.float32), (300, 2500, np.float64), (5000, 300, np.float32)):
        p0 = rng.randn(n0, 3).astype(dt)
        p1 = rng.randn(n1, 3).astype(dt)
        p1[n1 // 2:] = p1[: n1 - n1 // 2]          # every point twice: ties across in1 chunks -> lowest index
        p0[3] = [np.nan, 0, 0]
        p0[4] = [4e4, 0, 0]
        assert np.array_equal(tx.nn(cu(p0), cu(p1)).cpu().numpy(), oracle.nn(p0, p1)), (n0, n1, dt)


def test_crosscheck(tx, golden):
    g = golden("crosscheck")
    got = tx.crosscheck(cu(g["in0"]), cu(g["in1"]))
    assert got.dtype == torch.uint8
    assert np.array_equal(got.cpu().numpy(), g["out"])
    assert tx.crosscheck(cu(g["kat_in0"]), cu(g["kat_in1"])).cpu().tolist() == [1, 1, 0, 0, 0]
    rng = np.random.RandomState(4)
    for n in (1, 3, 1001, 307200):
        perm = rng.permutation(n).astype(np.int64)
        inv = np.empty(n, np.int64)
        inv[perm] = np.arange(n)
        perm[rng.rand(n) < 0.1] = -1
        inv[rng.rand(n) < 0.1] = rng.randint(-1, n)
        assert np.array_equal(tx.crosscheck(cu(perm), cu(inv)).cpu().numpy(), oracle.crosscheck(perm, inv))
        assert np.array_equal(tx.crosscheck(cu(perm[1:]), cu(inv)).cpu().numpy(), oracle.crosscheck(perm[1:], inv))
    wide = np.array([2**32 + 1, 1], np.int64)   # int64 -> int32 truncation of the index (ext.h:59)
    back = np.array([5, 0], np.int64)
    assert np.array_equal(tx.crosscheck(cu(wide), cu(back)).cpu().numpy(), oracle.crosscheck(wide, back))
    with pytest.raises(RuntimeError):
        tx.crosscheck(cu(perm).view(1, -1), cu(inv))


def test_geometric_step_composition(tx):
    """BASELINE config 4 as composed in SURVEY.md section 8d: for a 4-frame track, proj_nn both ways
    for each frame pair + crosscheck both ways; checked bit-exact against the oracle."""
    from connecting_the_dots_b200 import synth
    xyz, K, poses = synth.make_clouds(4, 60, 80, seed=1)
    Kd = cu(K)
    for i in range(4):
        for j in range(i + 1, 4):
            xij, xji = synth.transform(xyz[i], poses[j])[None], synth.transform(xyz[j], poses[i])[None]
            i01 = tx.proj_nn(cu(xij), cu(xyz[j][None]), Kd, 3)
            i10 = tx.proj_nn(cu(xji), cu(xyz[i][None]), Kd, 3)
            m01 = tx.crosscheck(i01.view(-1), i10.view(-1))
            m10 = tx.crosscheck(i10.view(-1), i01.view(-1))
            o01, o10 = oracle.proj_nn(xij, xyz[j][None], K, 3), oracle.proj_nn(xji, xyz[i][None], K, 3)
            assert np.array_equal(i01.cpu().numpy(), o01) and np.array_equal(i10.cpu().numpy(), o10)
            assert np.array_equal(m01.cpu().numpy(), oracle.crosscheck(o01.ravel(), o10.ravel()))
            assert np.array_equal(m10.cpu().numpy(), oracle.crosscheck(o10.ravel(), o01.ravel()))


def test_geometric_step_full_size(tx):
    """BASELINE configs[3] at its stated size: a 4-frame track at 480x640 -- ProjNN (patch 3) in both directions for the
    6 frame pairs as ONE batched launch of 12 queries, CrossCheck in both directions, and PhotometricLoss census_sad
    forward + backward on the 4 frames.  Indices and masks bit-exact, loss and gradient within 1e-5 of the oracle."""
    from connecting_the_dots_b200 import synth
    T, H, W = 4, 480, 640
    xyz, K, poses = synth.make_clouds(T, H, W)
    pairs = [(i, j) for i in range(T) for j in range(T) if i != j]
    rev = [pairs.index((j, i)) for i, j in pairs]
    x0 = np.stack([synth.transform(xyz[i], poses[j]) for i, j in pairs])
    x1 = np.stack([xyz[j] for i, j in pairs])
    idx = tx.proj_nn(cu(x0), cu(x1), cu(K), 3)
    o_idx = oracle.proj_nn(x0, x1, K, 3)
    assert np.array_equal(idx.cpu().numpy(), o_idx)
    assert (o_idx >= 0).mean() > 0.5   # the synthetic track overlaps: the test is not vacuous
    # CrossCheck pair p against its reverse pair, on per-image (shard-local) flat indices as the reference would see them
    hw = H * W
    loc = idx.view(len(pairs), -1) - (torch.arange(len(pairs), device=DEV) * hw).view(-1, 1)
    loc = torch.where(idx.view(len(pairs), -1) >= 0, loc, idx.view(len(pairs), -1))
    o_loc = np.where(o_idx.reshape(len(pairs), -1) >= 0, o_idx.reshape(len(pairs), -1) - (np.arange(len(pairs)) * hw)[:, None], -1)
    n_mutual = 0
    for p, q in enumerate(rev):
        m = tx.crosscheck(loc[p].contiguous(), loc[q].contiguous())
        om = oracle.crosscheck(o_loc[p], o_loc[q])
        assert np.array_equal(m.cpu().numpy(), om)
        n_mutual += int(om.sum())
    assert n_mutual > 0
    d = synth.make_batch(T, H, W)
    fwd, bwd = photometric_both(tx, d["es"], d["ta"], d["go"], 9, 3, 0.5)
    assert_close(fwd, oracle.photometric_loss_forward(d["es"], d["ta"], 9, 3, 0.5), what="census_sad fwd, 4 frames")
    assert_close(bwd, oracle.photometric_loss_backward(d["es"], d["ta"], d["go"], 9, 3, 0.5), what="census_sad bwd, 4 frames")


# ---------------------------------------------------------------- host-buffer C ABI
def test_host_api(golden):
    from connecting_the_dots_b200 import _lib
    L = _lib.lib()
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    rng = np.random.RandomState(12)
    es = rng.randn(2, 1, 40, 72).astype(np.float32)
    ta = rng.randn(2, 1, 40, 72).astype(np.float32)
    go = rng.rand(2, 1, 40, 72).astype(np.float32)
    out, gi = np.empty_like(go), np.empty_like(es)
    _lib.call("ctd_host_photometric_fwd_bwd_f32", P(es), P(ta), P(go), P(out), P(gi), 2, 1, 40, 72, 9, 3, 0.5)
    assert_close(out, oracle.photometric_loss_forward(es, ta, 9, 3, 0.5))
    assert_close(gi, oracle.photometric_loss_backward(es, ta, go, 9, 3, 0.5))
    out2 = np.empty_like(go)
    _lib.call("ctd_host_photometric_fwd_f32", P(es), P(ta), P(out2), 2, 1, 40, 72, 9, 3, 0.5)
    assert_close(out2, out, tol=2e-6)   # forward-only call: pair-symmetric kernel, fused call: gather kernel (other summation order)
    l, s = np.empty_like(es), np.empty_like(es)
    _lib.call("ctd_host_lcn_f32", P(es), P(l), P(s), 2, 40, 72, 5, 0.05)
    lo, so = oracle.lcn(es, 5, 0.05)
    assert_close(l, lo)
    assert_close(s, so)
    g = golden("proj_nn")
    idx = np.empty(g["ps3"].shape, np.int64)
    B, H, W, _ = g["xyz0"].shape
    _lib.call("ctd_host_proj_nn_f32", P(g["xyz0"]), P(g["xyz1"]), P(g["K"]), P(idx), B, H, W, 3)
    assert np.array_equal(idx, g["ps3"])
    g = golden("nn")
    idx = np.empty(len(g["p0"]), np.int64)
    _lib.call("ctd_host_nn_f32", P(g["p0"]), P(g["p1"]), P(idx), len(g["p0"]), len(g["p1"]))
    assert np.array_equal(idx, g["idx"])
    g = golden("crosscheck")
    m = np.empty(len(g["in0"]), np.uint8)
    _lib.call("ctd_host_crosscheck", P(g["in0"]), P(g["in1"]), P(m), len(g["in0"]), len(g["in1"]))
    assert np.array_equal(m, g["out"])
    g = golden("xcorrvol")
    k = "C1_H10_W24_D6_bs9"
    vol = np.empty_like(g[k + "_out"])
    _lib.call("ctd_host_xcorrvol_f32", P(g[k + "_in0"]), P(g[k + "_in1"]), P(vol), 1, 1, 10, 24, 6, 9)
    assert_close(vol, g[k + "_out"])
    with pytest.raises(_lib.CtdError, match="invalid loss type"):
        _lib.call("ctd_host_photometric_fwd_f32", P(es), P(ta), P(out2), 2, 1, 40, 72, 9, 7, 0.5)
    assert _lib.launch_count() > 0
    L.ctd_host_release()


def test_runs_on_current_stream_and_device(tx):
    """Launches go to torch's current stream (the reference uses the legacy default stream)."""
    x = torch.randn(2, 1, 64, 64, device=DEV)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        y = x * 2                      # produced on s; the op below must be ordered after it on s
        out = tx.photometric_loss(y, x, 9, "sad")
    s.synchronize()
    assert_close(out.cpu().numpy(), oracle.photometric_loss_forward((x * 2).cpu().numpy(), x.cpu().numpy(), 9, 1, 0.1))


def test_masked_sums(tx):
    """(mask*diff).sum() and mask.sum() of model/networks.py:377 in one deterministic kernel."""
    rng = np.random.RandomState(6)
    for n in (1, 5, 4096, 8 * 480 * 640, 1000003):
        d = rng.rand(n).astype(np.float32)
        m = rng.rand(n).astype(np.float32)
        a = tx.masked_mean_terms(cu(d), cu(m))
        b = tx.masked_mean_terms(cu(d), cu(m))
        assert torch.equal(a, b)
        want = np.array([(m.astype(np.float64) * d).sum(), m.astype(np.float64).sum()])
        assert np.abs(a.cpu().numpy() - want).max() <= 2e-6 * want.max()


@pytest.mark.parametrize("ty", (0, 1))
def test_box_tma_path_matches_tile_path(tx, ty):
    """mse/sad at C=1 run persistent TMA kernels (multi-iteration ring at batch 8); the shared-memory tile
    kernels (disable_tma) are a second implementation of the same arithmetic."""
    from connecting_the_dots_b200 import _lib
    torch.manual_seed(ty)
    for shape in ((8, 1, 480, 640), (3, 1, 50, 260), (1, 1, 300, 12)):
        es = torch.randn(*shape, device=DEV)
        ta = torch.randn(*shape, device=DEV)
        go = torch.rand(shape[0], 1, *shape[2:], device=DEV)
        f1 = tx.ext_cuda.photometric_loss_forward(es, ta, 9, ty, 0.1)
        b1 = tx.ext_cuda.photometric_loss_backward(es, ta, go, 9, ty, 0.1)
        _lib.set_option("disable_tma", 1)
        try:
            f2 = tx.ext_cuda.photometric_loss_forward(es, ta, 9, ty, 0.1)
            b2 = tx.ext_cuda.photometric_loss_backward(es, ta, go, 9, ty, 0.1)
        finally:
            _lib.set_option("disable_tma", 0)
        assert_close(f1.cpu().numpy(), f2.cpu().numpy(), what="fwd %s" % (shape,))
        assert_close(b1.cpu().numpy(), b2.cpu().numpy(), what="bwd %s" % (shape,))
    # and against the oracle on one full-size image
    es, ta, go = (t[:1].cpu().numpy() for t in (es, ta, go))
    es = np.ascontiguousarray(es); ta = np.ascontiguousarray(ta); go = np.ascontiguousarray(go)
    f = tx.ext_cuda.photometric_loss_forward(cu(es), cu(ta), 9, ty, 0.1).cpu().numpy()
    assert_close(f, oracle.photometric_loss_forward(es, ta, 9, ty, 0.1))


def test_host_api_deferred_batch_matches_synchronous_calls(tx):
    """ctd_host_begin_batch / ctd_host_end_batch: the same calls, enqueued back to back, give the same bytes."""
    from connecting_the_dots_b200 import _lib, synth
    d = synth.make_batch(3, 64, 96)
    P = lambda a: ctypes.c_void_p(a.ctypes.data)
    B, H, W = 3, 64, 96
    res = []
    for deferred in (False, True):
        lcn, std = np.empty_like(d["im"]), np.empty_like(d["im"])
        o1, g1, o3, g3 = (np.empty_like(d["es"]) for _ in range(4))
        idx = np.empty((B, H, W), np.int64)
        xyz, K, poses = synth.make_clouds(B, H, W)
        xyz = np.ascontiguousarray(xyz)
        if deferred:
            _lib.call("ctd_host_begin_batch")
        _lib.call("ctd_host_lcn_f32", P(d["im"]), P(lcn), P(std), B, H, W, 5, 0.05)
        _lib.call("ctd_host_photometric_fwd_bwd_f32", P(d["es"]), P(d["ta"]), P(d["go"]), P(o1), P(g1), B, 1, H, W, 9, 1, 0.5)
        _lib.call("ctd_host_photometric_fwd_bwd_f32", P(d["es"]), P(d["ta"]), P(d["go"]), P(o3), P(g3), B, 1, H, W, 9, 3, 0.5)
        _lib.call("ctd_host_proj_nn_f32", P(xyz), P(xyz), P(K), P(idx), B, H, W, 3)
        if deferred:
            _lib.call("ctd_host_end_batch")
            # the second photometric call reads the same es / ta / grad_out: they crossed the bus once
            copied, saved = ctypes.c_uint64(0), ctypes.c_uint64(0)
            _lib.lib().ctd_host_batch_stats(ctypes.byref(copied), ctypes.byref(saved))
            plane = B * H * W * 4
            # ... and so did the point cloud that proj_nn reads as both xyz0 and xyz1 (3 floats per pixel)
            assert saved.value == (3 + 3) * plane and copied.value >= 4 * plane
        res.append((lcn, std, o1, g1, o3, g3, idx))
    for a, b in zip(*res):
        assert np.array_equal(a, b)
    assert_close(res[1][4], oracle.photometric_loss_forward(d["es"], d["ta"], 9, 3, 0.5), what="deferred census fwd")
    with pytest.raises(Exception):
        _lib.call("ctd_host_end_batch")  # no batch open


def test_host_api_repeated_batch_is_replayed_as_a_graph(tx):
    """A batch that repeats with pinned buffers: ordinary the first time, captured (and launched) the second, one graph
    launch from the third on.  The inputs change between repetitions -- a replayed batch has to read the host buffers
    again -- and every repetition is checked against the oracle.  Then the batch diverges in its third call (other loss
    type): issued the ordinary way, same answers.  The same calls on pageable (numpy) buffers never become a graph."""
    from connecting_the_dots_b200 import _lib, synth
    B, H, W = 4, 40, 64
    d = synth.make_batch(B, H, W)
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    h = {k: pin(d[k]) for k in ("im", "es", "ta", "go")}
    for k in ("lcn", "std", "gi1", "gi3"):
        h[k] = torch.empty(B, 1, H, W).pin_memory()
    h["sums"] = torch.zeros(4).pin_memory()
    L = _lib.lib()
    L.ctd_host_release()   # forget what earlier tests left in this thread's cache
    _lib.set_option("host_graphs", 1)

    def stats():
        c, l, b = ctypes.c_uint64(0), ctypes.c_uint64(0), ctypes.c_uint64(0)
        L.ctd_host_graph_stats(ctypes.byref(c), ctypes.byref(l), ctypes.byref(b))
        return c.value, l.value, b.value

    def batch(third_type=3):
        _lib.call("ctd_host_begin_batch")
        _lib.call("ctd_host_lcn_f32", P(h["im"]), P(h["lcn"]), P(h["std"]), B, H, W, 5, 0.05)
        _lib.call("ctd_host_photometric_fwd_bwd_masked_f32", P(h["es"]), P(h["ta"]), P(h["go"]), P(h["std"]), None, P(h["gi1"]),
                  ctypes.c_void_p(h["sums"].data_ptr()), B, 1, H, W, 9, 1, 0.5)
        _lib.call("ctd_host_photometric_fwd_bwd_masked_f32", P(h["es"]), P(h["ta"]), P(h["go"]), P(h["std"]), None, P(h["gi3"]),
                  ctypes.c_void_p(h["sums"].data_ptr() + 8), B, 1, H, W, 9, third_type, 0.5)
        _lib.call("ctd_host_end_batch")

    def check(third_type=3):
        es, ta, go, im = (h[k].numpy() for k in ("es", "ta", "go", "im"))
        lo, so = oracle.lcn(im, 5, 0.05)
        assert_close(h["lcn"].numpy(), lo, what="lcn")
        assert_close(h["std"].numpy(), so, what="std")
        assert_close(h["gi1"].numpy(), oracle.photometric_loss_backward(es, ta, go, 9, 1, 0.5), what="sad gradient")
        assert_close(h["gi3"].numpy(), oracle.photometric_loss_backward(es, ta, go, 9, third_type, 0.5), what="census gradient")
        for j, ty in ((0, 1), (2, third_type)):
            of = oracle.photometric_loss_forward(es, ta, 9, ty, 0.5)
            want = np.array([(so.astype(np.float64) * of).sum(), so.astype(np.float64).sum()])
            assert np.abs(h["sums"].numpy()[j:j + 2] - want).max() <= 1e-5 * np.abs(want).max()

    base = stats()
    rng = np.random.RandomState(3)
    for rep in range(5):
        for k in ("lcn", "std", "gi1", "gi3"):
            h[k].fill_(7.0)   # poison the outputs
        h["es"].copy_(torch.from_numpy(d["es"] + 0.1 * rep * rng.randn(B, 1, H, W).astype(np.float32)))
        h["im"].copy_(torch.from_numpy(np.roll(d["im"], rep, axis=3)))
        batch()
        check()
        c, l, b = (x - y for x, y in zip(stats(), base))
        assert (c, l, b) == ((0, 0, 0), (1, 1, 0), (1, 2, 0), (1, 3, 0), (1, 4, 0))[rep], "repetition %d: %r" % (rep, (c, l, b))
    batch(third_type=2)   # diverges at the third call: the first two are issued late, nothing is lost
    check(third_type=2)
    c, l, b = (x - y for x, y in zip(stats(), base))
    assert (c, l, b) == (1, 4, 1)
    batch()               # expected to be the other kind (most recent), recognised at the third call: the cached graph runs
    check()
    assert tuple(x - y for x, y in zip(stats(), base)) == (1, 5, 1)
    batch(third_type=2)   # second sighting of the other kind: starts as a replay of the first, becomes a capture
    check(third_type=2)
    assert tuple(x - y for x, y in zip(stats(), base)) == (2, 6, 1)
    for third in (2, 3, 3, 2):   # both kinds cached now, in any order
        batch(third_type=third)
        check(third_type=third)
    assert tuple(x - y for x, y in zip(stats(), base)) == (2, 10, 1)
    # pageable buffers: same calls three times, never captured
    n = {k: v.numpy().copy() for k, v in h.items()}
    Pn = lambda a, off=0: ctypes.c_void_p(a.ctypes.data + off)
    before = stats()
    for rep in range(3):
        _lib.call("ctd_host_begin_batch")
        _lib.call("ctd_host_lcn_f32", Pn(n["im"]), Pn(n["lcn"]), Pn(n["std"]), B, H, W, 5, 0.05)
        _lib.call("ctd_host_photometric_fwd_bwd_masked_f32", Pn(n["es"]), Pn(n["ta"]), Pn(n["go"]), Pn(n["std"]), None, Pn(n["gi3"]),
                  Pn(n["sums"]), B, 1, H, W, 9, 3, 0.5)
        _lib.call("ctd_host_end_batch")
        assert_close(n["gi3"], oracle.photometric_loss_backward(n["es"], n["ta"], n["go"], 9, 3, 0.5), what="pageable census gradient")
    after = stats()
    assert after[0] == before[0] and after[1] == before[1]
    _lib.set_option("host_graphs", 0)
    L.ctd_host_release()


def test_host_api_two_batches_in_flight(tx):
    """ctd_host_end_batch_async / ctd_host_wait_batch: steps issued two deep over three rotating sets of pinned buffers (the
    uploads of step k + 1 cross the bus under the downloads of step k) give the bytes of the same steps issued one at a
    time -- with and without graph replay, with a larger batch in the middle (the workspace has to grow while a batch is in
    flight) and a synchronous call at the end (waits for what is outstanding)."""
    from connecting_the_dots_b200 import _lib, synth
    H, W = 40, 64
    L = _lib.lib()
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    sizes = [4, 4, 4, 4, 7, 4, 4, 4, 4, 4]   # images per step
    rng = np.random.RandomState(8)
    steps = []
    for k, B in enumerate(sizes):
        d = synth.make_batch(B, H, W)
        steps.append({"im": np.roll(d["im"], k, axis=3), "es": d["es"] + 0.05 * k * rng.randn(B, 1, H, W).astype(np.float32),
                      "ta": d["ta"], "go": d["go"]})

    def buffers(B):
        h = {k: torch.empty(B, 1, H, W).pin_memory() for k in ("im", "es", "ta", "go", "lcn", "std", "gi")}
        h["sums"] = torch.zeros(2).pin_memory()
        return h

    def issue(h, B):
        _lib.call("ctd_host_lcn_f32", P(h["im"]), P(h["lcn"]), P(h["std"]), B, H, W, 5, 0.05)
        _lib.call("ctd_host_photometric_fwd_bwd_masked_f32", P(h["es"]), P(h["ta"]), P(h["go"]), P(h["std"]), None, P(h["gi"]),
                  P(h["sums"]), B, 1, H, W, 9, 3, 0.5)

    def fill(h, st):
        for k in ("im", "es", "ta", "go"):
            h[k].copy_(torch.from_numpy(st[k]))
        for k in ("lcn", "std", "gi"):
            h[k].fill_(7.0)

    def result(h):
        return tuple(h[k].numpy().copy() for k in ("lcn", "std", "gi", "sums"))

    for graphs in (0, 1):
        L.ctd_host_release()
        _lib.set_option("host_graphs", graphs)
        try:
            want = []
            for st, B in zip(steps, sizes):   # one at a time
                h = buffers(B)
                fill(h, st)
                _lib.call("ctd_host_begin_batch")
                issue(h, B)
                _lib.call("ctd_host_end_batch")
                want.append(result(h))
            sets = {}
            got, inflight = [], []
            for k, (st, B) in enumerate(zip(steps, sizes)):   # two deep
                h = sets.setdefault((k % 3, B), buffers(B))
                fill(h, st)
                _lib.call("ctd_host_begin_batch")
                issue(h, B)
                _lib.call("ctd_host_end_batch_async")
                inflight.append(h)
                if len(inflight) == 2:
                    _lib.call("ctd_host_wait_batch")
                    got.append(result(inflight.pop(0)))
            # a synchronous call now has to wait for the batch still in flight before it reuses the workspace
            l2, s2 = np.empty((1, 1, H, W), np.float32), np.empty((1, 1, H, W), np.float32)
            _lib.call("ctd_host_lcn_f32", ctypes.c_void_p(steps[0]["im"][:1].ctypes.data), ctypes.c_void_p(l2.ctypes.data),
                      ctypes.c_void_p(s2.ctypes.data), 1, H, W, 5, 0.05)
            got.append(result(inflight.pop(0)))
            _lib.call("ctd_host_wait_batch")   # nothing outstanding: returns at once
            assert len(got) == len(want)
            for k, (a, b) in enumerate(zip(got, want)):
                for x, y, name in zip(a, b, ("lcn", "std", "gi", "sums")):
                    assert np.array_equal(x, y), "step %d: %s differs (graphs %d)" % (k, name, graphs)
            assert np.array_equal(l2, want[0][0][:1])
        finally:
            _lib.set_option("host_graphs", 0)
            L.ctd_host_release()


def test_host_api_batch_output_feeds_later_call(tx):
    """Inside a deferred batch an OUTPUT of one call that is an INPUT of a later one (LCN's lcn / std as the loss's target
    and mask; ProjNN's indices into CrossCheck) must not be re-uploaded from the stale host buffer: exact matches are
    served from the producer's device buffer, partial overlaps wait for the download.  Checked against the same calls
    made synchronously, with the host output buffers poisoned beforehand."""
    from connecting_the_dots_b200 import _lib, synth
    B, H, W = 4, 64, 96
    d = synth.make_batch(B, H, W)
    P = lambda a, off=0: ctypes.c_void_p(a.ctypes.data + off)
    xyz, K, poses = synth.make_clouds(2, H, W)
    x01 = np.ascontiguousarray(synth.transform(xyz[0], poses[1])[None])
    x10 = np.ascontiguousarray(synth.transform(xyz[1], poses[0])[None])
    x0, x1 = np.ascontiguousarray(xyz[0][None]), np.ascontiguousarray(xyz[1][None])
    res = []
    for deferred in (False, True):
        lcn, std = np.full_like(d["im"], 7.0), np.full_like(d["im"], 7.0)   # poison: a stale upload would show
        out, gi = np.full_like(d["es"], 7.0), np.full_like(d["es"], 7.0)
        gi_half = np.full_like(d["es"][:2], 7.0)
        sums, sums_half = np.zeros(2, np.float32), np.zeros(2, np.float32)
        i01, i10 = np.full((1, H, W), -5, np.int64), np.full((1, H, W), -5, np.int64)
        m = np.full(H * W, 9, np.uint8)
        if deferred:
            _lib.call("ctd_host_begin_batch")
        _lib.call("ctd_host_lcn_f32", P(d["im"]), P(lcn), P(std), B, H, W, 5, 0.05)
        # exact match: ta = lcn output, mask = std output, same chunking
        _lib.call("ctd_host_photometric_fwd_bwd_masked_f32", P(d["es"]), P(lcn), P(d["go"]), P(std), P(out), P(gi), P(sums),
                  B, 1, H, W, 9, 3, 0.5)
        # partial overlap: the first two images only, no loss map wanted
        _lib.call("ctd_host_photometric_fwd_bwd_masked_f32", P(d["es"]), P(lcn), P(d["go"]), P(std), None, P(gi_half), P(sums_half),
                  2, 1, H, W, 9, 1, 0.5)
        _lib.call("ctd_host_proj_nn_f32", P(x01), P(x1), P(K), P(i01), 1, H, W, 3)
        _lib.call("ctd_host_proj_nn_f32", P(x10), P(x0), P(K), P(i10), 1, H, W, 3)
        _lib.call("ctd_host_crosscheck", P(i01), P(i10), P(m), H * W, H * W)
        if deferred:
            _lib.call("ctd_host_end_batch")
        res.append((lcn, std, out, gi, gi_half, sums, sums_half, i01, i10, m))
    for a, b in zip(*res):
        assert np.array_equal(a, b)
    lcn, std, out, gi, gi_half, sums, sums_half, i01, i10, m = res[1]
    lo, so = oracle.lcn(d["im"], 5, 0.05)
    assert_close(lcn, lo, what="lcn")
    assert_close(out, oracle.photometric_loss_forward(d["es"], lcn, 9, 3, 0.5), what="loss on the batch's own lcn")
    assert_close(gi, oracle.photometric_loss_backward(d["es"], lcn, d["go"], 9, 3, 0.5), what="grad")
    assert_close(gi_half, oracle.photometric_loss_backward(d["es"][:2], lcn[:2], d["go"][:2], 9, 1, 0.5), what="grad, half batch")
    want = np.array([(std.astype(np.float64) * out).sum(), std.astype(np.float64).sum()])
    assert np.abs(sums - want).max() <= 1e-5 * want.max()
    o2 = oracle.photometric_loss_forward(d["es"][:2], lcn[:2], 9, 1, 0.5)
    want = np.array([(std[:2].astype(np.float64) * o2).sum(), std[:2].astype(np.float64).sum()])
    assert np.abs(sums_half - want).max() <= 1e-5 * want.max()
    assert np.array_equal(m, oracle.crosscheck(i01.ravel(), i10.ravel())) and m.max() <= 1


def test_masked_loss_calls_do_not_share_reduction_slots(tx):
    """The ticket / block-partial workspace of the fused masked calls: captured calls own their slot, eager calls share
    one per stream.  Two graphs replayed on two streams while eager calls run on a third must all keep producing the
    sums of their own inputs."""
    from connecting_the_dots_b200 import _lib
    B, H, W = 2, 96, 160
    torch.manual_seed(3)
    def make(seed):
        g = torch.Generator(device="cpu").manual_seed(seed)
        t = {k: torch.randn(B, 1, H, W, generator=g).to(DEV) for k in ("es", "ta")}
        t["go"] = torch.rand(B, 1, H, W, generator=g).to(DEV)
        t["mask"] = torch.rand(B, 1, H, W, generator=g).to(DEV) + 0.5
        t["out"], t["gi"], t["sums"] = torch.empty(B, 1, H, W, device=DEV), torch.empty(B, 1, H, W, device=DEV), torch.zeros(2, device=DEV)
        return t
    def launch(t, ty, st):
        _lib.call("ctd_photometric_fwd_bwd_masked_f32", t["es"].data_ptr(), t["ta"].data_ptr(), t["go"].data_ptr(), t["mask"].data_ptr(),
                  t["out"].data_ptr(), t["gi"].data_ptr(), t["sums"].data_ptr(), B, 1, H, W, 9, ty, 0.5, st)
    sets = [make(s) for s in range(3)]
    want = []
    for i, t in enumerate(sets):
        launch(t, 3 if i != 1 else 1, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        want.append(t["sums"].clone())
        exp = torch.stack([(t["mask"].double() * t["out"].double()).sum(), t["mask"].double().sum()]).float()
        assert torch.allclose(want[-1], exp, rtol=1e-5)
    graphs = []
    for i in (0, 1):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            launch(sets[i], 3 if i != 1 else 1, torch.cuda.current_stream().cuda_stream)
        graphs.append(g)
    s0, s1, s2 = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    for it in range(20):
        for t in sets:
            t["sums"].zero_()
        torch.cuda.synchronize()
        with torch.cuda.stream(s0):
            graphs[0].replay()
        with torch.cuda.stream(s1):
            graphs[1].replay()
        launch(sets[2], 3, s2.cuda_stream)
        torch.cuda.synchronize()
        for t, w in zip(sets, want):
            assert torch.equal(t["sums"], w), it


def test_masked_calls_under_capture_when_static_slots_are_exhausted(tx):
    """When the static reduction slots run out (more than 96 captured masked calls in a process) the workspace comes from
    the stream-ordered scratch pool with a memset node: captured and replayed like any other call, same sums.  Runs in a
    fresh process so that the scratch pool's FIRST use happens inside the capture (pool creation must not break it)."""
    import subprocess, sys, os
    code = """
import sys, torch
sys.path.insert(0, %r)
from connecting_the_dots_b200 import _lib
B, H, W = 2, 64, 96
g = torch.Generator(device="cpu").manual_seed(1)
t = {k: torch.randn(B, 1, H, W, generator=g).cuda() for k in ("es", "ta")}
t["go"], t["mask"] = torch.rand(B, 1, H, W, generator=g).cuda(), torch.rand(B, 1, H, W, generator=g).cuda() + 0.5
out, gi, sums = torch.empty(B, 1, H, W, device="cuda"), torch.empty(B, 1, H, W, device="cuda"), torch.zeros(3, 2, device="cuda")
def launch(ty, k, st):
    _lib.call("ctd_photometric_fwd_bwd_masked_f32", t["es"].data_ptr(), t["ta"].data_ptr(), t["go"].data_ptr(), t["mask"].data_ptr(),
              out.data_ptr(), gi.data_ptr(), sums[k].data_ptr(), B, 1, H, W, 9, ty, 0.5, st)
_lib.set_option("ms_force_scratch", 1)
gr = torch.cuda.CUDAGraph()
with torch.cuda.graph(gr):
    st = torch.cuda.current_stream().cuda_stream
    launch(1, 0, st); launch(3, 1, st)
for _ in range(3):
    sums.zero_(); gr.replay(); torch.cuda.synchronize()
got = sums[:2].clone()
_lib.set_option("ms_force_scratch", 0)
launch(1, 0, torch.cuda.current_stream().cuda_stream); launch(3, 1, torch.cuda.current_stream().cuda_stream)
torch.cuda.synchronize()
assert torch.equal(got, sums[:2]), (got, sums)
print("OK")
""" % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "OK" in r.stdout, r.stderr[-2000:]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_xcorrvol_on_second_device(tx):
    """Per-device kernel attributes (dynamic shared memory above 48 KB) are set for every device a process uses."""
    rng = np.random.RandomState(0)
    a = rng.rand(1, 40, 150).astype(np.float32)
    b = rng.rand(1, 40, 150).astype(np.float32)
    want = oracle.xcorrvol(a, b, 32, 9)
    for dev in ("cuda:0", "cuda:1", "cuda:0"):
        got = tx.xcorrvol(torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev), 32, 9)
        assert_close(got.cpu().numpy(), want, what=dev)


# ---------------------------------------------------------------- warp + fused loss (SURVEY 8f rank 1)
class _OraclePhotometric(torch.autograd.Function):
    """photometric_loss evaluated by the CPU ORACLE (forward and backward), so the reference recipe below does not lean
    on the library under test for the loss half."""

    @staticmethod
    def forward(ctx, es, ta, bs, ty, eps):
        ctx.save_for_backward(es, ta)
        ctx.args = (bs, ty, eps)
        out = oracle.photometric_loss_forward(es.detach().cpu().numpy(), ta.detach().cpu().numpy(), bs, ty, eps)
        return torch.from_numpy(out).to(es.device)

    @staticmethod
    def backward(ctx, go):
        es, ta = ctx.saved_tensors
        bs, ty, eps = ctx.args
        gi = oracle.photometric_loss_backward(es.detach().cpu().numpy(), ta.detach().cpu().numpy(),
                                              np.ascontiguousarray(go.detach().cpu().numpy()), bs, ty, eps)
        return torch.from_numpy(gi).to(es.device), None, None, None, None


def _reference_pattern_loss(disp, pattern, im, std, loss_type, eps, tx):
    """model/networks.py:358-378 with torch ops (grid_sample on the GPU) and the ORACLE's photometric loss."""
    B, _, H, W = disp.shape
    v, u = torch.meshgrid(torch.arange(H, device=disp.device, dtype=torch.float32),
                          torch.arange(W, device=disp.device, dtype=torch.float32), indexing="ij")
    uv1 = torch.empty(B, H * W, 2, device=disp.device)
    uv1[..., 0] = u.reshape(1, -1) - disp.contiguous().view(B, -1)
    uv1[..., 1] = v.reshape(1, -1)
    uv1[..., 0] = 2 * (uv1[..., 0] / (W - 1) - 0.5)
    uv1[..., 1] = 2 * (uv1[..., 1] / (H - 1) - 0.5)
    uv1 = uv1.view(-1, H, W, 2).clone()
    pat = pattern.expand(B, *pattern.shape[1:])
    proj = torch.nn.functional.grid_sample(pat, uv1, padding_mode="border", align_corners=False)
    diff = _OraclePhotometric.apply(proj.contiguous(), im.contiguous(), 9, loss_type, eps)
    return (std * diff).sum() / std.sum(), proj


@pytest.mark.parametrize("shape", [(2, 96, 160, 96, 160), (1, 60, 80, 120, 160), (3, 33, 50, 33, 50)])
def test_warp_pattern_matches_grid_sample(tx, shape):
    """warp_pattern against torch's CUDA grid_sample fed the reference's grid, values and d/d disp."""
    B, H, W, Hp, Wp = shape
    g = torch.Generator(device="cpu").manual_seed(H)
    pattern = torch.randn(1, 1, Hp, Wp, generator=g).to(DEV)
    disp = (torch.rand(B, 1, H, W, generator=g) * (W * 0.4) - 4).to(DEV).requires_grad_(True)   # some samples leave the image
    go = torch.randn(B, 1, H, W, generator=g).to(DEV)
    ones = torch.ones(B, 1, H, W, device=DEV)
    _, proj_ref = _reference_pattern_loss(disp, pattern, ones, ones, "sad", 0.5, tx)
    (gref,) = torch.autograd.grad(proj_ref, disp, go)
    proj = tx.warp_pattern(pattern, disp)
    (g_,) = torch.autograd.grad(proj, disp, go)
    assert_close(proj.detach().cpu().numpy(), proj_ref.detach().cpu().numpy(), what="warp forward")
    assert_close(g_.cpu().numpy(), gref.cpu().numpy(), what="warp backward")


@pytest.mark.parametrize("loss_type", ("census_sad", "sad"))
def test_pattern_similarity_loss_matches_reference_recipe(tx, loss_type):
    """The whole RectifiedPatternSimilarityLoss.tforward: value, pattern_proj and the gradient w.r.t. the disparity."""
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(2, 96, 160)
    pattern = cu(d["pat_lcn"][:1])
    im, std = cu(d["ta"]), cu(d["std"])
    disp = cu(d["disp"] if d["disp"].ndim == 4 else d["disp"][:, None]).clone().requires_grad_(True)
    ref, proj_ref = _reference_pattern_loss(disp, pattern, im, std, loss_type, 0.5, tx)
    (gref,) = torch.autograd.grad(ref, disp)
    for fused in (True, False):   # one kernel (census modes) and the three-kernel composition
        val, proj = tx.pattern_similarity_loss(disp, pattern, im, std, loss_type, 0.5, fused=fused)
        (g_,) = torch.autograd.grad(val, disp)
        assert abs(val.item() - ref.item()) <= 1e-5 * abs(ref.item())
        assert_close(proj.detach().cpu().numpy(), proj_ref.detach().cpu().numpy(), what="pattern_proj")
        assert_close(g_.cpu().numpy(), gref.cpu().numpy(), what="d loss / d disp")


@pytest.mark.parametrize("shape", [(2, 96, 160, 96, 160), (1, 60, 83, 120, 160), (2, 33, 50, 33, 50), (1, 480, 640, 480, 640)])
@pytest.mark.parametrize("loss_type", ("census_sad", "census_mse"))
def test_pattern_similarity_single_kernel_matches_three_kernels(tx, shape, loss_type):
    """ctd_pattern_similarity_f32 (warp inside the census kernel's tile loader, gradient chained to the disparity in its
    epilogue) against the three-kernel composition: same pattern_proj bit for bit, same value and gradient; disparities
    that send samples off both sides of the pattern, ragged sizes, a pattern of another size than the image."""
    B, H, W, Hp, Wp = shape
    g = torch.Generator(device="cpu").manual_seed(H + W)
    pattern = torch.randn(1, 1, Hp, Wp, generator=g).to(DEV)
    disp = (torch.rand(B, 1, H, W, generator=g) * (W * 0.3) - 6).to(DEV)
    im = torch.randn(B, 1, H, W, generator=g).to(DEV)
    std = (torch.rand(B, 1, H, W, generator=g) + 0.1).to(DEV)
    res = []
    for fused in (True, False):
        d = disp.clone().requires_grad_(True)
        val, proj = tx.pattern_similarity_loss(d, pattern, im, std, loss_type, 0.5, fused=fused)
        (gd,) = torch.autograd.grad(val, d)
        res.append((val.detach(), proj.detach(), gd))
    assert torch.equal(res[0][1], res[1][1]), "pattern_proj differs"
    assert abs(res[0][0].item() - res[1][0].item()) <= 1e-6 * abs(res[1][0].item())
    assert_close(res[0][2].cpu().numpy(), res[1][2].cpu().numpy(), tol=1e-6, what="d loss / d disp")


def test_pyramid_pattern_similarity_loss(tx):
    """The photometric part of exp_synph.loss_forward over the four pyramid levels (exp_synph.py:25-27,107-111): every
    level's value and d value / d disp against the reference recipe (torch grid_sample + the ORACLE's photometric loss),
    and the whole pyramid (forward and backward) replayed as one CUDA graph giving the same numbers."""
    from connecting_the_dots_b200 import synth
    levels = [synth.make_batch(2, 480 >> s, 640 >> s) for s in range(4)]
    pats = [cu(d["pat_lcn"][:1]) for d in levels]
    ims, stds = [cu(d["ta"]) for d in levels], [cu(d["std"]) for d in levels]
    disps = [cu(d["disp"]).clone().requires_grad_(True) for d in levels]
    vals, proj0 = tx.pyramid_pattern_similarity_loss(disps, pats, ims, stds)
    grads = torch.autograd.grad(sum(vals), disps)
    assert len(vals) == 4 and proj0.shape == (2, 1, 480, 640) and not proj0.requires_grad
    for s in (1, 2, 3):   # the reference recipe on every level the oracle finishes quickly (level 0: test_pattern_similarity_loss...)
        ref, _ = _reference_pattern_loss(disps[s], pats[s], ims[s], stds[s], "census_sad", 0.5, tx)
        (gref,) = torch.autograd.grad(ref, disps[s])
        assert abs(vals[s].item() - ref.item()) <= 1e-5 * abs(ref.item()), s
        assert_close(grads[s].cpu().numpy(), gref.cpu().numpy(), what="level %d d loss / d disp" % s)
    # one graph for the 12 kernels of the pyramid
    static_d = [d.detach().clone().requires_grad_(True) for d in disps]
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        v_, _ = tx.pyramid_pattern_similarity_loss(static_d, pats, ims, stds)   # warm-up outside capture
        torch.autograd.grad(sum(v_), static_d)
    torch.cuda.current_stream().wait_stream(side)
    with torch.cuda.graph(g):
        gv, _ = tx.pyramid_pattern_similarity_loss(static_d, pats, ims, stds)
        gg = torch.autograd.grad(sum(gv), static_d)
    g.replay()
    torch.cuda.synchronize()
    for s in range(4):
        assert torch.equal(gv[s], vals[s]) and torch.equal(gg[s], grads[s]), s


def test_loss_path_is_cuda_graph_capturable(tx):
    """Every call of the loss path (LCN, warp, fused masked loss, warp gradient) can be captured into one CUDA graph
    (scratch comes from a stream-ordered pool / static slots, nothing synchronises); a replay reproduces the eager
    results bit for bit."""
    from connecting_the_dots_b200 import synth
    d = synth.make_batch(2, 96, 160)
    pattern = cu(d["pat_lcn"][:1])
    im_raw, disp = cu(d["im"]), cu(d["disp"])

    def run():
        lcn, std = tx.ext_cuda.lcn_forward(im_raw, 5, 0.05)
        proj = tx.ext_cuda.warp_pattern_forward(pattern, disp)
        out, gi, sums = tx.ext_cuda.photometric_loss_forward_backward_masked(proj, lcn, std, std, 9, 3, 0.5)
        gd = tx.ext_cuda.warp_pattern_backward(pattern, disp, gi)
        return lcn, proj, out, gi, sums, gd

    eager = [t.clone() for t in run()]
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        captured = run()
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()
    for a, b in zip(eager, captured):
        assert torch.equal(a, b)


# ---------------------------------------------------------------- geometric loss (SURVEY 8f rank 3)
from losses_torch import depth_similarity as _ref_depth_similarity, disparity_loss as _ref_disparity_loss  # noqa: E402


def _grad_close(got, ref, what, tol=1e-5, outliers=2e-3):
    """Gradients of |d - s| jump by 2/N where d - s changes sign and by a finite-difference step where the sample
    crosses a pixel boundary, so a rounding-level difference in the projection (bmm summation order) flips a few
    pixels: all but a fraction `outliers` of the pixels must agree to tol * max|ref|, and the flips must be bounded."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    scale = np.abs(ref).max()
    err = np.abs(got - ref)
    bad = err > tol * scale
    assert bad.mean() <= outliers, f"{what}: {bad.mean():.2e} of the pixels differ (max err {err.max():.3e}, scale {scale:.3e})"
    assert err.max() <= 4.5 * scale, f"{what}: outlier of {err.max():.3e} against scale {scale:.3e}"


@pytest.mark.parametrize("name,clamp", (("noclamp", -1), ("clamp", 0.1), ("tight", 0.004)))
def test_depth_similarity_golden(tx, golden, name, clamp):
    """Against values and autograd gradients of the reference's own ProjectionDepthSimilarityLoss on CPU torch
    (tests/golden/make_golden_geometric.py)."""
    g = golden("geometric")
    d0, d1 = cu(g["depth0"]).requires_grad_(True), cu(g["depth1"]).requires_grad_(True)
    val = tx.projection_depth_similarity_loss(d0, d1, cu(g["R0"]), cu(g["t0"]), cu(g["R1"]), cu(g["t1"]), cu(g["K"]), cu(g["ray"]), clamp)
    val.backward()
    assert abs(float(val) - float(g[name + "_val"])) <= 1e-5 * abs(float(g[name + "_val"]))
    _grad_close(d0.grad.cpu().numpy(), g[name + "_g0"], name + " grad depth0", outliers=5e-3)
    _grad_close(d1.grad.cpu().numpy(), g[name + "_g1"], name + " grad depth1", outliers=5e-3)


def test_depth_similarity_vs_torch_full_size(tx):
    """Batch 4 at 480x640 against the torch restatement of networks.py:436-503 on the same GPU, value and both
    gradients, plus the upstream-gradient scaling and the ray table helper."""
    from connecting_the_dots_b200 import synth
    d = synth.make_depth_pairs(4, 480, 640, seed=3)
    ray = tx.projection_rays(d["Ki"], 480, 640).to(DEV)
    args = [cu(d[k]) for k in ("R0", "t0", "R1", "t1", "K")]
    for clamp in (-1, 0.1):
        a0, a1 = cu(d["depth0"]).requires_grad_(True), cu(d["depth1"]).requires_grad_(True)
        b0, b1 = cu(d["depth0"]).requires_grad_(True), cu(d["depth1"]).requires_grad_(True)
        val = tx.projection_depth_similarity_loss(a0, a1, *args, ray, clamp)
        ref = _ref_depth_similarity(b0, b1, *args, ray, clamp)
        (3.0 * val).backward()
        (3.0 * ref).backward()
        assert abs(float(val) - float(ref)) <= 1e-5 * abs(float(ref)), (float(val), float(ref))
        _grad_close(a0.grad.cpu().numpy(), b0.grad.cpu().numpy(), "grad depth0 clamp %g" % clamp)
        _grad_close(a1.grad.cpu().numpy(), b1.grad.cpu().numpy(), "grad depth1 clamp %g" % clamp)


def test_depth_similarity_identity_and_errors(tx):
    """Identical frames and poses: every pixel projects onto itself, and what is left is the reference's own
    sampling convention (grid normalised with W-1, sampled with align_corners=False: position x*W/(W-1) - 0.5) --
    small against the depth and equal to the torch restatement.  Shape / device / dtype violations raise like the
    other ops."""
    from connecting_the_dots_b200 import synth
    d = synth.make_depth_pairs(2, 48, 64, seed=5)
    ray = tx.projection_rays(d["Ki"], 48, 64).to(DEV)
    dep = cu(d["depth0"])
    val = tx.projection_depth_similarity_loss(dep, dep.clone(), cu(d["R0"]), cu(d["t0"]), cu(d["R0"]), cu(d["t0"]), cu(d["K"]), ray, 0.1)
    ref = _ref_depth_similarity(dep, dep.clone(), cu(d["R0"]), cu(d["t0"]), cu(d["R0"]), cu(d["t0"]), cu(d["K"]), ray, 0.1)
    assert abs(float(val) - float(ref)) <= 1e-5 * float(ref)
    assert float(val) <= 0.2 * float(dep.mean())
    with pytest.raises(RuntimeError):
        tx.projection_depth_similarity_loss(dep.cpu(), dep.cpu(), cu(d["R0"]), cu(d["t0"]), cu(d["R0"]), cu(d["t0"]), cu(d["K"]), ray, 0.1)
    with pytest.raises(RuntimeError):
        tx.projection_depth_similarity_loss(dep, dep[:, :, :-1].contiguous(), cu(d["R0"]), cu(d["t0"]), cu(d["R0"]), cu(d["t0"]), cu(d["K"]), ray, 0.1)
    with pytest.raises((RuntimeError, NotImplementedError)):
        tx.projection_depth_similarity_loss(dep.double(), dep.double(), cu(d["R0"]), cu(d["t0"]), cu(d["R0"]), cu(d["t0"]), cu(d["K"]), ray, 0.1)


# ---------------------------------------------------------------- disparity loss (SURVEY 8f rank 4)
@pytest.mark.parametrize("name", ("edge", "noedge"))
def test_disparity_loss_golden(tx, golden, name):
    """Against the reference's own DisparityLoss / SobelFilter on CPU torch (tests/golden/make_golden_geometric.py)."""
    g = golden("disparity_loss")
    d = cu(g["disp"]).requires_grad_(True)
    e = cu(g["edge"]).requires_grad_(True) if name == "edge" else None
    val = tx.disparity_loss(d, e)
    val.backward()
    ref = float(g[name + "_val"])
    assert abs(float(val.detach()) - ref) <= 1e-5 * abs(ref), (float(val.detach()), ref)
    assert_close(d.grad.cpu().numpy(), g[name + "_gdisp"], tol=2e-5, what=name + " grad disp")
    if e is not None:
        assert_close(e.grad.cpu().numpy(), g[name + "_gedge"], tol=2e-5, what=name + " grad edge")


def test_disparity_loss_vs_torch_full_size(tx):
    """Batch 8 at 480x640 (a full-resolution disparity map and a sigmoid edge map, exp_synph.py:115-116) against the
    torch restatement on the same GPU; odd sizes that do not fill the 32x32 tiles; upstream-gradient scaling."""
    from connecting_the_dots_b200 import synth
    torch.backends.cudnn.allow_tf32 = False  # the reference's two convolutions in fp32, not TF32 (cuDNN's default)
    for (B, H, W) in ((8, 480, 640), (3, 61, 83)):
        base = np.stack([synth.smooth_disparity(np.random.RandomState(60 + n), H, W) for n in range(B)])[:, None].astype(np.float32)
        base = base / 8.0 if H < 100 else base
        rng = np.random.RandomState(B)
        edge = (1.0 / (1.0 + np.exp(-rng.randn(B, 1, H, W) * 2))).astype(np.float32)
        for use_edge in (True, False):
            a, b = cu(base).requires_grad_(True), cu(base).requires_grad_(True)
            ea = cu(edge).requires_grad_(True) if use_edge else None
            eb = cu(edge).requires_grad_(True) if use_edge else None
            val = tx.disparity_loss(a, ea)
            ref = _ref_disparity_loss(b, eb)
            (2.5 * val).backward()
            (2.5 * ref).backward()
            assert abs(float(val.detach()) - float(ref.detach())) <= 1e-5 * abs(float(ref.detach()))
            assert_close(a.grad.cpu().numpy(), b.grad.cpu().numpy(), tol=2e-5, what="grad disp %dx%d edge=%s" % (H, W, use_edge))
            if use_edge:
                assert_close(ea.grad.cpu().numpy(), eb.grad.cpu().numpy(), tol=2e-5, what="grad edge %dx%d" % (H, W))
    with pytest.raises(RuntimeError):
        tx.disparity_loss(cu(base).cpu(), None)
    with pytest.raises(RuntimeError):
        tx.disparity_loss(cu(base), cu(edge)[:, :, :-1].contiguous())


# ---------------------------------------------------------------- no writes outside the outputs
def _guarded(shape, dtype=torch.float32, pad=4096, fill=-777.0):
    """A tensor view in the middle of a larger allocation whose margins are filled with a sentinel."""
    n = int(np.prod(shape))
    raw = torch.full((n + 2 * pad,), fill, dtype=dtype, device=DEV)
    return raw, raw[pad:pad + n].view(*shape)


def _margins_intact(raw, n, pad=4096, fill=-777.0):
    return bool((raw[:pad] == fill).all()) and bool((raw[pad + n:] == fill).all())


def test_kernels_write_only_their_outputs(tx):
    """Odd sizes (partial tiles, scalar-store paths) with the outputs placed inside sentinel-filled allocations:
    the margins must come back untouched (compute-sanitizer is not available on the GPU pool)."""
    from connecting_the_dots_b200 import _lib, synth
    rng = np.random.RandomState(3)
    st = torch.cuda.current_stream().cuda_stream
    # XCorrVol, separable kernel + sweep / eval fix-up, width not a multiple of 4 and a ragged last disparity chunk
    B, H, W, D = 2, 23, 37, 19
    a = cu((0.5 + 0.02 * rng.randn(B, 1, H, W)).astype(np.float32))
    b = cu((0.5 + 0.02 * rng.randn(B, 1, H, W)).astype(np.float32))
    raw, out = _guarded((B, D, H, W))
    _lib.call("ctd_xcorrvol_f32", a.data_ptr(), b.data_ptr(), out.data_ptr(), B, 1, H, W, D, 9, st)
    torch.cuda.synchronize()
    assert _margins_intact(raw, out.numel())
    assert_close(out[0].cpu().numpy(), oracle.xcorrvol(a[0].cpu().numpy(), b[0].cpu().numpy(), D, 9), what="guarded xcorrvol")
    # mse / sad TMA kernels with a partial last tile column (W = 132) and a partial last tile row
    B, H, W = 2, 40, 132
    es, ta, go = (cu(rng.randn(B, 1, H, W).astype(np.float32)) for _ in range(3))
    for ty in (0, 1):
        raw_o, o = _guarded((B, 1, H, W))
        raw_g, g = _guarded((B, 1, H, W))
        _lib.call("ctd_photometric_fwd_bwd_f32", es.data_ptr(), ta.data_ptr(), go.data_ptr(), o.data_ptr(), g.data_ptr(), B, 1, H, W, 9, ty, 0.5, st)
        torch.cuda.synchronize()
        assert _margins_intact(raw_o, o.numel()) and _margins_intact(raw_g, g.numel())
        assert_close(o.cpu().numpy(), oracle.photometric_loss_forward(es.cpu().numpy(), ta.cpu().numpy(), 9, ty, 0.5), what="guarded fwd %d" % ty)
        assert_close(g.cpu().numpy(), oracle.photometric_loss_backward(es.cpu().numpy(), ta.cpu().numpy(), go.cpu().numpy(), 9, ty, 0.5),
                     what="guarded bwd %d" % ty)
    # geometric loss: pixel count not a multiple of the 1024-pixel step
    d = synth.make_depth_pairs(3, 19, 23, seed=9)
    ray = tx.projection_rays(d["Ki"], 19, 23).to(DEV)
    raw0, g0 = _guarded((3, 1, 19, 23))
    raw1, g1 = _guarded((3, 1, 19, 23))
    g1.zero_()
    sums = torch.zeros(2, device=DEV)
    args = [cu(d[k]) for k in ("depth0", "depth1")]
    _lib.call("ctd_depth_similarity_f32", args[0].data_ptr(), args[1].data_ptr(), ray.data_ptr(), cu(d["K"]).data_ptr(), cu(d["R0"]).data_ptr(),
              cu(d["t0"]).data_ptr(), cu(d["R1"]).data_ptr(), cu(d["t1"]).data_ptr(), g0.data_ptr(), g1.data_ptr(), sums.data_ptr(), 3, 19, 23,
              0.1, 1.0 / (3 * 19 * 23), 0, st)
    torch.cuda.synchronize()
    assert _margins_intact(raw0, g0.numel()) and _margins_intact(raw1, g1.numel())
    assert float(sums[1]) == 3 * 19 * 23
    # disparity loss: image smaller than / not a multiple of the 32x32 tile
    for (B, H, W) in ((2, 33, 35), (1, 7, 5)):
        disp = cu((rng.rand(B, 1, H, W) * 3).astype(np.float32))
        edge = cu(rng.rand(B, 1, H, W).astype(np.float32))
        raw_d, gd = _guarded((B, 1, H, W))
        raw_e, ge = _guarded((B, 1, H, W))
        _lib.call("ctd_disparity_loss_f32", disp.data_ptr(), edge.data_ptr(), gd.data_ptr(), ge.data_ptr(), sums.data_ptr(), B, H, W,
                  1.0 / (B * H * W), st)
        torch.cuda.synchronize()
        assert _margins_intact(raw_d, gd.numel()) and _margins_intact(raw_e, ge.numel())
        d_ref, e_ref = disp.clone().requires_grad_(True), edge.clone().requires_grad_(True)
        ref = _ref_disparity_loss(d_ref, e_ref)
        ref.backward()
        assert abs(float(sums[0] / sums[1]) - float(ref.detach())) <= 1e-5 * abs(float(ref.detach()))
        assert_close(gd.cpu().numpy(), d_ref.grad.cpu().numpy(), tol=2e-5, what="guarded grad disp %dx%d" % (H, W))
