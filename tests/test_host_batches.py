"""The host-buffer C ABI (ctd_host_*) at its chunk edges and in batches.

A host call cuts the image-wise ops into chunks of whole images (chunk c of B images in n chunks starts at image
B*c/n), so the kernels see sub-batches whose device base pointers are not 16-byte aligned when an image is not a
multiple of four floats.  Inside ctd_host_begin_batch / end_batch the calls only enqueue, and the library keeps its own
bookkeeping of what the batch has uploaded and what it is still downloading, so that a later call can reuse a device
copy instead of reading a stale host range.  include/ctd_b200.h promises that a batch leaves every host buffer holding
what the same calls made one at a time leave there, whatever the calls' buffers share.

* test_host_imagewise_ops_at_chunk_edges / test_host_point_ops: every ctd_host_* op against the CPU oracle at batch
  sizes below, at and above the chunk counts, odd widths, C = 1 and 2, pinned and pageable buffers.
* test_generated_batches_match_sequential_calls: seeded programs of 6-12 calls over a small pool of buffers that the
  calls share (one call's output is a later call's input, in whole or in part; outputs overwritten; inputs shared;
  in-place calls), made one at a time (each call checked against the oracle on a snapshot of its inputs), then as one
  batch, as a batch repeated under graph replay, and as batches two in flight.  With equal chunk counts in every mode
  the results must be bit-equal; at the default options (batches cut fewer chunks) they must agree to the oracle's
  tolerance.
* test_batch_*: the two stale-input hazards those programs found, as fixed three- and four-call batches.
* test_program_generator_covers_every_aliasing_pattern (CPU): the seeds above do contain every aliasing pattern.

Every host buffer sits inside a larger allocation whose margins hold a sentinel; the tests check the margins afterwards.
"""
import collections
import contextlib
import ctypes

import numpy as np
import pytest
import torch

import oracle
from conftest import assert_close

DEFAULTS = (("host_chunks", 4), ("host_chunks_batch", 2), ("host_chunks_graph", 2), ("host_graphs", 0))
PAD = 61                                   # sentinel elements on each side of a host buffer (odd: unaligned hosts too)
SENTINEL = {np.dtype(np.float32): -777.0, np.dtype(np.int64): -7770001, np.dtype(np.uint8): 0xA5}
TORCH_DTYPE = {np.dtype(np.float32): torch.float32, np.dtype(np.int64): torch.int64, np.dtype(np.uint8): torch.uint8}
EPS, LCN_R, LCN_EPS = 0.5, 5, 0.05
SEEDS = range(24)
SETTINGS = (1, 2, 3, None)                 # host_chunks = host_chunks_batch = host_chunks_graph = k; None: the defaults


def _lib():
    from connecting_the_dots_b200 import _lib
    return _lib


@contextlib.contextmanager
def host_options(**opts):
    """Set library options for a block; the library defaults and an empty workspace / graph cache afterwards."""
    L = _lib()
    L.lib().ctd_host_release()
    try:
        for k, v in opts.items():
            L.set_option(k, v)
        yield
    finally:
        for k, v in DEFAULTS:
            L.set_option(k, v)
        L.lib().ctd_host_release()


def graph_stats():
    c, l, b = ctypes.c_uint64(0), ctypes.c_uint64(0), ctypes.c_uint64(0)
    _lib().lib().ctd_host_graph_stats(ctypes.byref(c), ctypes.byref(l), ctypes.byref(b))
    return c.value, l.value, b.value


class HostBuf:
    """n elements of `dtype` inside an allocation (pinned or pageable) with PAD sentinel elements on each side."""

    def __init__(self, n, dtype, pinned):
        dtype = np.dtype(dtype)
        if pinned:
            self._t = torch.empty(n + 2 * PAD, dtype=TORCH_DTYPE[dtype]).pin_memory()
            self.raw = self._t.numpy()
        else:
            self.raw = np.empty(n + 2 * PAD, dtype)
        self.raw[:] = SENTINEL[dtype]
        self.a = self.raw[PAD:PAD + n]

    def ptr(self, off=0):
        return ctypes.c_void_p(self.a.ctypes.data + off * self.a.itemsize)

    def margins_intact(self):
        s = SENTINEL[self.raw.dtype]
        return bool((self.raw[:PAD] == s).all() and (self.raw[PAD + self.a.size:] == s).all())


def _placed(x, pinned):
    x = np.ascontiguousarray(x)
    h = HostBuf(x.size, x.dtype, pinned)
    h.a[:] = x.ravel()
    return h


def _sums_close(got, mask, loss, what):
    """sums2 of a masked call against float64 sums; the scale is the sum of magnitudes (masks may have either sign).
    Returns the scale."""
    m, o = mask.astype(np.float64).ravel(), loss.astype(np.float64).ravel()
    want = np.array([(m * o).sum(), m.sum()])
    scale = np.maximum(np.array([np.abs(m * o).sum(), np.abs(m).sum()]), 1e-30)
    err = np.abs(np.asarray(got, np.float64) - want)
    assert (err <= 1e-5 * scale).all(), "%s: sums2 %r, float64 %r" % (what, list(got), list(want))
    return scale


# ---------------------------------------------------------------- chunk edges against the oracle
H_EDGE = 13   # W = 45: 585 floats per plane, so chunk c of a call starts 2340*i0 bytes in: not 16-byte aligned


@pytest.mark.gpu
@pytest.mark.parametrize("nch", (1, 2, 4, 16))
@pytest.mark.parametrize("B", (1, 3, 5, 17))
def test_host_imagewise_ops_at_chunk_edges(tx, B, nch):
    """Photometric (all four types through fwd, bwd, fwd_bwd and the masked call with and without a loss map; block 9
    and the generic block 5), LCN and XCorrVol (D = 6, C = 1 fast path and C = 2 generic path) with B images cut into
    `nch` chunks: fewer images than chunks, uneven splits, the 16-chunk cap."""
    L = _lib()
    pinned = nch in (2, 16)
    with host_options(host_chunks=nch):
        for C in (1, 2):
            for W in (72, 45):
                H = H_EDGE
                tag = "B %d, %d chunks, C %d, W %d" % (B, nch, C, W)
                rng = np.random.RandomState(1000 * B + 10 * nch + C + W)
                es = rng.randn(B, C, H, W).astype(np.float32)
                ta = (es + 0.7 * rng.randn(B, C, H, W)).astype(np.float32)
                go = rng.rand(B, 1, H, W).astype(np.float32)
                mk = rng.rand(B, 1, H, W).astype(np.float32)
                hes, hta, hgo, hmk = (_placed(x, pinned) for x in (es, ta, go, mk))
                hout, hgi, hs = HostBuf(B * H * W, np.float32, pinned), HostBuf(B * C * H * W, np.float32, pinned), HostBuf(2, np.float32, pinned)
                bufs = [hes, hta, hgo, hmk, hout, hgi, hs]
                for bs in (9, 5):
                    for ty in range(4):
                        what = "%s, block %d, type %d" % (tag, bs, ty)
                        f = oracle.photometric_loss_forward(es, ta, bs, ty, EPS)
                        g = oracle.photometric_loss_backward(es, ta, go, bs, ty, EPS)
                        args = (B, C, H, W, bs, ty, EPS)
                        hout.a[:] = 7.0
                        L.call("ctd_host_photometric_fwd_f32", hes.ptr(), hta.ptr(), hout.ptr(), *args)
                        assert_close(hout.a.reshape(f.shape), f, what="fwd " + what)
                        hgi.a[:] = 7.0
                        L.call("ctd_host_photometric_bwd_f32", hes.ptr(), hta.ptr(), hgo.ptr(), hgi.ptr(), *args)
                        assert_close(hgi.a.reshape(g.shape), g, what="bwd " + what)
                        hout.a[:] = 7.0
                        hgi.a[:] = 7.0
                        L.call("ctd_host_photometric_fwd_bwd_f32", hes.ptr(), hta.ptr(), hgo.ptr(), hout.ptr(), hgi.ptr(), *args)
                        assert_close(hout.a.reshape(f.shape), f, what="fwd_bwd out " + what)
                        assert_close(hgi.a.reshape(g.shape), g, what="fwd_bwd grad " + what)
                        for with_out in (False, True):
                            hout.a[:] = 7.0
                            hgi.a[:] = 7.0
                            L.call("ctd_host_photometric_fwd_bwd_masked_f32", hes.ptr(), hta.ptr(), hgo.ptr(), hmk.ptr(),
                                   hout.ptr() if with_out else None, hgi.ptr(), hs.ptr(), *args)
                            if with_out:
                                assert_close(hout.a.reshape(f.shape), f, what="masked out " + what)
                            else:
                                assert (hout.a == 7.0).all(), "masked call without a loss map wrote one: " + what
                            assert_close(hgi.a.reshape(g.shape), g, what="masked grad " + what)
                            _sums_close(hs.a, mk, f, "masked " + what)
                # XCorrVol: D not a multiple of 4 (C = 1: separable fast path, C = 2: generic kernel)
                D = 6
                hv = HostBuf(B * D * H * W, np.float32, pinned)
                hv.a[:] = 7.0
                L.call("ctd_host_xcorrvol_f32", hes.ptr(), hta.ptr(), hv.ptr(), B, C, H, W, D, 9)
                want = np.stack([oracle.xcorrvol(es[b], ta[b], D, 9) for b in range(B)])
                assert_close(hv.a.reshape(want.shape), want, what="xcorrvol " + tag)
                bufs.append(hv)
                if C == 1:
                    hl, hsd = HostBuf(B * H * W, np.float32, pinned), HostBuf(B * H * W, np.float32, pinned)
                    L.call("ctd_host_lcn_f32", hes.ptr(), hl.ptr(), hsd.ptr(), B, H, W, LCN_R, LCN_EPS)
                    lo, so = oracle.lcn(es, LCN_R, LCN_EPS)
                    assert_close(hl.a.reshape(lo.shape), lo, what="lcn " + tag)
                    assert_close(hsd.a.reshape(so.shape), so, what="lcn std " + tag)
                    bufs += [hl, hsd]
                assert all(b.margins_intact() for b in bufs), "a download wrote past its range: " + tag


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", (False, True))
def test_host_point_ops(tx, pinned):
    """ProjNN (fixed and generic patch sizes), NN (N1 below and above the split into in1 chunks) and CrossCheck on the
    ProjNN results, exact against the oracle."""
    from connecting_the_dots_b200 import synth
    L = _lib()
    B, H, W = 2, H_EDGE, 45
    xyz, K, poses = synth.make_clouds(B, H, W)
    x0 = np.ascontiguousarray(xyz)
    x01 = np.ascontiguousarray(np.stack([synth.transform(xyz[b], poses[1 - b]) for b in range(B)]))
    bufs = []
    with host_options():
        hx0, hx01, hK = _placed(x0, pinned), _placed(x01, pinned), _placed(K, pinned)
        i01, i10 = HostBuf(B * H * W, np.int64, pinned), HostBuf(B * H * W, np.int64, pinned)
        bufs += [hx0, hx01, hK, i01, i10]
        for ps in (3, 4):
            i01.a[:] = -5
            i10.a[:] = -5
            L.call("ctd_host_proj_nn_f32", hx01.ptr(), hx0.ptr(), hK.ptr(), i01.ptr(), B, H, W, ps)
            L.call("ctd_host_proj_nn_f32", hx0.ptr(), hx01.ptr(), hK.ptr(), i10.ptr(), B, H, W, ps)
            w01, w10 = oracle.proj_nn(x01, x0, K, ps), oracle.proj_nn(x0, x01, K, ps)
            assert np.array_equal(i01.a, w01.ravel()) and np.array_equal(i10.a, w10.ravel()), "proj_nn, patch %d" % ps
            assert (w01 >= 0).mean() > 0.5
            m = HostBuf(B * H * W, np.uint8, pinned)
            L.call("ctd_host_crosscheck", i01.ptr(), i10.ptr(), m.ptr(), B * H * W, B * H * W)
            want = oracle.crosscheck(w01.ravel(), w10.ravel())
            assert np.array_equal(m.a, want) and want.sum() > 0, "crosscheck, patch %d" % ps
            bufs.append(m)
        rng = np.random.RandomState(5)
        for N0, N1 in ((300, 700), (300, 5000), (1, 2049)):   # 5000, 2049: in1 is split over several blocks
            p0 = rng.rand(N0, 3).astype(np.float32)
            p1 = rng.rand(N1, 3).astype(np.float32)
            h0, h1, ho = _placed(p0, pinned), _placed(p1, pinned), HostBuf(N0, np.int64, pinned)
            L.call("ctd_host_nn_f32", h0.ptr(), h1.ptr(), ho.ptr(), N0, N1)
            assert np.array_equal(ho.a, oracle.nn(p0, p1)), "nn %d x %d" % (N0, N1)
            bufs += [h0, h1, ho]
    assert all(b.margins_intact() for b in bufs), "a download wrote past its range"


# ---------------------------------------------------------------- generated programs
# A region is (buffer, first element, element count).  Float buffers "f0".."f3" hold planes of H*W floats and are what
# LCN, the photometric calls and XCorrVol read and write; "p0", "p1" are point clouds (read-only) that ProjNN and NN
# read; "i0", "i1" are int64 index buffers that ProjNN and NN write and CrossCheck reads; "m0" takes CrossCheck's masks.
Region = collections.namedtuple("Region", "buf off n")
FLOATS, CLOUDS, INDICES = ("f0", "f1", "f2", "f3"), ("p0", "p1"), ("i0", "i1")
PATTERNS = ("exact_raw", "partial_raw", "wwr_exact", "wwr_partial", "rwwr", "in_place", "shared_input", "masked_no_out")


def _overlap(a, b):
    return a.buf == b.buf and a.off < b.off + b.n and b.off < a.off + a.n


class _Gen:
    """Seeded generator of one program: dims, and a list of calls (dicts) whose buffers alias on purpose."""

    def __init__(self, seed):
        rng = self.rng = np.random.RandomState(seed)
        self.H, self.W = [(16, 45), (20, 48), (24, 64), (64, 96)][rng.choice(4, p=[0.35, 0.3, 0.25, 0.1])]
        self.B = int(rng.randint(1, 6))
        self.D = 3
        self.P = self.H * self.W                      # floats per plane, a multiple of 4: device chunks stay aligned
        self.NP = max(2 * self.B, self.D * self.B) + 2   # planes per float buffer
        self.NI = self.B * self.P                     # points per cloud, entries per index / mask buffer
        self.calls, self.written, self.read = [], [], []
        n = int(rng.randint(6, 13))
        while len(self.calls) < n:
            room = n - len(self.calls)
            u = rng.rand()
            made = None
            if u < 0.15 and room >= 3:
                made = self._macro_write_write_read()
            elif u < 0.3 and room >= 4:
                made = self._macro_read_write_wait_read()
            else:
                for _ in range(20):
                    made = self._random_call()
                    if made:
                        break
            for c in made or ():
                self._add(c)

    # -- bookkeeping
    def _add(self, c):
        r, w = call_io(c)
        self.read += r
        self.written += w
        c["slot"] = sum(1 for x in self.calls if x["op"] == "photo" and x["kind"] == "masked") if c["op"] == "photo" else 0
        self.calls.append(c)

    def _fplanes(self, n_planes, buf=None):
        """a fresh float region of n_planes planes"""
        rng = self.rng
        buf = buf or FLOATS[rng.randint(len(FLOATS))]
        off = rng.randint(0, self.NP - n_planes + 1)
        return Region(buf, off * self.P, n_planes * self.P)

    def _pick(self, lst):
        return lst[self.rng.randint(len(lst))] if lst else None

    # -- float regions
    def _primary_read(self):
        """A float region the call reads first; the call's image count follows from it."""
        rng, P = self.rng, self.P
        w = [r for r in self.written if r.buf in FLOATS]
        rd = [r for r in self.read if r.buf in FLOATS]
        u = rng.rand()
        if w and u < 0.3:                                            # exact read after write
            return w[-1] if rng.rand() < 0.5 else self._pick(w)
        if w and u < 0.6:                                            # partial read after write
            r = w[-1] if rng.rand() < 0.5 else self._pick(w)
            v = rng.randint(3)
            if v == 0 and r.n > P:                                   # the first k images
                return Region(r.buf, r.off, P * rng.randint(1, r.n // P))
            if v == 1 and r.off + r.n + P <= self.NP * P:            # offset by one image
                return Region(r.buf, r.off + P, r.n)
            end = max(x.off + x.n for x in w if x.buf == r.buf)      # the whole span written in this buffer
            return Region(r.buf, 0, end)
        if rd and u < 0.75:                                          # an input shared with an earlier call
            return self._pick(rd)
        return self._fplanes(rng.randint(1, self.B + 1))

    def _same_size_read(self, n):
        rng = self.rng
        cand = [r for r in self.written + self.read if r.buf in FLOATS and r.n == n]
        if cand and rng.rand() < 0.5:
            return self._pick(cand)
        return self._fplanes(n // self.P)

    def _output(self, n, avoid, in_place=None):
        """A float region of n elements for a call output, disjoint from `avoid` (the call's other regions)."""
        rng = self.rng
        if in_place is not None:
            return in_place
        cand = []
        u = rng.rand()
        if u < 0.35:                                                  # overwrite an earlier output, whole or in part
            for r in self.written:
                if r.buf in FLOATS:
                    if r.n == n:
                        cand.append(r)
                    elif r.n > n:
                        cand.append(Region(r.buf, r.off, n))
        elif u < 0.6:                                                 # overwrite an earlier input
            cand = [r for r in self.read if r.buf in FLOATS and r.n == n]
        rng.shuffle(cand)
        cand += [self._fplanes(n // self.P) for _ in range(12)]
        for r in cand:
            if r.off + r.n <= self.NP * self.P and not any(_overlap(r, a) for a in avoid):
                return r
        return None

    def _random_call(self):
        rng, P = self.rng, self.P
        op = ("photo", "photo", "photo", "lcn", "xcorr", "proj_nn", "nn", "crosscheck")[rng.randint(8)]
        if op in ("photo", "lcn", "xcorr"):
            first = self._primary_read()
            planes = first.n // P
            C = 2 if op != "lcn" and planes % 2 == 0 and rng.rand() < 0.4 else 1
            nb = planes // C
            if op == "lcn":
                lcn = self._output(nb * P, [first])
                std = lcn and self._output(nb * P, [first, lcn])
                return std and [dict(op="lcn", nb=nb, x=first, lcn=lcn, std=std)]
            second = self._same_size_read(first.n)
            if op == "xcorr":
                if nb * self.D > self.NP:
                    return None
                out = self._output(nb * self.D * P, [first, second])
                return out and [dict(op="xcorr", nb=nb, C=C, bs=(9, 5)[rng.randint(2)], in0=first, in1=second, out=out)]
            kind = ("fwd", "bwd", "fwd_bwd", "masked")[rng.randint(4)]
            es, ta = (first, second) if rng.rand() < 0.5 else (second, first)
            go = self._same_size_read(nb * P) if kind != "fwd" else None
            mask = self._same_size_read(nb * P) if kind == "masked" else None
            ins = [x for x in (es, ta, go, mask) if x is not None]
            gi = out = None
            if kind != "fwd":
                gi = self._output(nb * C * P, ins, in_place=es if C == 1 and rng.rand() < 0.2 else None)
                if gi is None:
                    return None
            if kind in ("fwd", "fwd_bwd") or (kind == "masked" and rng.rand() < 0.5):
                out = self._output(nb * P, ins + [x for x in (gi,) if x is not None])
                if out is None:
                    return None
            if gi is not None and gi != es and any(_overlap(gi, x) for x in ins):
                return None
            return [dict(op="photo", kind=kind, nb=nb, C=C, bs=(9, 5)[rng.randint(2)], ty=int(rng.randint(4)),
                         es=es, ta=ta, go=go, mask=mask, out=out, gi=gi)]
        NI = self.NI
        if op == "proj_nn":
            nbp = int(rng.randint(1, self.B + 1))
            o0, o1 = (P * rng.randint(0, self.B - nbp + 1) for _ in range(2))
            x0, x1 = Region(self._pick(CLOUDS), o0, nbp * P), Region(self._pick(CLOUDS), o1, nbp * P)
            return [dict(op="proj_nn", nbp=nbp, xyz0=x0, xyz1=x1, out=self._index_out(nbp * P))]
        if op == "nn":
            N0, N1 = int(rng.randint(1, min(NI, 1500) + 1)), int(rng.randint(1, min(NI, 3000) + 1))
            x0 = Region(self._pick(CLOUDS), int(rng.randint(0, NI - N0 + 1)), N0)
            x1 = Region(self._pick(CLOUDS), int(rng.randint(0, NI - N1 + 1)), N1)
            return [dict(op="nn", in0=x0, in1=x1, out=self._index_out(N0))]
        # crosscheck: in1 is a whole index buffer (every index an index buffer can hold is in range), in0 any part of one
        w = [r for r in self.written if r.buf in INDICES]
        if w and rng.rand() < 0.6:
            r = self._pick(w)
            in0 = r if rng.rand() < 0.5 else Region(r.buf, r.off, int(rng.randint(1, r.n + 1)))
        else:
            N0 = int(rng.randint(1, NI + 1))
            in0 = Region(self._pick(INDICES), int(rng.randint(0, NI - N0 + 1)), N0)
        in1 = Region(self._pick(INDICES), 0, NI)
        out = Region("m0", int(rng.randint(0, NI - in0.n + 1)), in0.n)
        return [dict(op="crosscheck", in0=in0, in1=in1, out=out)]

    def _index_out(self, n):
        rng = self.rng
        w = [r for r in self.written if r.buf in INDICES and r.n >= n]
        if w and rng.rand() < 0.4:
            r = self._pick(w)
            return Region(r.buf, r.off, n)
        return Region(self._pick(INDICES), int(rng.randint(0, self.NI - n + 1)), n)

    # -- the two hazards as call patterns
    def _macro_write_write_read(self):
        """LCN writes X, a second LCN writes X again (whole or its first images), a masked loss reads X."""
        rng, P = self.rng, self.P
        nb = int(rng.randint(2, self.B + 2))
        X = self._fplanes(nb)
        S = self._output(nb * P, [X])
        src = self._output(nb * P, [X, S])
        if S is None or src is None:
            return None
        k = nb if rng.rand() < 0.5 else int(rng.randint(1, nb))
        X2 = Region(X.buf, X.off, k * P)
        src2, S2 = self._output(k * P, [X, S, src]), self._output(k * P, [X, S, src])
        if src2 is None or S2 is None or _overlap(src2, S2):
            return None
        es = self._output(nb * P, [X, S])
        gi = es and self._output(nb * P, [X, S, es])
        if gi is None:
            return None
        return [dict(op="lcn", nb=nb, x=src, lcn=X, std=S),
                dict(op="lcn", nb=k, x=src2, lcn=X2, std=S2),
                dict(op="photo", kind="masked", nb=nb, C=1, bs=9, ty=int(rng.randint(4)), es=es, ta=X, go=S, mask=S,
                     out=None, gi=gi)]

    def _macro_read_write_wait_read(self):
        """A loss reads E; LCN overwrites E; a read one image longer than an output in flight forces a wait; the loss
        reads E again."""
        rng, P = self.rng, self.P
        nb = int(rng.randint(1, self.B + 1))
        E = self._fplanes(nb)
        if E.off + E.n + P > self.NP * P:
            return None
        T = self._output(nb * P, [E])
        O1 = T and self._output(nb * P, [E, T])
        src = O1 and self._output(nb * P, [E, T, O1])
        S = src and self._output(nb * P, [E, T, O1, src])
        if S is None or S.off + S.n + P > self.NP * P:
            return None
        wide = Region(S.buf, S.off, S.n + P)            # one image longer than LCN's std output
        L2 = self._output(wide.n, [wide, E, T, O1, src, S])
        S2 = L2 and self._output(wide.n, [wide, E, T, O1, src, S, L2])
        O2 = S2 and self._output(nb * P, [E, T, O1, src, S, L2, S2])
        if O2 is None:
            return None
        ty, bs = int(rng.randint(4)), (9, 5)[rng.randint(2)]
        return [dict(op="photo", kind="fwd", nb=nb, C=1, bs=bs, ty=ty, es=E, ta=T, go=None, mask=None, out=O1, gi=None),
                dict(op="lcn", nb=nb, x=src, lcn=E, std=S),
                dict(op="lcn", nb=nb + 1, x=wide, lcn=L2, std=S2),
                dict(op="photo", kind="fwd", nb=nb, C=1, bs=bs, ty=ty, es=E, ta=T, go=None, mask=None, out=O2, gi=None)]


def call_io(c):
    """(regions read, regions written) of a call, sums2 excluded (it is never an input)."""
    op = c["op"]
    if op == "photo":
        return [x for x in (c["es"], c["ta"], c["go"], c["mask"]) if x is not None], [x for x in (c["out"], c["gi"]) if x is not None]
    if op == "lcn":
        return [c["x"]], [c["lcn"], c["std"]]
    if op == "xcorr":
        return [c["in0"], c["in1"]], [c["out"]]
    if op == "proj_nn":
        return [c["xyz0"], c["xyz1"]], [c["out"]]
    return [c["in0"], c["in1"]], [c["out"]]


def gen_program(seed):
    return _Gen(seed)


def classify(prog):
    """Set of PATTERNS a program contains, from its calls alone."""
    found = set()
    writes = []                               # (call index, region), in order
    reads = []
    partial_at = []                           # call indices with a partial read after write
    for i, c in enumerate(prog.calls):
        r, w = call_io(c)
        for x in r:
            over = [(j, y) for j, y in writes if _overlap(x, y)]
            if over:
                newest = over[-1][1]
                if newest == x:
                    found.add("exact_raw")
                else:
                    found.add("partial_raw")
                    partial_at.append(i)
                if len(over) >= 2 and over[-2][1] == x:
                    found.add("wwr_exact" if newest == x else "wwr_partial")
            for j, y in reads:
                if y == x and j < i and not any(_overlap(x, z) for k, z in writes if k > j):
                    found.add("shared_input")
                if y == x and j < i:
                    between = [k for k, z in writes if j < k < i and _overlap(x, z)]
                    if between and any(between[0] < p < i for p in partial_at):
                        found.add("rwwr")
        if c["op"] == "photo":
            if c["gi"] is not None and c["gi"] == c["es"]:
                found.add("in_place")
            if c["kind"] == "masked" and c["out"] is None:
                found.add("masked_no_out")
        reads += [(i, x) for x in r]
        writes += [(i, y) for y in w]
    return found


def test_program_generator_covers_every_aliasing_pattern():
    """Over the seeds the GPU test runs, every aliasing pattern occurs in several programs, and every program is
    well formed (no call's outputs overlap each other or its inputs, except the exact in-place gradient)."""
    count = collections.Counter()
    for s in SEEDS:
        g = gen_program(s)
        assert 6 <= len(g.calls) <= 12
        for c in g.calls:
            r, w = call_io(c)
            for i, a in enumerate(w):
                assert a.n > 0 and a.off >= 0
                for b in w[i + 1:] + r:
                    assert not _overlap(a, b) or (c["op"] == "photo" and a == c["gi"] == c["es"] == b and c["C"] == 1), c
        count.update(classify(g))
    for p in PATTERNS:
        assert count[p] >= 3, (p, dict(count))


# ---- running a program
def _make_pool(g, pinned=True):
    from connecting_the_dots_b200 import synth
    P, NI = g.P, g.NI
    pool = {b: HostBuf(g.NP * P, np.float32, pinned) for b in FLOATS}
    xyz, K, poses = synth.make_clouds(g.B, g.H, g.W)
    pool["p0"] = _placed(xyz, pinned)
    pool["p1"] = _placed(np.stack([synth.transform(xyz[b], poses[(b + 1) % g.B]) for b in range(g.B)]), pinned)
    pool["K"] = _placed(K, pinned)
    for b in INDICES:
        pool[b] = HostBuf(NI, np.int64, pinned)
    pool["m0"] = HostBuf(NI, np.uint8, pinned)
    pool["s"] = HostBuf(2 * 12, np.float32, pinned)
    return pool


def _fill(g, pool, seed):
    """Fresh contents for every buffer a program may read or write (clouds and K stay)."""
    rng = np.random.RandomState(seed)
    for b in FLOATS:
        pool[b].a[:] = rng.randn(pool[b].a.size)
    for b in INDICES:
        pool[b].a[:] = rng.randint(-1, g.NI, g.NI)
    pool["m0"].a[:] = rng.randint(0, 256, g.NI)
    pool["s"].a[:] = rng.randn(pool["s"].a.size)


def _ptr(pool, r, g):
    if r is None:
        return None
    if r.buf in CLOUDS:
        return pool[r.buf].ptr(3 * r.off)        # clouds: regions count points
    return pool[r.buf].ptr(r.off)


def _issue(g, pool, c):
    L, H, W = _lib(), g.H, g.W
    p = lambda r: _ptr(pool, r, g)
    op = c["op"]
    if op == "photo":
        args = (c["nb"], c["C"], H, W, c["bs"], c["ty"], EPS)
        kind = c["kind"]
        if kind == "fwd":
            L.call("ctd_host_photometric_fwd_f32", p(c["es"]), p(c["ta"]), p(c["out"]), *args)
        elif kind == "bwd":
            L.call("ctd_host_photometric_bwd_f32", p(c["es"]), p(c["ta"]), p(c["go"]), p(c["gi"]), *args)
        elif kind == "fwd_bwd":
            L.call("ctd_host_photometric_fwd_bwd_f32", p(c["es"]), p(c["ta"]), p(c["go"]), p(c["out"]), p(c["gi"]), *args)
        else:
            L.call("ctd_host_photometric_fwd_bwd_masked_f32", p(c["es"]), p(c["ta"]), p(c["go"]), p(c["mask"]), p(c["out"]),
                   p(c["gi"]), pool["s"].ptr(2 * c["slot"]), *args)
    elif op == "lcn":
        L.call("ctd_host_lcn_f32", p(c["x"]), p(c["lcn"]), p(c["std"]), c["nb"], H, W, LCN_R, LCN_EPS)
    elif op == "xcorr":
        L.call("ctd_host_xcorrvol_f32", p(c["in0"]), p(c["in1"]), p(c["out"]), c["nb"], c["C"], H, W, g.D, c["bs"])
    elif op == "proj_nn":
        L.call("ctd_host_proj_nn_f32", p(c["xyz0"]), p(c["xyz1"]), pool["K"].ptr(), p(c["out"]), c["nbp"], H, W, 3)
    elif op == "nn":
        L.call("ctd_host_nn_f32", p(c["in0"]), p(c["in1"]), p(c["out"]), c["in0"].n, c["in1"].n)
    else:
        L.call("ctd_host_crosscheck", p(c["in0"]), p(c["in1"]), p(c["out"]), c["in0"].n, c["in1"].n)


def _view(snap, r, g, shape=None):
    """contents of region r in a snapshot {buffer: raw array}"""
    k = 3 if r.buf in CLOUDS else 1
    a = snap[r.buf][PAD + k * r.off:PAD + k * (r.off + r.n)]
    return a.reshape(shape) if shape else a


def _check_call(g, c, snap, pool, what, scales):
    """Outputs of call c against the oracle on its inputs as they were before the call (snap), and no other byte
    of any buffer changed.  scales[slot] = the magnitude of a masked call's sums (see _sums_close)."""
    H, W, P = g.H, g.W, g.P
    now = {b: h.raw for b, h in pool.items()}
    op = c["op"]
    if op == "photo":
        nb, C = c["nb"], c["C"]
        es, ta = _view(snap, c["es"], g, (nb, C, H, W)), _view(snap, c["ta"], g, (nb, C, H, W))
        f = oracle.photometric_loss_forward(es, ta, c["bs"], c["ty"], EPS) if c["out"] is not None or c["kind"] == "masked" else None
        if c["out"] is not None:
            assert_close(_view(now, c["out"], g, (nb, 1, H, W)), f, what=what + ": loss map")
        if c["gi"] is not None:
            go = _view(snap, c["go"], g, (nb, 1, H, W))
            assert_close(_view(now, c["gi"], g, (nb, C, H, W)), oracle.photometric_loss_backward(es, ta, go, c["bs"], c["ty"], EPS),
                         what=what + ": gradient")
        if c["kind"] == "masked":
            scales[c["slot"]] = _sums_close(pool["s"].a[2 * c["slot"]:2 * c["slot"] + 2], _view(snap, c["mask"], g), f, what)
    elif op == "lcn":
        lo, so = oracle.lcn(_view(snap, c["x"], g, (c["nb"], 1, H, W)), LCN_R, LCN_EPS)
        assert_close(_view(now, c["lcn"], g, lo.shape), lo, what=what + ": lcn")
        assert_close(_view(now, c["std"], g, so.shape), so, what=what + ": std")
    elif op == "xcorr":
        nb, C, D = c["nb"], c["C"], g.D
        i0, i1 = _view(snap, c["in0"], g, (nb, C, H, W)), _view(snap, c["in1"], g, (nb, C, H, W))
        want = np.stack([oracle.xcorrvol(i0[b], i1[b], D, c["bs"]) for b in range(nb)])
        assert_close(_view(now, c["out"], g, want.shape), want, what=what + ": volume")
    elif op == "proj_nn":
        nbp = c["nbp"]
        want = oracle.proj_nn(_view(snap, c["xyz0"], g, (nbp, H, W, 3)), _view(snap, c["xyz1"], g, (nbp, H, W, 3)),
                              pool["K"].a.reshape(3, 3), 3)
        assert np.array_equal(_view(now, c["out"], g), want.ravel()), what + ": indices"
    elif op == "nn":
        want = oracle.nn(_view(snap, c["in0"], g, (-1, 3)), _view(snap, c["in1"], g, (-1, 3)))
        assert np.array_equal(_view(now, c["out"], g), want), what + ": indices"
    else:
        want = oracle.crosscheck(_view(snap, c["in0"], g), _view(snap, c["in1"], g))
        assert np.array_equal(_view(now, c["out"], g), want), what + ": mask"
    allowed = {b: np.zeros(h.raw.size, bool) for b, h in pool.items()}
    for r in call_io(c)[1]:
        allowed[r.buf][PAD + r.off:PAD + r.off + r.n] = True
    if op == "photo" and c["kind"] == "masked":
        allowed["s"][PAD + 2 * c["slot"]:PAD + 2 * c["slot"] + 2] = True
    for b, h in pool.items():
        bad = np.flatnonzero(_differs(h.raw, snap[b]) & ~allowed[b])
        assert bad.size == 0, "%s: wrote %s outside its outputs (element %d)" % (what, b, bad[0] - PAD)


def _differs(x, y):
    """per element: do the bytes of x and y differ (NaN-safe)"""
    return (x.view(np.uint8).reshape(x.size, -1) != y.view(np.uint8).reshape(y.size, -1)).any(axis=1)


def _snapshot(pool):
    return {b: h.raw.copy() for b, h in pool.items()}


def _sequential(g, pool, seed, check):
    """The program's calls one at a time from fresh contents: (final contents, {sums slot: magnitude} when checked)."""
    _fill(g, pool, seed)
    scales = {}
    for i, c in enumerate(g.calls):
        snap = _snapshot(pool) if check else None
        _issue(g, pool, c)
        if check:
            _check_call(g, c, snap, pool, "call %d (%s)" % (i, c["op"] if c["op"] != "photo" else c["kind"]), scales)
    return _snapshot(pool), scales


def _compare(g, got, expected, exact, what):
    """every buffer of `got` against the contents the calls made one at a time left (expected = (contents, sums
    magnitudes)): bit-equal, or (exact=False) floats per plane to the oracle tolerance, each sums2 pair within 2e-5 of
    its magnitude (both sides are within 1e-5 of the float64 sums), integers, margins and unused sums slots bit-equal"""
    want, scales = expected
    for b in want:
        x, y = got[b], want[b]
        if exact or x.dtype != np.float32:
            d = np.flatnonzero(_differs(x, y))
            if d.size:
                i = int(d[0])
                raise AssertionError("%s: buffer %s differs from the calls made one at a time at element %d: %r, want %r"
                                     % (what, b, i - PAD, x[i], y[i]))
            continue
        assert np.array_equal(x[:PAD], y[:PAD]) and np.array_equal(x[x.size - PAD:], y[y.size - PAD:]), what + ": margins of " + b
        if b == "s":
            for j in range(12):
                xs, ys = x[PAD + 2 * j:PAD + 2 * j + 2], y[PAD + 2 * j:PAD + 2 * j + 2]
                if j in scales:
                    assert (np.abs(xs.astype(np.float64) - ys) <= 2e-5 * scales[j]).all(), "%s: sums2 of slot %d" % (what, j)
                else:
                    assert np.array_equal(xs, ys), "%s: unused sums slot %d" % (what, j)
            continue
        for k in range(g.NP):
            sl = slice(PAD + k * g.P, PAD + (k + 1) * g.P)
            assert_close(x[sl], y[sl], what="%s: buffer %s, plane %d" % (what, b, k))


def _chunks(n, k):
    nch = min(max(n, 1), min(max(k, 1), 16))
    return [(n * c // nch, n * (c + 1) // nch) for c in range(nch)]


def _has_partial_overlap(g, k):
    """Whether some upload of the batch overlaps a download still in flight without matching it exactly (the newest such
    download decides): the library then waits, which a graph capture cannot do.  Mirrors the chunking of host_api.cu."""
    P = g.P
    pending = []
    for c in g.calls:
        op = c["op"]
        steps = []                                     # per chunk: (reads, writes)
        if op in ("photo", "lcn", "xcorr"):
            nb = c["nb"]
            if op == "photo":
                C = c["C"]
                rd = [(c["es"], C), (c["ta"], C)] + ([(c["go"], 1)] if c["gi"] is not None else []) + \
                     ([(c["mask"], 1)] if c["kind"] == "masked" else [])
                wr = [(c["out"], 1)] * (c["out"] is not None) + [(c["gi"], C)] * (c["gi"] is not None)
            elif op == "lcn":
                rd, wr = [(c["x"], 1)], [(c["lcn"], 1), (c["std"], 1)]
            else:
                rd, wr = [(c["in0"], c["C"]), (c["in1"], c["C"])], [(c["out"], g.D)]
            for i0, i1 in _chunks(nb, k):
                sub = lambda r, pl: Region(r.buf, r.off + i0 * pl * P, (i1 - i0) * pl * P)
                steps.append(([sub(r, pl) for r, pl in rd], [sub(r, pl) for r, pl in wr]))
        else:
            r, w = call_io(c)
            steps.append(([x for x in r if x.buf not in CLOUDS], w))
        for rd, wr in steps:
            for x in rd:
                for p in reversed(pending):
                    if _overlap(p, x):
                        if p != x:
                            return True
                        break
            pending += wr
    return False


@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS)
def test_generated_batches_match_sequential_calls(tx, seed):
    """One program, four ways: calls one at a time (each checked against the oracle), one batch, a batch repeated under
    graph replay (eager, capture, replay, replay: fresh inputs every time), and batches two in flight over three buffer
    pools.  Bit-equal where every mode cuts the same chunks, within the oracle's tolerance at the default options."""
    g = gen_program(seed)
    L = _lib()
    pool = _make_pool(g)
    pools = [pool, _make_pool(g), _make_pool(g)]
    for k in SETTINGS:
        opts = dict(host_chunks=k, host_chunks_batch=k, host_chunks_graph=k) if k else {}
        exact = k is not None
        tag = "seed %d, %s" % (seed, "%d chunks" % k if k else "default chunks")
        with host_options(**opts):
            fills = [seed * 1000 + 17 * (k or 0) + rep for rep in range(4)]
            # checked against the oracle once; at the default options every repetition, for the magnitudes of its sums
            want = [_sequential(g, pool, f, check=(rep == 0 or not exact)) for rep, f in enumerate(fills)]
            # one deferred batch
            _fill(g, pool, fills[0])
            L.call("ctd_host_begin_batch")
            for c in g.calls:
                _issue(g, pool, c)
            L.call("ctd_host_end_batch")
            _compare(g, _snapshot(pool), want[0], exact, tag + ", one batch")
        with host_options(host_graphs=1, **opts):
            base = graph_stats()
            partial = _has_partial_overlap(g, k or 2)
            for rep in range(4):
                _fill(g, pool, fills[rep])
                L.call("ctd_host_begin_batch")
                for c in g.calls:
                    _issue(g, pool, c)
                L.call("ctd_host_end_batch")
                _compare(g, _snapshot(pool), want[rep], exact, tag + ", graph mode, repetition %d" % rep)
                got = tuple(x - y for x, y in zip(graph_stats(), base))
                expect = ((0, 0, 0), (0, 0, 1), (0, 0, 1), (0, 0, 1)) if partial else ((0, 0, 0), (1, 1, 0), (1, 2, 0), (1, 3, 0))
                assert got == expect[rep], "%s, repetition %d: graph stats %r, want %r (partial overlap: %s)" % (
                    tag, rep, got, expect[rep], partial)
        with host_options(**opts):
            inflight = []
            for step in range(4):
                p = pools[step % 3]
                _fill(g, p, fills[step])
                L.call("ctd_host_begin_batch")
                for c in g.calls:
                    _issue(g, p, c)
                L.call("ctd_host_end_batch_async")
                inflight.append((step, p))
                if len(inflight) == 2:
                    L.call("ctd_host_wait_batch")
                    s, q = inflight.pop(0)
                    _compare(g, _snapshot(q), want[s], exact, tag + ", two in flight, step %d" % s)
            L.call("ctd_host_wait_batch")
            s, q = inflight.pop(0)
            _compare(g, _snapshot(q), want[s], exact, tag + ", two in flight, step %d" % s)
    for p in pools:
        assert all(h.margins_intact() for h in p.values()), "seed %d: a download wrote past its range" % seed


# ---------------------------------------------------------------- the two hazards as fixed batches
def _regression_pool(B, H, W):
    rng = np.random.RandomState(77)
    pin = lambda a: _placed(a, True)
    h = {k: pin(rng.randn(B, 1, H, W).astype(np.float32)) for k in ("imA", "imB", "es", "ta", "go", "E")}
    for k in ("L", "S", "gi", "out1", "out2"):
        h[k] = HostBuf(B * H * W, np.float32, True)
    for k in ("wide", "L3", "S3"):   # B + 1 images
        h[k] = HostBuf((B + 1) * H * W, np.float32, True)
    h["sums"] = HostBuf(2, np.float32, True)
    return h


def _in_modes(prepare, run, check):
    """prepare(); run() as a deferred batch; check(), once, then four times with host_graphs = 1 (eager, capture,
    replay, replay)."""
    L = _lib()
    with host_options():
        prepare()
        L.call("ctd_host_begin_batch")
        run()
        L.call("ctd_host_end_batch")
        check("one batch")
    with host_options(host_graphs=1):
        for rep in range(4):
            prepare()
            L.call("ctd_host_begin_batch")
            run()
            L.call("ctd_host_end_batch")
            check("graph mode, repetition %d" % rep)


@pytest.mark.gpu
@pytest.mark.parametrize("newer", ("whole", "first_image"))
def test_batch_write_write_read_reads_the_newest_write(tx, newer):
    """lcn(imA -> L, S); lcn(imB -> L, S) (whole, or its first image only); masked loss with ta = L, mask = S.  The loss
    must see what the second LCN left in L and S, as the same calls made one at a time do."""
    B, H, W = 2, 32, 48
    h = _regression_pool(B, H, W)
    L = _lib()
    nb2 = B if newer == "whole" else 1
    P = lambda k: h[k].ptr()

    def prepare():
        for k in ("L", "S", "gi"):
            h[k].a[:] = 7.0

    def run():
        L.call("ctd_host_lcn_f32", P("imA"), P("L"), P("S"), B, H, W, LCN_R, LCN_EPS)
        L.call("ctd_host_lcn_f32", P("imB"), P("L"), P("S"), nb2, H, W, LCN_R, LCN_EPS)
        L.call("ctd_host_photometric_fwd_bwd_masked_f32", P("es"), P("L"), P("go"), P("S"), None, P("gi"), P("sums"),
               B, 1, H, W, 9, 3, EPS)

    imA, imB = (h[k].a.reshape(B, 1, H, W) for k in ("imA", "imB"))
    la, sa = oracle.lcn(imA, LCN_R, LCN_EPS)
    lb, sb = oracle.lcn(imB[:nb2], LCN_R, LCN_EPS)
    lw, sw = la.copy(), sa.copy()
    lw[:nb2], sw[:nb2] = lb, sb
    es, go = h["es"].a.reshape(B, 1, H, W), h["go"].a.reshape(B, 1, H, W)

    def check(mode):
        # L and S as the library computed them, checked against the oracle, are the loss's inputs: the loss is then
        # compared with the oracle on exactly those bytes (a stale L or S gives another loss, far outside 1e-5)
        Lb, Sb = h["L"].a.reshape(lw.shape), h["S"].a.reshape(sw.shape)
        assert_close(Lb, lw, what=mode + ": L")
        assert_close(Sb, sw, what=mode + ": S")
        gw = oracle.photometric_loss_backward(es, Lb, go, 9, 3, EPS)
        assert_close(h["gi"].a.reshape(gw.shape), gw, what=mode + ": loss gradient on the newest L (stale L read?)")
        _sums_close(h["sums"].a, Sb, oracle.photometric_loss_forward(es, Lb, 9, 3, EPS), mode + ": sums on the newest S")
        assert all(x.margins_intact() for x in h.values())

    _in_modes(prepare, run, check)


@pytest.mark.gpu
def test_batch_read_write_wait_read_uploads_again(tx):
    """photometric_fwd(es = E); lcn(imA -> lcn = E, std = the first B images of Y); lcn reading all B + 1 images of Y (it
    overlaps the std download still in flight, so the batch waits for the downloads); photometric_fwd(es = E) again.  The
    last call must see E as the LCN left it, not the device copy of E that the first call uploaded."""
    B, H, W = 2, 32, 48
    h = _regression_pool(B, H, W)
    L = _lib()
    P = lambda k: h[k].ptr()
    E0, Y0 = h["E"].a.copy(), np.random.RandomState(78).randn(h["wide"].a.size).astype(np.float32)

    def prepare():
        h["E"].a[:] = E0
        h["wide"].a[:] = Y0
        for k in ("out1", "out2", "L3", "S3"):
            h[k].a[:] = 7.0

    def run():
        L.call("ctd_host_photometric_fwd_f32", P("E"), P("ta"), P("out1"), B, 1, H, W, 9, 1, EPS)
        L.call("ctd_host_lcn_f32", P("imA"), P("E"), P("wide"), B, H, W, LCN_R, LCN_EPS)
        L.call("ctd_host_lcn_f32", P("wide"), P("L3"), P("S3"), B + 1, H, W, LCN_R, LCN_EPS)
        L.call("ctd_host_photometric_fwd_f32", P("E"), P("ta"), P("out2"), B, 1, H, W, 9, 1, EPS)

    ta = h["ta"].a.reshape(B, 1, H, W)
    la, sa = oracle.lcn(h["imA"].a.reshape(B, 1, H, W), LCN_R, LCN_EPS)
    want1 = oracle.photometric_loss_forward(E0.reshape(B, 1, H, W), ta, 9, 1, EPS)

    def check(mode):
        # what the LCN wrote (E, the first B images of Y), checked against the oracle, is what the later calls read:
        # they are compared with the oracle on exactly those bytes.  LCN of a std map divides small local deviations
        # by a small local std, so the oracle's own std would be no fair input for the third call at 1e-5.
        E, Y = h["E"].a.reshape(la.shape), h["wide"].a.reshape(B + 1, 1, H, W)
        assert_close(h["out1"].a.reshape(want1.shape), want1, what=mode + ": loss on E before the LCN")
        assert_close(E, la, what=mode + ": E written by the LCN")
        assert_close(Y[:B], sa, what=mode + ": std written by the LCN")
        assert np.array_equal(Y[B:].ravel(), Y0[B * H * W:]), mode + ": the image of Y after the std output changed"
        l3, _ = oracle.lcn(Y, LCN_R, LCN_EPS)
        assert_close(h["L3"].a.reshape(l3.shape), l3, what=mode + ": lcn of the std written in the same batch")
        want2 = oracle.photometric_loss_forward(E, ta, 9, 1, EPS)
        assert_close(h["out2"].a.reshape(want2.shape), want2, what=mode + ": loss on E after the LCN (stale upload of E?)")
        assert all(x.margins_intact() for x in h.values())

    _in_modes(prepare, run, check)
