#!/usr/bin/env python
"""Per-op device timings of every kernel family on the BASELINE.json configs (CUDA events on the
launching stream, rotating buffer sets larger than L2 where the op is HBM-bound).  Prints one JSON
object; bench.py stays the contract benchmark, this is the per-op table that goes into profiles/.

    python tools/bench_ops.py [--iters 30] [--only photometric,ssim,lcn,xcorrvol,xcorr_disparity,sgm,census_match,disparity_check,speckle,proj_nn,nn,crosscheck]

The printed result names the GPU and its power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))  # losses_torch: comparison legs only (torch formulation of the reference)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import connecting_the_dots_b200 as ctd  # noqa: E402
from connecting_the_dots_b200 import _lib, synth  # noqa: E402

H, W = 480, 640
PEAK = 6453.4
try:
    PEAK = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
except Exception:
    pass


NREP = 10  # launches per graph replay (cycling over the buffer sets)


def timeit(fn, iters, warmup=5, nrep=NREP):
    """fn(i, stream_handle) enqueues launch i.  nrep launches are captured into one CUDA graph and the graph
    is replayed `iters` times between events, so host launch latency is not part of the figure; returns the
    per-launch (median, min) in ms."""
    cur = torch.cuda.current_stream()
    for i in range(warmup):
        fn(i, cur.cuda_stream)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        cs = torch.cuda.current_stream().cuda_stream
        for i in range(nrep):
            fn(i, cs)
    g.replay()
    torch.cuda.synchronize()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(iters + 1)]
    evs[0].record()
    for i in range(iters):
        g.replay()
        evs[i + 1].record()
    torch.cuda.synchronize()
    ts = [evs[i].elapsed_time(evs[i + 1]) / nrep for i in range(iters)]
    return float(np.median(ts)), float(np.min(ts))


def device_info(index):
    """Name and power limit of the GPU the timings are taken on (nvidia-smi only reads them)."""
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        info["nvidia_smi"] = out
    except Exception as e:  # the timings stand without it, but say why it is missing
        info["nvidia_smi"] = "unavailable: %s" % e
    return info


def census_traffic(B, C, H, W, D):
    """Least HBM bytes of the census calls, from shapes: the volume writes 4 B per pixel and disparity and reads both fp32
    inputs; the fused disparity reads the inputs and writes disp and score (16 B/px at C = 1)."""
    npx = B * H * W
    return {"volume": (4 * D + 8 * C) * npx, "disparity": (8 * C + 8) * npx}


ALL = "calib,photometric,ssim,warp,pyramid,geometric,disparity,lcn,xcorrvol,xcorr_disparity,sgm,census_match,disparity_check,speckle,proj_nn,config4,nn,crosscheck,reduce,gpu_reference"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--only", default=ALL)
    ap.add_argument("--batch", type=int, default=8)
    args = ap.parse_args()
    res = run(args.only, args.iters, args.batch)
    res["device"] = device_info(0)
    print(json.dumps(res))


def run(only=ALL, iters=30, batch=8, device_index=0, verbose=True):
    """Times the selected op families and returns the result dict (bench.py calls this for the ops beyond its step)."""
    import types
    args = types.SimpleNamespace(iters=iters, batch=batch)
    only = set(only.split(","))
    dev = torch.device("cuda", device_index)
    tx = ctd.torchext
    B = args.batch
    npx = B * H * W
    res = {"batch": B, "height": H, "width": W, "peak_gbs": PEAK, "ops": {}}

    def add(name, ms, ms_min, bytes_, px=npx, extra=None):
        r = {"ms_median": ms, "ms_min": ms_min, "mpix_s": px / ms / 1e3, "algo_bytes": bytes_,
             "achieved_gbs": bytes_ / ms / 1e6, "frac_hbm": bytes_ / ms / 1e6 / PEAK}
        if extra:
            r.update(extra)
        res["ops"][name] = r
        if verbose:
            print(name, json.dumps(r), file=sys.stderr, flush=True)

    NS = 5
    base = synth.make_batch(B, H, W)
    sets = []
    for s in range(NS):
        d = {k: torch.from_numpy(np.ascontiguousarray(np.roll(base[k], 5 * s, axis=2))).to(dev) for k in ("im", "es", "ta", "go", "std", "pat_lcn", "disp")}
        d["o1"] = torch.empty(B, 1, H, W, device=dev)
        d["o2"] = torch.empty(B, 1, H, W, device=dev)
        sets.append(d)

    if "calib" in only:
        # what the memory system delivers at THIS problem size (launch ramp + tail included): a plain
        # 2-reads-1-write elementwise pass and a 1-read-1-write copy over the same tensors, torch kernels
        def f(i, st):
            d = sets[i % NS]
            torch.add(d["es"], d["ta"], out=d["o1"])  # torch launches on the current (capture) stream
        add("calib_add_2r1w", *timeit(f, args.iters), 12 * npx)
        def f(i, st):
            d = sets[i % NS]
            d["o1"].copy_(d["es"])
        add("calib_copy_1r1w", *timeit(f, args.iters), 8 * npx)
    if "photometric" in only:
        for ty, name in enumerate(("mse", "sad", "census_mse", "census_sad")):
            def f(i, st, ty=ty):
                d = sets[i % NS]
                _lib.call("ctd_photometric_fwd_f32", d["es"].data_ptr(), d["ta"].data_ptr(), d["o1"].data_ptr(), B, 1, H, W, 9, ty, 0.5, st)
            def g(i, st, ty=ty):
                d = sets[i % NS]
                _lib.call("ctd_photometric_bwd_f32", d["es"].data_ptr(), d["ta"].data_ptr(), d["go"].data_ptr(), d["o2"].data_ptr(), B, 1, H, W, 9, ty, 0.5, st)
            add(name + "_fwd", *timeit(f, args.iters), 12 * npx)
            add(name + "_bwd", *timeit(g, args.iters), 16 * npx)
    if "ssim" in only:
        # the SSIM loss (ssim.cu) at block 3 and 9: forward, backward, and the fused forward + backward + masked sums, against
        # the usual torch formulation on the same GPU (avg_pool2d window moments over a replicate-padded copy, autograd backward)
        gis = [torch.empty(B, 1, H, W, device=dev) for _ in range(NS)]
        sums = torch.zeros(2, device=dev)
        c1, c2 = tx.SSIM_C1, tx.SSIM_C2
        for bs in (3, 9):
            def f(i, st, bs=bs):
                d = sets[i % NS]
                _lib.call("ctd_ssim_fwd_f32", d["es"].data_ptr(), d["ta"].data_ptr(), d["o1"].data_ptr(), B, 1, H, W, bs, c1, c2, st)
            def g(i, st, bs=bs):
                d = sets[i % NS]
                _lib.call("ctd_ssim_bwd_f32", d["es"].data_ptr(), d["ta"].data_ptr(), d["go"].data_ptr(), d["o2"].data_ptr(), B, 1, H, W, bs,
                          c1, c2, st)
            def h(i, st, bs=bs):
                d = sets[i % NS]
                _lib.call("ctd_ssim_fwd_bwd_masked_f32", d["es"].data_ptr(), d["ta"].data_ptr(), d["std"].data_ptr(), d["std"].data_ptr(),
                          d["o1"].data_ptr(), gis[i % NS].data_ptr(), sums.data_ptr(), B, 1, H, W, bs, c1, c2, st)
            add("ssim_bs%d_fwd" % bs, *timeit(f, args.iters), 12 * npx)
            add("ssim_bs%d_bwd" % bs, *timeit(g, args.iters), 16 * npx)
            add("ssim_bs%d_fwd_bwd_masked" % bs, *timeit(h, args.iters), 24 * npx)

            def torch_ref(bs=bs):
                pool = lambda t: torch.nn.functional.avg_pool2d(
                    torch.nn.functional.pad(t, (bs // 2, bs - 1 - bs // 2, bs // 2, bs - 1 - bs // 2), mode="replicate"), bs, stride=1)
                x = sets[0]["es"].detach().requires_grad_(True)
                y, m = sets[0]["ta"], sets[0]["std"]
                mx, my = pool(x), pool(y)
                vxx, vyy, vxy = pool(x * x) - mx * mx, pool(y * y) - my * my, pool(x * y) - mx * my
                s_ = (2 * mx * my + c1) * (2 * vxy + c2) / ((mx * mx + my * my + c1) * (vxx + vyy + c2))
                ((m * (1 - s_) / 2).sum() / m.sum()).backward()
            for _ in range(3):
                torch_ref()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                torch_ref()
            e1.record()
            torch.cuda.synchronize()
            r = res["ops"]["ssim_bs%d_fwd_bwd_masked" % bs]
            r["torch_eager_ms"] = e0.elapsed_time(e1) / 10
            r["speedup_vs_torch_eager"] = r["torch_eager_ms"] / r["ms_median"]
    if "warp" in only:
        # SURVEY 8(f) rank 1: the disparity warp in front of the loss, and the whole RectifiedPatternSimilarityLoss step
        # (warp -> fused census_sad loss forward+backward+masked mean -> warp backward)
        pat = torch.from_numpy(np.ascontiguousarray(base["pat_lcn"][:1])).to(dev)
        disps = [torch.from_numpy(np.ascontiguousarray(np.roll(base["disp"], 5 * s, axis=2))).to(dev) for s in range(NS)]
        sums = torch.zeros(2, device=dev)
        def f(i, st):
            d = sets[i % NS]
            _lib.call("ctd_warp_pattern_fwd_f32", pat.data_ptr(), disps[i % NS].data_ptr(), d["o1"].data_ptr(), B, 1, H, W, H, W, st)
        add("warp_fwd", *timeit(f, args.iters), 8 * npx)
        def f(i, st):
            d = sets[i % NS]
            _lib.call("ctd_warp_pattern_bwd_f32", pat.data_ptr(), disps[i % NS].data_ptr(), d["go"].data_ptr(), d["o2"].data_ptr(), B, 1, H, W, H, W, st)
        add("warp_bwd", *timeit(f, args.iters), 12 * npx)
        gis = [torch.empty(B, 1, H, W, device=dev) for _ in range(NS)]
        def f(i, st):
            d = sets[i % NS]
            _lib.call("ctd_warp_pattern_fwd_f32", pat.data_ptr(), disps[i % NS].data_ptr(), d["o1"].data_ptr(), B, 1, H, W, H, W, st)
            _lib.call("ctd_photometric_fwd_bwd_masked_f32", d["o1"].data_ptr(), d["ta"].data_ptr(), d["std"].data_ptr(), d["std"].data_ptr(),
                      d["o2"].data_ptr(), gis[i % NS].data_ptr(), sums.data_ptr(), B, 1, H, W, 9, 3, 0.5, st)
            _lib.call("ctd_warp_pattern_bwd_f32", pat.data_ptr(), disps[i % NS].data_ptr(), gis[i % NS].data_ptr(), d["o2"].data_ptr(), B, 1, H, W, H, W, st)
        add("pattern_similarity_loss_step", *timeit(f, args.iters), (8 + 24 + 12) * npx,
            extra={"note": "RectifiedPatternSimilarityLoss.tforward + backward to the disparity: warp, fused census_sad loss, warp gradient"})
        projs = [torch.empty(B, 1, H, W, device=dev) for _ in range(NS)]
        def f(i, st):
            d = sets[i % NS]
            _lib.call("ctd_pattern_similarity_f32", pat.data_ptr(), disps[i % NS].data_ptr(), d["ta"].data_ptr(), d["std"].data_ptr(), d["std"].data_ptr(),
                      projs[i % NS].data_ptr(), d["o1"].data_ptr(), d["o2"].data_ptr(), sums.data_ptr(), B, 1, H, W, H, W, 3, 0.5, st)
        add("pattern_similarity_loss_step_one_kernel", *timeit(f, args.iters), (4 + 8 + 4 + 4 + 4) * npx,
            extra={"note": "the same step as ONE kernel (ctd_pattern_similarity_f32): disp, im, std in; pattern_proj, loss map, d loss / d disp out"})
    if "pyramid" in only:
        # SURVEY 8(f) rank 2: the loss at the model's four pyramid levels (exp_synph.py:25-27,107-111) -- 4 x (warp, fused
        # census_sad loss, warp gradient) = 12 kernels.  Every entry point is capture-safe, so the whole pyramid is ONE
        # CUDA graph replay; the same 12 calls issued from Python on a stream are reported next to it.
        levels = []
        for s_ in range(4):
            h_, w_ = H >> s_, W >> s_
            dd = synth.make_batch(min(B, 8), h_, w_)
            t_ = {k: torch.from_numpy(np.ascontiguousarray(np.concatenate([dd[k]] * ((B + 7) // 8))[:B])).to(dev) for k in ("ta", "std", "disp", "pat_lcn")}
            t_["pat"] = t_["pat_lcn"][:1].contiguous()
            for k in ("proj", "loss", "gi", "gd"):
                t_[k] = torch.empty(B, 1, h_, w_, device=dev)
            t_["sums"] = torch.zeros(2, device=dev)
            levels.append((h_, w_, t_))
        def chain(st):
            for h_, w_, t_ in levels:
                _lib.call("ctd_warp_pattern_fwd_f32", t_["pat"].data_ptr(), t_["disp"].data_ptr(), t_["proj"].data_ptr(), B, 1, h_, w_, h_, w_, st)
                _lib.call("ctd_photometric_fwd_bwd_masked_f32", t_["proj"].data_ptr(), t_["ta"].data_ptr(), t_["std"].data_ptr(), t_["std"].data_ptr(),
                          t_["loss"].data_ptr(), t_["gi"].data_ptr(), t_["sums"].data_ptr(), B, 1, h_, w_, 9, 3, 0.5, st)
                _lib.call("ctd_warp_pattern_bwd_f32", t_["pat"].data_ptr(), t_["disp"].data_ptr(), t_["gi"].data_ptr(), t_["gd"].data_ptr(), B, 1, h_, w_, h_, w_, st)
        def chain1(st):
            for h_, w_, t_ in levels:
                _lib.call("ctd_pattern_similarity_f32", t_["pat"].data_ptr(), t_["disp"].data_ptr(), t_["ta"].data_ptr(), t_["std"].data_ptr(), t_["std"].data_ptr(),
                          t_["proj"].data_ptr(), t_["loss"].data_ptr(), t_["gd"].data_ptr(), t_["sums"].data_ptr(), B, 1, h_, w_, h_, w_, 3, 0.5, st)
        px_all = sum(B * h_ * w_ for h_, w_, _ in levels)
        add("pyramid_4_levels_graph_one_kernel_per_level", *timeit(lambda i, st: chain1(st), args.iters, nrep=1), 24 * px_all, px=px_all,
            extra={"note": "one CUDA graph replay = 4 kernels (ctd_pattern_similarity_f32 per level)"})
        add("pyramid_4_levels_graph", *timeit(lambda i, st: chain(st), args.iters, nrep=1), 44 * px_all, px=px_all,
            extra={"note": "one CUDA graph replay = 12 kernels (4 levels x warp, fused census_sad loss, warp gradient)"})
        cur = torch.cuda.current_stream().cuda_stream
        for _ in range(5):
            chain(cur)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.iters):
            chain(cur)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.iters
        add("pyramid_4_levels_stream_launches", ms, ms, 44 * px_all, px=px_all, extra={"note": "the same 12 calls issued one by one from Python"})
    if "geometric" in only:
        # SURVEY 8(f) rank 3: ProjectionDepthSimilarityLoss.tforward (both directions, loss + both depth gradients) for B
        # frame pairs: two kernels, against the reference's own torch formulation (4 bmm, 2 grid_sample, ~20 elementwise
        # kernels and their autograd twins) on the same GPU
        gd = synth.make_depth_pairs(B, H, W, seed=0)
        cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        ray = tx.projection_rays(gd["Ki"], H, W).to(dev)
        g = {k: cu(v) for k, v in gd.items()}
        deps = [(cu(np.roll(gd["depth0"], 5 * s, axis=3)), cu(np.roll(gd["depth1"], 5 * s, axis=3))) for s in range(NS)]
        g0s = [torch.empty(B, 1, H, W, device=dev) for _ in range(NS)]
        g1s = [torch.empty(B, 1, H, W, device=dev) for _ in range(NS)]
        sums = torch.zeros(2, 2, device=dev)
        scale = 1.0 / npx
        def f(i, st):
            d0, d1 = deps[i % NS]
            a0, a1 = g0s[i % NS], g1s[i % NS]
            a1.zero_()
            _lib.call("ctd_depth_similarity_f32", d0.data_ptr(), d1.data_ptr(), ray.data_ptr(), g["K"].data_ptr(), g["R0"].data_ptr(),
                      g["t0"].data_ptr(), g["R1"].data_ptr(), g["t1"].data_ptr(), a0.data_ptr(), a1.data_ptr(), sums[0].data_ptr(),
                      B, H, W, 0.1, scale, 0, st)
            _lib.call("ctd_depth_similarity_f32", d1.data_ptr(), d0.data_ptr(), ray.data_ptr(), g["K"].data_ptr(), g["R1"].data_ptr(),
                      g["t1"].data_ptr(), g["R0"].data_ptr(), g["t0"].data_ptr(), a1.data_ptr(), a0.data_ptr(), sums[1].data_ptr(),
                      B, H, W, 0.1, scale, 1, st)
        # per direction: depthA + grad depthA (8 B) and the gather / scatter on depthB, grad depthB (8 B); + the memset
        add("depth_similarity_both_directions", *timeit(f, args.iters), (2 * 16 + 4) * npx,
            extra={"note": "ProjectionDepthSimilarityLoss.tforward, value + gradients w.r.t. both depth maps, clamp 0.1; Mpix/s counts one frame of each pair"})
        import losses_torch  # oracle/: the reference's torch formulation, used here only as the comparison leg
        def torch_ref():
            d0, d1 = deps[0][0].clone().requires_grad_(True), deps[0][1].clone().requires_grad_(True)
            losses_torch.depth_similarity(d0, d1, g["R0"], g["t0"], g["R1"], g["t1"], g["K"], ray, 0.1).backward()
        for _ in range(3):
            torch_ref()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            torch_ref()
        e1.record()
        torch.cuda.synchronize()
        res["ops"]["depth_similarity_both_directions"]["torch_eager_ms"] = e0.elapsed_time(e1) / 10
    if "disparity" in only:
        # SURVEY 8(f) rank 4: DisparityLoss.tforward (5x5 Sobel, two-Laplacian mixture weighted by the edge map) with the
        # gradients w.r.t. disp and edge, one kernel, against the reference's torch formulation on the same GPU
        disps = [torch.from_numpy(np.ascontiguousarray(np.roll(base["disp"], 5 * s, axis=3))).to(dev) for s in range(NS)]
        edges = [torch.sigmoid(torch.randn(B, 1, H, W, device=dev, generator=torch.Generator(device=dev).manual_seed(s))) for s in range(NS)]
        gds = [torch.empty(B, 1, H, W, device=dev) for _ in range(NS)]
        ges = [torch.empty(B, 1, H, W, device=dev) for _ in range(NS)]
        sums = torch.zeros(2, device=dev)
        def f(i, st):
            _lib.call("ctd_disparity_loss_f32", disps[i % NS].data_ptr(), edges[i % NS].data_ptr(), gds[i % NS].data_ptr(), ges[i % NS].data_ptr(),
                      sums.data_ptr(), B, H, W, 1.0 / npx, st)
        add("disparity_loss_fwd_bwd", *timeit(f, args.iters), 16 * npx,
            extra={"note": "DisparityLoss.tforward with edge map: loss + gradients w.r.t. disp and edge"})
        import losses_torch  # oracle/: comparison leg only
        torch.backends.cudnn.allow_tf32 = False  # the reference's convolutions in fp32 (what the kernel is checked against)
        def torch_ref():
            d, e = disps[0].clone().requires_grad_(True), edges[0].clone().requires_grad_(True)
            losses_torch.disparity_loss(d, e).backward()
        for _ in range(3):
            torch_ref()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            torch_ref()
        e1.record()
        torch.cuda.synchronize()
        res["ops"]["disparity_loss_fwd_bwd"]["torch_eager_ms"] = e0.elapsed_time(e1) / 10
    if "lcn" in only:
        def f(i, st):
            d = sets[i % NS]
            _lib.call("ctd_lcn_f32", d["im"].data_ptr(), d["o1"].data_ptr(), d["o2"].data_ptr(), B, H, W, 5, 0.05, st)
        add("lcn_fwd", *timeit(f, args.iters), 12 * npx)
    if "reduce" in only:
        ws = torch.zeros(int(_lib.lib().ctd_masked_sums_workspace_bytes()), dtype=torch.uint8, device=dev)
        out2 = torch.zeros(2, device=dev)
        def f(i, st):
            d = sets[i % NS]
            _lib.call("ctd_masked_sums_f32", d["es"].data_ptr(), d["std"].data_ptr(), npx, out2.data_ptr(), ws.data_ptr(), st)
        add("masked_sums", *timeit(f, args.iters), 8 * npx)
    if "xcorrvol" in only:
        D = 128
        vols = [torch.empty(B, D, H, W, device=dev) for _ in range(2)]
        for bs in (9, 5):
            def f(i, st, bs=bs):
                d = sets[i % NS]
                _lib.call("ctd_xcorrvol_f32", d["ta"].data_ptr(), d["pat_lcn"].data_ptr(), vols[i % 2].data_ptr(), B, 1, H, W, D, bs, st)
            add("xcorrvol_D128_bs%d" % bs, *timeit(f, max(3, args.iters // 6), warmup=1, nrep=2), (8 + 4 * D) * npx)
        del vols
    if "xcorr_disparity" in only:
        # the fused winner-take-all disparity (ctd_xcorr_disparity_f32, sub-pixel on) against what a caller does without it,
        # on the same inputs in the same run: xcorrvol, then torch.max over d and the three-point parabola in torch
        D = 128
        vol = torch.empty(B, D, H, W, device=dev)
        outs = [(torch.empty(B, 1, H, W, device=dev), torch.empty(B, 1, H, W, device=dev)) for _ in range(2)]
        for bs in (9, 5):
            def f(i, st, bs=bs):
                d, (o_d, o_s) = sets[i % NS], outs[i % 2]
                _lib.call("ctd_xcorr_disparity_f32", d["ta"].data_ptr(), d["pat_lcn"].data_ptr(), o_d.data_ptr(), o_s.data_ptr(),
                          B, 1, H, W, D, bs, 1, st)
            def g(i, st, bs=bs):
                d = sets[i % NS]
                _lib.call("ctd_xcorrvol_f32", d["ta"].data_ptr(), d["pat_lcn"].data_ptr(), vol.data_ptr(), B, 1, H, W, D, bs, st)
                c0, di = vol.max(dim=1, keepdim=True)
                cm, cp = vol.gather(1, (di - 1).clamp(min=0)), vol.gather(1, (di + 1).clamp(max=D - 1))
                den = cm - 2 * c0 + cp
                ok = (di > 0) & (di < D - 1) & (den < 0)
                outs[i % 2][0].copy_(di + torch.where(ok, (cm - cp) / (2 * den), 0.0).clamp(-0.5, 0.5))
                outs[i % 2][1].copy_(c0)
            def f0(i, st, bs=bs):
                d, (o_d, o_s) = sets[i % NS], outs[i % 2]
                _lib.call("ctd_xcorr_disparity_f32", d["ta"].data_ptr(), d["pat_lcn"].data_ptr(), o_d.data_ptr(), o_s.data_ptr(),
                          B, 1, H, W, D, bs, 0, st)
            fused, unfused = "xcorr_disparity_D128_bs%d" % bs, "xcorrvol_then_torch_argmax_D128_bs%d" % bs
            add(fused, *timeit(f, max(3, args.iters // 6), warmup=1, nrep=2), 16 * npx,
                extra={"note": "in0, in1 in; disp (sub-pixel) and score out"})
            add(fused + "_integer", *timeit(f0, max(3, args.iters // 6), warmup=1, nrep=2), 16 * npx,
                extra={"note": "the same without sub-pixel refinement"})
            add(unfused, *timeit(g, max(3, args.iters // 6), warmup=1, nrep=2), (8 + 8 * D + 16) * npx,
                extra={"note": "xcorrvol writes the volume, torch.max reads it back, parabola from gathers"})
            res["ops"][fused]["speedup_vs_volume_then_argmax"] = res["ops"][unfused]["ms_median"] / res["ops"][fused]["ms_median"]
        del vol
    if "sgm" in only:
        # semi-global matching over the xcorrvol block-9 volume of the bench frames: the fused call (ctd_sgm_f32, sub-pixel
        # on) at 4 and 8 paths, against sgm_aggregate followed by disparity_from_volume in the same run.  The volume is
        # larger than L2 at batch 8 already, so one input serves every launch.
        D = 128
        vol = torch.empty(B, D, H, W, device=dev)
        _lib.call("ctd_xcorrvol_f32", sets[0]["ta"].data_ptr(), sets[0]["pat_lcn"].data_ptr(), vol.data_ptr(), B, 1, H, W, D, 9,
                  torch.cuda.current_stream().cuda_stream)
        agg = torch.empty_like(vol)
        o_d, o_s = torch.empty(B, 1, H, W, device=dev), torch.empty(B, 1, H, W, device=dev)
        floor = (4 * D + 8) * npx
        it = max(3, args.iters // 6)
        for P in (4, 8):
            def f(i, st, P=P):
                _lib.call("ctd_sgm_f32", vol.data_ptr(), agg.data_ptr(), o_d.data_ptr(), o_s.data_ptr(), B, D, H, W, 0.2, 2.0, P, 1, st)

            def g(i, st, P=P):
                _lib.call("ctd_sgm_f32", vol.data_ptr(), agg.data_ptr(), None, None, B, D, H, W, 0.2, 2.0, P, 1, st)
                d, s = tx.disparity_from_volume(agg, True)
                o_d.copy_(d)
                o_s.copy_(s)
            fused, unfused = "sgm_disparity_%dpaths_D128" % P, "sgm_aggregate_then_disparity_from_volume_%dpaths_D128" % P
            design = (3 * P - 1) * 4 * D * npx + 8 * npx
            add(fused, *timeit(f, it, warmup=1, nrep=2), floor,
                extra={"note": "algo_bytes: V in (4D B/px), disp and score out (8 B/px); A is written too (caller-owned)",
                       "design_bytes": design})
            res["ops"][fused]["frac_design_at_peak"] = design / res["ops"][fused]["ms_median"] / 1e6 / PEAK
            res["ops"][fused]["achieved_design_gbs"] = design / res["ops"][fused]["ms_median"] / 1e6
            add(unfused, *timeit(g, it, warmup=1, nrep=2), floor,
                extra={"note": "the same aggregation without disp/score, then disparity_from_volume reads A back in torch"})
            res["ops"][fused]["speedup_vs_unfused"] = res["ops"][unfused]["ms_median"] / res["ops"][fused]["ms_median"]
        if B <= 8:
            # the torch restatement on the GPU: launch-bound (a few ops per scan-line step), timed eagerly over two calls
            tx.disparity_from_volume(tx.sgm_aggregate_pytorch(vol, 0.2, 2.0, 8), True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(2):
                tx.disparity_from_volume(tx.sgm_aggregate_pytorch(vol, 0.2, 2.0, 8), True)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 2
            add("sgm_pytorch_restatement_8paths_D128", ms, ms, floor, extra={"note": "sgm_aggregate_pytorch + disparity_from_volume"})
            res["ops"]["sgm_disparity_8paths_D128"]["speedup_vs_torch"] = ms / res["ops"]["sgm_disparity_8paths_D128"]["ms_median"]
        del vol, agg
    if "census_match" in only:
        # census matching (7x9 window, D = 128) on the bench frames (ta against pat_lcn), in the same run on the same inputs:
        # the volume at block 1 (what SGM consumes), the fused disparity at block 9 (sub-pixel on), the unfused pair
        # census_vol(bs 9) + disparity_from_volume, the torch restatement on the GPU, and census_vol(bs 1) -> sgm_disparity.
        D = 128
        floors = census_traffic(B, 1, H, W, D)
        vol = torch.empty(B, D, H, W, device=dev)
        o_d, o_s = torch.empty(B, 1, H, W, device=dev), torch.empty(B, 1, H, W, device=dev)
        it = max(3, args.iters // 6)

        def vol_call(i, st, bs):
            d = sets[i % NS]
            _lib.call("ctd_census_vol_f32", d["ta"].data_ptr(), d["pat_lcn"].data_ptr(), vol.data_ptr(), B, 1, H, W, D, 7, 9, bs, st)

        def f(i, st):
            d = sets[i % NS]
            _lib.call("ctd_census_disparity_f32", d["ta"].data_ptr(), d["pat_lcn"].data_ptr(), o_d.data_ptr(), o_s.data_ptr(),
                      B, 1, H, W, D, 7, 9, 9, 1, st)

        def g(i, st):
            vol_call(i, st, 9)
            dd, ss = tx.disparity_from_volume(vol, True)
            o_d.copy_(dd)
            o_s.copy_(ss)

        def sgm(i, st):
            vol_call(i, st, 1)
            dd, ss = tx.sgm_disparity(vol, 6, 400, 8)
            o_d.copy_(dd)
            o_s.copy_(ss)
        add("census_vol_D128_bs1", *timeit(lambda i, st: vol_call(i, st, 1), it, warmup=1, nrep=2), floors["volume"],
            extra={"note": "algo_bytes: in0, in1 in (8 B/px), V out (4D B/px)"})
        add("census_disparity_D128_bs9", *timeit(f, it, warmup=1, nrep=2), floors["disparity"],
            extra={"note": "algo_bytes: in0, in1 in, disp and score out (16 B/px); the volume is never written"})
        add("census_vol_bs9_then_disparity_from_volume_D128", *timeit(g, it, warmup=1, nrep=2), floors["volume"],
            extra={"note": "census_vol(bs 9) writes V, disparity_from_volume reads it back in torch"})
        res["ops"]["census_disparity_D128_bs9"]["speedup_vs_unfused"] = (
            res["ops"]["census_vol_bs9_then_disparity_from_volume_D128"]["ms_median"] / res["ops"]["census_disparity_D128_bs9"]["ms_median"])
        add("census_vol_bs1_then_sgm_disparity_8paths_D128", *timeit(sgm, it, warmup=1, nrep=2), floors["volume"],
            extra={"note": "census_vol(bs 1) then sgm_disparity(p1 = 6, p2 = 400, 8 paths); algo_bytes is the volume's floor only"})
        if B <= 8:
            # the torch restatement on the GPU (a loop over d of gathers, XOR and a byte popcount table), timed eagerly
            a, b = sets[0]["ta"], sets[0]["pat_lcn"]
            tx.disparity_from_volume(tx.census_vol_pytorch(a, b, D, (7, 9), 9), True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(2):
                tx.disparity_from_volume(tx.census_vol_pytorch(a, b, D, (7, 9), 9), True)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 2
            add("census_pytorch_restatement_bs9_D128", ms, ms, floors["volume"],
                extra={"note": "disparity_from_volume(census_vol_pytorch(bs 9))"})
            res["ops"]["census_disparity_D128_bs9"]["speedup_vs_torch"] = ms / res["ops"]["census_disparity_D128_bs9"]["ms_median"]
        del vol
    if "disparity_check" in only:
        # left-right consistency and uniqueness checks over the census block-1 volume of the bench frames (7x9 window,
        # D = 128): the fused call (disp, score and valid; max_diff = 1, uniqueness = 16), the torch restatement on the GPU
        # and disparity_from_volume alone, in the same run.  The volume is larger than L2 at batch 8 already, so one input
        # serves every launch; the floor is one read of it (4D B/px).
        D = 128
        vol = torch.empty(B, D, H, W, device=dev)
        _lib.call("ctd_census_vol_f32", sets[0]["ta"].data_ptr(), sets[0]["pat_lcn"].data_ptr(), vol.data_ptr(), B, 1, H, W, D,
                  7, 9, 1, torch.cuda.current_stream().cuda_stream)
        o_d, o_s = torch.empty(B, 1, H, W, device=dev), torch.empty(B, 1, H, W, device=dev)
        o_v = torch.empty(B, 1, H, W, dtype=torch.uint8, device=dev)
        floor = 4 * D * npx
        it = max(3, args.iters // 6)

        def f(i, st):
            _lib.call("ctd_disparity_check_f32", vol.data_ptr(), o_d.data_ptr(), o_s.data_ptr(), None, None, o_v.data_ptr(),
                      B, D, H, W, 1, 16.0, 1, st)

        def g(i, st):
            dd, ss = tx.disparity_from_volume(vol, True)
            o_d.copy_(dd)
            o_s.copy_(ss)
        add("disparity_check_D128", *timeit(f, it, warmup=2, nrep=4), floor,
            extra={"note": "census_vol(bs 1) volume in (4D B/px, the floor); disp, score and valid out (9 B/px)"})
        add("disparity_from_volume_D128", *timeit(g, it, warmup=2, nrep=4), floor,
            extra={"note": "torch winner-take-all with sub-pixel offset only: no right view, no checks"})
        tx.disparity_check_pytorch(vol, 1, 16.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(2):
            tx.disparity_check_pytorch(vol, 1, 16.0)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 2
        add("disparity_check_pytorch_D128", ms, ms, floor, extra={"note": "disparity_check_pytorch on the GPU, timed eagerly"})
        r = res["ops"]["disparity_check_D128"]
        r["speedup_vs_torch"] = ms / r["ms_median"]
        r["ratio_vs_disparity_from_volume"] = res["ops"]["disparity_from_volume_D128"]["ms_median"] / r["ms_median"]
        r["valid_frac"] = float(o_v.float().mean())
        del vol
    if "speckle" in only:
        # speckle filter (max_size 200, max_diff 1) of the census block-9 integer disparities of the bench frames (7x9
        # window, D = 128) after disparity_check(max_diff 1): the fused call against speckle_filter_pytorch on the GPU.  The
        # floor is disp and valid in, valid_out out (6 B/px); labels and sizes add 8 B/px of scratch, written once and
        # read about once.  One input serves every launch: at batch 8 it and the scratch (54 MB in all) fit in L2.
        vol = torch.empty(B, 128, H, W, device=dev)
        _lib.call("ctd_census_vol_f32", sets[0]["ta"].data_ptr(), sets[0]["pat_lcn"].data_ptr(), vol.data_ptr(), B, 1, H, W, 128,
                  7, 9, 9, torch.cuda.current_stream().cuda_stream)
        disp, _, ok = tx.disparity_check(vol, 1, 0.0, subpixel=False)
        del vol
        o_v = torch.empty(B, 1, H, W, dtype=torch.uint8, device=dev)

        def f(i, st):
            _lib.call("ctd_speckle_filter_f32", disp.data_ptr(), ok.data_ptr(), o_v.data_ptr(), B, H, W, 200, 1.0, st)
        add("speckle_filter", *timeit(f, args.iters), 6 * npx,
            extra={"note": "disp (4 B/px) and valid (1 B/px) in, valid_out (1 B/px) out; 4 launches",
                   "scratch_bytes": 16 * npx})
        ref = tx.speckle_filter_pytorch(disp, ok, 200, 1.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(3):
            tx.speckle_filter_pytorch(disp, ok, 200, 1.0)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 3
        add("speckle_filter_pytorch", ms, ms, 6 * npx, extra={"note": "speckle_filter_pytorch on the GPU, timed eagerly"})
        r = res["ops"]["speckle_filter"]
        r["speedup_vs_torch"] = ms / r["ms_median"]
        r["bit_equal_to_torch"] = bool(torch.equal(o_v.bool(), ref))
        r["valid_in_frac"] = float(ok.float().mean())
        r["valid_out_frac"] = float(o_v.float().mean())
        del disp, ok, ref
    if "proj_nn" in only:
        T = 4
        xyz, K, poses = synth.make_clouds(T, H, W)
        Kd = torch.from_numpy(K).to(dev)
        pairs = [(i, j) for i in range(T) for j in range(T) if i != j]
        x0 = torch.from_numpy(np.stack([synth.transform(xyz[i], poses[j]) for i, j in pairs])).to(dev)   # [12,H,W,3]
        x1 = torch.from_numpy(np.stack([xyz[j] for i, j in pairs])).to(dev)
        out = torch.empty(len(pairs), H, W, dtype=torch.int64, device=dev)
        for ps in (3, 5):
            def f(i, st, ps=ps):
                _lib.call("ctd_proj_nn_f32", x0.data_ptr(), x1.data_ptr(), Kd.data_ptr(), out.data_ptr(), len(pairs), H, W, ps, st)
            add("proj_nn_ps%d_12pairs" % ps, *timeit(f, args.iters), 32 * len(pairs) * H * W, px=len(pairs) * H * W,
                extra={"valid_frac": float((out >= 0).float().mean())})
        if "crosscheck" in only:
            n = len(pairs) * H * W
            i01 = out.view(-1)
            i10 = out.view(len(pairs), -1).flip(0).contiguous().view(-1)
            m = torch.empty(n, dtype=torch.uint8, device=dev)
            def f(i, st):
                _lib.call("ctd_crosscheck", i01.data_ptr(), i10.data_ptr(), m.data_ptr(), n, n, st)
            add("crosscheck_%d" % n, *timeit(f, args.iters), 17 * n, px=n)
    if "config4" in only:
        # BASELINE configs[3]: one geometric step on a 4-frame track -- for the 6 frame pairs, ProjNN in both directions
        # (12 image-sized queries, one batched launch), CrossCheck in both directions, and PhotometricLoss census_sad
        # forward+backward on the 4 frames
        T = 4
        xyz, K, poses = synth.make_clouds(T, H, W)
        Kd = torch.from_numpy(K).to(dev)
        pairs = [(i, j) for i in range(T) for j in range(T) if i != j]
        rev = [pairs.index((j, i)) for i, j in pairs]
        x0 = torch.from_numpy(np.stack([synth.transform(xyz[i], poses[j]) for i, j in pairs])).to(dev)
        x1 = torch.from_numpy(np.stack([xyz[j] for i, j in pairs])).to(dev)
        idx = torch.empty(len(pairs), H, W, dtype=torch.int64, device=dev)
        idx_rev = torch.empty_like(idx)
        m01 = torch.empty(len(pairs) * H * W, dtype=torch.uint8, device=dev)
        rev_t = torch.tensor(rev, device=dev)
        f4 = {k: sets[0][k][:T].contiguous() if B >= T else sets[0][k] for k in ("es", "ta", "go")}
        o4, g4 = torch.empty(T, 1, H, W, device=dev), torch.empty(T, 1, H, W, device=dev)
        n = len(pairs) * H * W
        def f(i, st):
            _lib.call("ctd_proj_nn_f32", x0.data_ptr(), x1.data_ptr(), Kd.data_ptr(), idx.data_ptr(), len(pairs), H, W, 3, st)
            # indices are per launch-batch flat indices (image p at offset p*H*W): crosscheck pair p against its reverse
            torch.index_select(idx, 0, rev_t, out=idx_rev)
            _lib.call("ctd_crosscheck", idx.data_ptr(), idx_rev.data_ptr(), m01.data_ptr(), n, n, st)
            _lib.call("ctd_photometric_fwd_bwd_f32", f4["es"].data_ptr(), f4["ta"].data_ptr(), f4["go"].data_ptr(), o4.data_ptr(),
                      g4.data_ptr(), T, 1, H, W, 9, 3, 0.5, st)
        add("config4_geometric_step_4frames", *timeit(f, args.iters, nrep=4), 32 * n + 17 * n + 20 * T * H * W, px=T * H * W,
            extra={"note": "ProjNN ps=3 on 12 ordered frame pairs + CrossCheck + census_sad fwd+bwd on 4 frames; Mpix/s counts the 4 frames"})
    if "nn" in only:
        n = 16384
        rng = np.random.RandomState(0)
        p0 = torch.from_numpy(rng.randn(n, 3).astype(np.float32)).to(dev)
        p1 = torch.from_numpy(rng.randn(n, 3).astype(np.float32)).to(dev)
        out = torch.empty(n, dtype=torch.int64, device=dev)
        def f(i, st):
            _lib.call("ctd_nn_f32", p0.data_ptr(), p1.data_ptr(), out.data_ptr(), n, n, st)
        ms, mn = timeit(f, args.iters)
        res["ops"]["nn_16384x16384"] = {"ms_median": ms, "ms_min": mn, "gpair_s": n * n / ms / 1e6}
        if verbose:
            print("nn", res["ops"]["nn_16384x16384"], file=sys.stderr)
    if "gpu_reference" in only:
        # the reference's OWN CUDA extension (oracle/_ref/ctd_ref_ext_cuda.so, unmodified, sm_100) on the same box and the
        # same rotating buffers: the "existing GPU kernel" bar.  Stream launches on the legacy default stream, as the
        # reference issues them.
        import ref_gpu  # oracle/: comparison leg only
        T = 4
        xyz, K, poses = synth.make_clouds(T, H, W)
        pairs = [(i, j) for i in range(T) for j in range(T) if i != j]
        x0 = torch.from_numpy(np.stack([synth.transform(xyz[i], poses[j]) for i, j in pairs])).to(dev)
        x1 = torch.from_numpy(np.stack([xyz[j] for i, j in pairs])).to(dev)
        r = ref_gpu.time_ops(sets, B, H, W, iters=5, clouds=(x0, x1, torch.from_numpy(K).to(dev)), xcorr_images=min(B, 2))
        if r is None:
            res["gpu_reference"] = {"unavailable": "oracle/_ref/ctd_ref_ext_cuda.so not built"}
        else:
            res["gpu_reference"] = r
            for name, v in r.items():
                mine = res["ops"].get(name)
                if mine:
                    v["speedup_vs_reference_cuda"] = v["ms"] / mine["ms_median"]
            if verbose:
                print("gpu_reference", json.dumps(r), file=sys.stderr, flush=True)
    return res


if __name__ == "__main__":
    main()
