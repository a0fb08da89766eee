#!/usr/bin/env python
"""Benchmark of the torchext op path on B200 (BASELINE.json metric, configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this framework (libctd_b200.so)
    python bench.py --dump-outputs DIR [...]                        # + the last timed step's outputs as DIR/<name>.npy
    python bench.py --impl reference [...]                          # the reference's CPU path, host cores
    torchrun --nproc-per-node N ... bench.py --gpus N ...           # one rank per GPU, weak scaling

A "step" is one pass of the hot path over one batch of synthetic 480x640 dot-pattern pairs
(SURVEY.md section 8d data), batch 8 per GPU:
    LCN(5, 0.05) forward  ->  PhotometricLoss 'sad' ("l1") forward + backward
                          ->  PhotometricLoss 'census_sad' (the reference's structural mode, standing in
                              for "ssim", SURVEY.md D1) forward + backward -- each through
                              ctd_photometric_fwd_bwd_masked_f32, which produces the loss map, the gradient
                              (grad_out = std / sum(std) is an input, as in networks.py:377) and the caller's
                              masked loss reduction (networks.py:377) in ONE pass
The same chain with every forward, backward and masked reduction as separate calls (what torch autograd does with
photometric_loss) is timed as well and reported as `separate_calls`.
and, for N > 1, one packed NCCL all-reduce of the four loss scalars.  value = pixels per second through
that whole chain (N * B * H * W / step time); per-op figures are in "ops".

Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks;
inputs AND outputs rotate over NSETS buffer sets whose footprint exceeds L2, so every step streams
from HBM.  roofline: per-kernel CUDA-event durations measured inside the same timed steps;
algorithmic bytes per pixel from SURVEY.md section 8d; peak from MEASURED_PEAKS.json.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

H, W, B_PER_GPU, BS, EPS, LCN_R, LCN_EPS = 480, 640, 8, 9, 0.5, 5, 0.05
NSETS = 4
METRIC = "Mpix/s through LCN fwd + PhotometricLoss sad fwd+bwd + census_sad fwd+bwd (batch 8, 480x640); per-op Mpix/s in ops"
WORKLOAD = ("configs[1]: LCN(5,0.05) fwd + PhotometricLoss l1(sad) fwd+bwd + census_sad (stands in for ssim) fwd+bwd "
            "+ masked loss sums (one fused call per loss), batch 8 per GPU, 480x640, block 9, eps 0.5, C=1")
# algorithmic bytes per pixel, fp32, C=1 (SURVEY.md section 8d)
BYTES_PER_PX = {"lcn_fwd": 12, "sad_fwd": 12, "sad_bwd": 16, "census_sad_fwd": 12, "census_sad_bwd": 16,
                "sad_fwd_bwd": 24, "census_sad_fwd_bwd": 24,  # fused: es, ta, grad_out, mask in; loss map, grad_in out -- each tensor once
                "masked_sums": 8}



# The contract is ONE JSON line on stdout.  Libraries write to file descriptor 1 behind Python's back (NCCL prints
# its version banner there at the first collective), so fd 1 is pointed at stderr for the whole run and the line
# goes out through a private duplicate of the original stdout.
_REAL_STDOUT = None


def claim_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit_line(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    print(json.dumps(line), file=out, flush=True)

def workload_config(world, batch_per_gpu=None, global_batch=None, strong=False):
    """`config` of the JSON line: identical for the B200 arm and the reference arm (the driver compares them)."""
    b = B_PER_GPU if batch_per_gpu is None else batch_per_gpu
    return {"workload": WORKLOAD, "batch_per_gpu": b, "global_batch": b * world if global_batch is None else global_batch,
            "height": H, "width": W, "block_size": BS, "census_eps": EPS, "lcn_radius": LCN_R, "lcn_eps": LCN_EPS, "channels": 1,
            "l2_policy": "inputs and outputs rotate over %d buffer sets larger than the 126 MB L2" % NSETS}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md, 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks and throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU implementations (test infrastructure, used ONLY as the reported baseline / reference arm)
# ------------------------------------------------------------------------------------------------
def _cpu_chain_factory():
    """Returns (run(images: dict of [n,1,H,W] arrays) -> None, kind).  kind 'reference' = the unmodified
    reference extension compiled into oracle/_ref (photometric ops) + the reference's torch LCN recipe on
    CPU; 'port' = the plain-C oracle."""
    import oracle
    ref = None
    try:
        import build_ref
        ref = build_ref.load_ref()
    except Exception:
        ref = None
    if ref is not None:
        import torch
        torch.set_num_threads(1)

        def lcn_torch(x):  # model/networks.py:523-533 restated with the same torch ops
            k = 2 * LCN_R + 1
            w = torch.ones(1, 1, k, k)
            pad = torch.nn.functional.pad(x, (LCN_R,) * 4, mode="reflect")
            box = torch.nn.functional.conv2d(pad, w)
            box2 = torch.nn.functional.conv2d(pad * pad, w)
            avg = box / k ** 2
            std = torch.sqrt(box2 / k ** 2 - avg ** 2 + 1e-6) + LCN_EPS
            return (x - avg) / std, std

        def run(d):
            t = {k: torch.from_numpy(v) for k, v in d.items()}
            lcn_torch(t["im"])
            for ty in (1, 3):
                ref.photometric_loss_forward(t["es"], t["ta"], BS, ty, EPS)
                ref.photometric_loss_backward(t["es"], t["ta"], t["go"], BS, ty, EPS)
        return run, "reference"

    def run(d):
        oracle.lcn(d["im"], LCN_R, LCN_EPS)
        for ty in (1, 3):
            oracle.photometric_loss_forward(d["es"], d["ta"], BS, ty, EPS)
            oracle.photometric_loss_backward(d["es"], d["ta"], d["go"], BS, ty, EPS)
    return run, "port"


_POOL_RUN = None


def _pool_init():
    global _POOL_RUN
    _POOL_RUN = _cpu_chain_factory()[0]


def _pool_task(d):
    t0 = time.perf_counter()
    _POOL_RUN(d)
    return time.perf_counter() - t0


def run_reference_arm(args, rank, world):
    """The reference's own CPU implementation of the path on this box's host cores (all of them: one
    image per worker process, because the reference's loop is serial, ext_cpu.cpp:7-12)."""
    if rank != 0:
        return
    import multiprocessing as mp
    from connecting_the_dots_b200 import synth
    cores = max(1, min(os.cpu_count() or 1, 64))
    kind = _cpu_chain_factory()[1]
    batch = synth.make_batch(min(cores, 8), H, W)
    images = [{k: np.ascontiguousarray(batch[k][i % batch["im"].shape[0]:i % batch["im"].shape[0] + 1]) for k in ("im", "es", "ta", "go")}
              for i in range(cores)]
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_pool_init) as pool:
        for _ in range(args.warmup):
            pool.map(_pool_task, images[:cores])
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.map(_pool_task, images)
        dt = time.perf_counter() - t0
    ms = dt / args.steps * 1e3
    value = cores * H * W / (ms * 1e-3) / 1e6
    sample = "%d images of 480x640 per step (one per worker process), full chain LCN + sad f+b + census_sad f+b" % cores
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "Mpix/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(max(args.gpus, 1)),
            "note": "CPU arm: each step is a bounded sample of the workload (one image per worker process)",
            "cpu_baseline": {"value": value, "unit": "Mpix/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit_line(line)


def cpu_baseline_leg(n_images=4):
    """Single-threaded reference CPU path on a bounded sample (the reference's own figure is 1 core)."""
    from connecting_the_dots_b200 import synth
    run, kind = _cpu_chain_factory()
    batch = synth.make_batch(n_images, H, W)
    d = {k: batch[k] for k in ("im", "es", "ta", "go")}
    one = {k: v[:1] for k, v in d.items()}
    run(one)  # warm-up (page in the library)
    t0 = time.perf_counter()
    run(d)
    dt = time.perf_counter() - t0
    return {"value": n_images * H * W / dt / 1e6, "unit": "Mpix/s", "cores": 1, "kind": kind,
            "sample": "%d images of 480x640, full chain LCN + sad f+b + census_sad f+b, one pass, %.1f s" % (n_images, dt)}


# ------------------------------------------------------------------------------------------------
# the B200 arm
# ------------------------------------------------------------------------------------------------
def run_b200_arm(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import connecting_the_dots_b200 as ctd
    from connecting_the_dots_b200 import _lib, synth, shard_range

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = _lib.lib()
    if args.census_sym >= 0:
        _lib.set_option("census_sym", args.census_sym)
    strong = args.global_batch > 0   # the MAIN figure as strong scaling (a fixed global batch split over the ranks)
    if strong:
        lo, hi = shard_range(args.global_batch, rank, world)
        B = hi - lo
        assert B > 0, "global batch smaller than the number of ranks"
    else:
        B = B_PER_GPU
    npx = B * H * W
    npx_global = args.global_batch * H * W if strong else world * npx
    P = lambda t_: ctypes.c_void_p(t_.data_ptr())

    # ---- inputs: NSETS distinct device-resident sets (and pinned host copies for the e2e leg)
    base = synth.make_batch(min(B, 8), H, W)
    if B > 8:  # synthetic frames repeat beyond 8 (generation is the slow part, not the content)
        base = {k: np.concatenate([v] * ((B + 7) // 8))[:B] for k, v in base.items()}
    # every set's four loss scalars, contiguous, in TWO slots: ONE all-reduce covers the NSETS steps of a round, and the
    # rounds alternate between the slots so that round r+1 never waits for the reduction of round r
    sums_all = torch.zeros(2, NSETS, 2, 2, device=dev)
    sets, host_sets = [], []
    for s in range(NSETS):
        arrs = {k: np.ascontiguousarray(np.roll(base[k], 3 * s + rank, axis=2)) for k in ("im", "es", "ta", "go")}
        host = {k: torch.from_numpy(v).pin_memory() for k, v in arrs.items()}
        for k in ("lcn", "std", "gi_sad", "gi_cs"):
            host[k] = torch.empty(B, 1, H, W).pin_memory()
        host["sums"] = torch.zeros(2, 2).pin_memory()
        host_sets.append(host)
        d = {k: host[k].to(dev) for k in ("im", "es", "ta", "go")}
        for k in ("lcn", "std", "out_sad", "gi_sad", "out_cs", "gi_cs"):
            d[k] = torch.empty(B, 1, H, W, device=dev)
        d["sums"] = sums_all[0, s]
        d["sums1"] = sums_all[1, s]
        sets.append(d)
    ws = torch.zeros(int(L.ctd_masked_sums_workspace_bytes()), dtype=torch.uint8, device=dev)
    footprint_mb = NSETS * 10 * npx * 4 / 1e6
    stream = torch.cuda.current_stream(dev)
    st = stream.cuda_stream
    OPS = ("lcn_fwd", "sad_fwd_bwd", "census_sad_fwd_bwd")  # the fused calls include the masked sums
    OPS_SEP = ("lcn_fwd", "sad_fwd", "sad_bwd", "census_sad_fwd", "census_sad_bwd", "masked_sums")

    def launch_chain(d, st_, mark, fused=True, slot=0):
        p = {n: t.data_ptr() for n, t in d.items()}
        if slot:
            p["sums"] = p["sums1"]
        i = 0
        mark(i)
        _lib.call("ctd_lcn_f32", p["im"], p["lcn"], p["std"], B, H, W, LCN_R, LCN_EPS, st_)
        i += 1
        mark(i)
        if fused:
            _lib.call("ctd_photometric_fwd_bwd_masked_f32", p["es"], p["ta"], p["go"], p["std"], p["out_sad"], p["gi_sad"], p["sums"],
                      B, 1, H, W, BS, 1, EPS, st_)
            i += 1
            mark(i)
            _lib.call("ctd_photometric_fwd_bwd_masked_f32", p["es"], p["ta"], p["go"], p["std"], p["out_cs"], p["gi_cs"], p["sums"] + 8,
                      B, 1, H, W, BS, 3, EPS, st_)
            i += 1
            mark(i)
            return
        _lib.call("ctd_photometric_fwd_f32", p["es"], p["ta"], p["out_sad"], B, 1, H, W, BS, 1, EPS, st_)
        i += 1
        mark(i)
        _lib.call("ctd_photometric_bwd_f32", p["es"], p["ta"], p["go"], p["gi_sad"], B, 1, H, W, BS, 1, EPS, st_)
        i += 1
        mark(i)
        _lib.call("ctd_photometric_fwd_f32", p["es"], p["ta"], p["out_cs"], B, 1, H, W, BS, 3, EPS, st_)
        i += 1
        mark(i)
        _lib.call("ctd_photometric_bwd_f32", p["es"], p["ta"], p["go"], p["gi_cs"], B, 1, H, W, BS, 3, EPS, st_)
        i += 1
        mark(i)
        _lib.call("ctd_masked_sums_f32", p["out_sad"], p["std"], npx, p["sums"], ws.data_ptr(), st_)
        _lib.call("ctd_masked_sums_f32", p["out_cs"], p["std"], npx, p["sums"] + 8, ws.data_ptr(), st_)
        i += 1
        mark(i)

    # The two losses both wait for LCN's std but not for each other: as graph branches the memory-bound sad kernel
    # runs beside the issue-bound census kernel instead of in front of it.
    side = torch.cuda.Stream(dev)

    def launch_forked(d, cs, slot=0):
        p = {n: t.data_ptr() for n, t in d.items()}
        if slot:
            p["sums"] = p["sums1"]
        _lib.call("ctd_lcn_f32", p["im"], p["lcn"], p["std"], B, H, W, LCN_R, LCN_EPS, cs.cuda_stream)
        side.wait_stream(cs)
        first, second = (side, cs) if args.fork == 1 else (cs, side)
        _lib.call("ctd_photometric_fwd_bwd_masked_f32", p["es"], p["ta"], p["go"], p["std"], p["out_sad"], p["gi_sad"], p["sums"],
                  B, 1, H, W, BS, 1, EPS, first.cuda_stream)
        _lib.call("ctd_photometric_fwd_bwd_masked_f32", p["es"], p["ta"], p["go"], p["std"], p["out_cs"], p["gi_cs"], p["sums"] + 8,
                  B, 1, H, W, BS, 3, EPS, second.cuda_stream)
        cs.wait_stream(side)

    # One CUDA graph per buffer set: the step's kernels (plus, in the evented flavour, event-record nodes between the
    # ops), so neither `value` nor the per-op durations contain host launch latency (the kernels are 10-200 us long).
    set_events = [[torch.cuda.Event(enable_timing=True, external=True) for _ in range(len(OPS) + 1)] for _ in range(NSETS)]
    sep_events = [[torch.cuda.Event(enable_timing=True, external=True) for _ in range(len(OPS_SEP) + 1)] for _ in range(NSETS)]
    graphs, sep_graphs, plain_graphs, chain_graphs, use_graph = [], [], [], [], not args.no_graph
    kernels_per_graph = 0
    if use_graph:
        try:
            launch_chain(sets[0], st, lambda i: None)  # load modules / set attributes before capturing
            launch_chain(sets[0], st, lambda i: None, fused=False)
            torch.cuda.synchronize(dev)
            for si in range(NSETS):
                c0 = _lib.launch_count()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    cs = torch.cuda.current_stream(dev)
                    launch_chain(sets[si], cs.cuda_stream, lambda i, si=si, cs=cs: set_events[si][i].record(cs))
                graphs.append(g)
                kernels_per_graph = _lib.launch_count() - c0  # kernel nodes captured (counted by the library)
                pair = []
                for slot in (0, 1):  # the same step without the event-record nodes, the two losses as branches
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        cs = torch.cuda.current_stream(dev)
                        if args.fork:
                            launch_forked(sets[si], cs, slot)
                        else:
                            launch_chain(sets[si], cs.cuda_stream, lambda i: None, slot=slot)
                    pair.append(g)
                plain_graphs.append(pair)
                pair = []
                for slot in (0, 1):  # the step as ONE chain without event nodes (the un-overlapped figure)
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        cs = torch.cuda.current_stream(dev)
                        launch_chain(sets[si], cs.cuda_stream, lambda i: None, slot=slot)
                    pair.append(g)
                chain_graphs.append(pair)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    cs = torch.cuda.current_stream(dev)
                    launch_chain(sets[si], cs.cuda_stream, lambda i, si=si, cs=cs: sep_events[si][i].record(cs), fused=False)
                sep_graphs.append(g)
        except Exception as e:  # capture unsupported: fall back to stream launches (says so in config)
            print("bench: CUDA graph capture failed (%s); timing stream launches" % e, file=sys.stderr)
            graphs, sep_graphs, plain_graphs, chain_graphs, use_graph = [], [], [], [], False
            torch.cuda.synchronize(dev)

    # The only inter-GPU traffic of the path is the loss scalars.  They are not needed before the next step starts, so
    # the ranks reduce them ONCE PER NSETS STEPS: one NCCL all-reduce of all NSETS x 4 floats on a side stream
    # (a per-step 4-float all-reduce cost ~5 % of an 0.16 ms step at 8 GPUs: pure latency).  The kernels that overwrite a
    # set's scalars wait for the reduction that read them.
    comm_stream = torch.cuda.Stream(dev) if world > 1 else None
    state = {"comm_done": [None, None], "reduces": 0}

    def reduce_scalars(after, slot):
        comm_stream.wait_stream(after)
        with torch.cuda.stream(comm_stream):
            dist.all_reduce(sums_all[slot])
            state["comm_done"][slot] = comm_stream.record_event()
        state["reduces"] += 1

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed_run(n_steps, graph_list, n_lanes, evented_tail=0):
        """n_steps steps replayed round-robin over the buffer sets on n_lanes streams (a buffer set always uses the
        same stream); the last `evented_tail` steps are the evented single-stream replays.  Returns ms per step
        (CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks)."""
        lanes = [stream] + [torch.cuda.Stream(dev) for _ in range(min(max(n_lanes, 1), NSETS) - 1)] if use_graph else [stream]
        assert NSETS % len(lanes) == 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        e0.record(stream)
        for other in lanes[1:]:
            other.wait_stream(stream)  # no lane starts before the timed region does
        state["reduces"] = 0
        for k in range(n_steps):
            si = k % NSETS
            evented = k >= n_steps - evented_tail
            slot = 0 if (evented or graph_list in (graphs, sep_graphs)) else (k // NSETS) % 2
            lane = stream if evented else lanes[k % len(lanes)]
            if evented:
                for other in lanes[1:]:
                    stream.wait_stream(other)   # the evented replays run alone: their per-op times are undisturbed
            if world > 1 and state["comm_done"][slot] is not None and (si == 0 or evented):
                for ln in lanes:
                    ln.wait_event(state["comm_done"][slot])  # this slot's previous scalars (two rounds ago) have been reduced
            if use_graph:
                with torch.cuda.stream(lane):
                    g = (graphs if evented else graph_list)[si]
                    (g[slot] if isinstance(g, list) else g).replay()
            else:
                launch_chain(sets[si], st, lambda i: set_events[si][i].record(stream))
            if world > 1 and (si == NSETS - 1 or k == n_steps - 1 or evented):
                # the reduction waits for the round's steps (on all lanes); the lanes do not wait for it
                for other in lanes:
                    if other is not lane:
                        comm_stream.wait_stream(other)
                reduce_scalars(lane, slot)
        for other in lanes[1:]:
            stream.wait_stream(other)
        if world > 1:
            stream.wait_stream(comm_stream)  # the timed region contains every reduction
        e1.record(stream)
        sync_all()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / n_steps

    warm = max(args.warmup, 3)
    timed_run(warm, plain_graphs, args.pipeline)
    timed_run(NSETS, graphs, 1, evented_tail=NSETS)  # both graph flavours get warm
    launches0 = _lib.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    # evented (sequential, single-stream) replays at the end of the timed region: one per buffer set when there are
    # enough steps, fewer in a short run so that they stay about a tenth of it
    n_evented = min(NSETS, max(1, args.steps // 10), args.steps)
    ms_per_step = timed_run(args.steps, plain_graphs, args.pipeline, evented_tail=n_evented)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:  # before the legs below overwrite the buffers
        dump_outputs(args.dump_outputs, sets[(args.steps - 1) % NSETS])
    used = sorted({k % NSETS for k in range(args.steps - n_evented, args.steps)})
    op_ms = {n: float(np.mean([set_events[si][i].elapsed_time(set_events[si][i + 1]) for si in used])) for i, n in enumerate(OPS)}
    launches = (_lib.launch_count() - launches0) if not use_graph else kernels_per_graph * args.steps
    # the same steps with NO overlap between steps or between the two losses: one stream, one chain per step
    seq_steps = max(NSETS, min(args.steps, 20))
    seq_ms = timed_run(seq_steps, chain_graphs if use_graph else None, 1)
    # the same chain with census_sad forward and backward as separate calls (the autograd path), a few steps
    sep_steps = max(NSETS, min(args.steps, 20))
    if use_graph:
        timed_run(NSETS, sep_graphs, 1)
        sep_ms_per_step = timed_run(sep_steps, sep_graphs, 1)
        sep_ms = {n: float(np.mean([sep_events[si][i].elapsed_time(sep_events[si][i + 1]) for si in range(NSETS)])) for i, n in enumerate(OPS_SEP)}
    else:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        e0.record(stream)
        for k in range(sep_steps):
            launch_chain(sets[k % NSETS], st, lambda i, si=k % NSETS: sep_events[si][i].record(stream), fused=False)
        e1.record(stream)
        sync_all()
        sep_ms_per_step = e0.elapsed_time(e1) / sep_steps
        sep_ms = {n: float(np.mean([sep_events[si][i].elapsed_time(sep_events[si][i + 1]) for si in range(NSETS)])) for i, n in enumerate(OPS_SEP)}
    for n in ("sad_fwd", "sad_bwd", "census_sad_fwd", "census_sad_bwd", "masked_sums"):
        op_ms[n] = sep_ms[n]
    op_ms["masked_sums"] /= 2  # two launches in that interval

    # ---- e2e leg: the C ABI's host-buffer entry points, pinned host inputs/outputs, copies timed.  One deferred batch per
    # step: LCN (im -> lcn, std), then the two losses through the masked call, which returns what the reference's caller
    # uses (model/networks.py:376-377): the masked-mean scalars and d loss / d es.  The loss MAPS stay on the device (out =
    # NULL: nothing downstream reads them), and the mask is LCN's std of the same batch, served from its device buffer.
    def e2e_issue(k, wait):
        h = host_sets[k % NSETS]
        _lib.call("ctd_host_begin_batch")
        _lib.call("ctd_host_lcn_f32", P(h["im"]), P(h["lcn"]), P(h["std"]), B, H, W, LCN_R, LCN_EPS)
        _lib.call("ctd_host_photometric_fwd_bwd_masked_f32", P(h["es"]), P(h["ta"]), P(h["go"]), P(h["std"]), None, P(h["gi_sad"]),
                  ctypes.c_void_p(h["sums"].data_ptr()), B, 1, H, W, BS, 1, EPS)
        _lib.call("ctd_host_photometric_fwd_bwd_masked_f32", P(h["es"]), P(h["ta"]), P(h["go"]), P(h["std"]), None, P(h["gi_cs"]),
                  ctypes.c_void_p(h["sums"].data_ptr() + 8), B, 1, H, W, BS, 3, EPS)
        _lib.call("ctd_host_end_batch" if wait else "ctd_host_end_batch_async")

    def e2e_run(n_steps, two_deep):
        """n_steps steps; two_deep: step k + 1 is issued before step k is waited for (its uploads cross the bus under step
        k's downloads; the host buffer sets rotate, NSETS >= 3).  Every step's results are in host memory at the end."""
        t0 = time.perf_counter()
        for k in range(n_steps):
            e2e_issue(k, wait=not two_deep)
            if two_deep and k > 0:
                _lib.call("ctd_host_wait_batch")  # step k - 1
        if two_deep:
            _lib.call("ctd_host_wait_batch")
        return time.perf_counter() - t0

    def e2e_measure(two_deep):
        e2e_run(3 * NSETS, two_deep)
        sync_all()
        t = torch.tensor([e2e_run(e2e_steps, two_deep)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / e2e_steps * 1e3

    assert NSETS >= 3
    e2e_steps = max(3, min(args.steps, 20))
    e2e_sync_ms = e2e_measure(False)   # one step at a time: each returns when its results are in host memory
    e2e_ms = e2e_measure(True)         # two steps in flight
    e2e_issue(0, wait=True)            # a synchronous batch last: its byte counters are read below
    # bytes per step as the library counted them for the last batch: es / ta / grad_out are read by both loss calls and
    # uploaded once; the mask (LCN's std) never crosses the bus upwards
    copied, saved = ctypes.c_uint64(0), ctypes.c_uint64(0)
    L.ctd_host_batch_stats(ctypes.byref(copied), ctypes.byref(saved))
    h2d = int(copied.value)
    assert h2d == 4 * npx * 4 and h2d + int(saved.value) == (1 + 4 + 4) * npx * 4, "host API byte accounting"
    d2h = (2 + 1 + 1) * npx * 4 + 16

    strong_block = None
    if not args.no_strong and not strong:
        strong_block = run_strong_block(args, rank, world, dev, sync_all)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = measured_peak()
    ops = {}
    for n in OPS + ("sad_fwd", "sad_bwd", "census_sad_fwd", "census_sad_bwd", "masked_sums"):
        gbs = BYTES_PER_PX[n] * npx / (op_ms[n] * 1e-3) / 1e9
        ops[n] = {"ms": op_ms[n], "mpix_s": npx / (op_ms[n] * 1e-3) / 1e6, "algo_bytes_per_px": BYTES_PER_PX[n],
                  "achieved_gbs": gbs, "frac_hbm": gbs / peak, "in_step": n in OPS}
    dom = max(OPS[:3], key=lambda n: op_ms[n])
    traffic, traffic_src = None, None
    try:  # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        traffic, traffic_src = tj["kernels"][dom]["dram_bytes"], tj["source"]
    except Exception:
        pass
    hbm = {"achieved": ops[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": ops[dom]["frac_hbm"], "peak_source": peak_src,
           "algo_bytes_per_launch": BYTES_PER_PX[dom] * npx}
    if dom == "census_sad_fwd_bwd":
        # the census kernels are bound by the XU (MUFU) pipe: the fused gather kernel evaluates 81 taps x 2 reciprocal square
        # roots per pixel; 16 MUFU lanes per clock and SM, 148 SMs, at the SM clock sampled during the timed region
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        xu_peak = 148 * 16 * sm_mhz * 1e6 / 1e9
        xu_ach = 162.0 * npx / (op_ms[dom] * 1e-3) / 1e9
        roofline = {"kernel": dom, "bound": "xu", "achieved": xu_ach, "peak": xu_peak, "unit": "G MUFU.RSQ/s", "frac": xu_ach / xu_peak,
                    "mufu_per_px": 162, "floor_ms_per_launch": 162.0 * npx / (xu_peak * 1e9) * 1e3,
                    "peak_source": "148 SMs x 16 XU lanes/clk x %.0f MHz (SM clock sampled under load)" % sm_mhz, "hbm": hbm,
                    "note": "162 reciprocal square roots per pixel put this kernel on the XU pipe, not on HBM (ncu: profiles/); frac against "
                            "HBM is in `hbm` and stays small by construction"}
    else:
        roofline = dict(hbm, kernel=dom, bound="hbm")
    roofline.update({"traffic": traffic, "traffic_source": traffic_src, "ms_per_launch": op_ms[dom],
                     "share_of_step": op_ms[dom] / sum(op_ms[n] for n in OPS)})
    cfg = workload_config(world, B, args.global_batch if strong else None)
    line = {"metric": METRIC, "value": npx_global / (ms_per_step * 1e-3) / 1e6, "unit": "Mpix/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "timing": {"footprint_mb": footprint_mb,
                       "launch": ("one CUDA graph replay per step" + (", consecutive steps on %d alternating streams" % min(max(args.pipeline, 1), NSETS) if args.pipeline > 1 else "") + (", the sad and the census loss as parallel branches behind LCN (both need its std, not each other)" if args.fork else "") + "; the last replay of each buffer set in the timed region is the plain chain with the event-record nodes the per-op durations are read from") if use_graph else "stream launches",
                       "parallelism": "batch-sharded x%d; one packed NCCL all-reduce of %d floats per %d steps on a side stream, two alternating scalar slots so no step waits for the previous round's reduction" % (world, NSETS * 4, NSETS) if world > 1 else "one GPU"},
            "sequential": {"ms_per_step": seq_ms, "value": npx_global / (seq_ms * 1e-3) / 1e6, "steps": seq_steps,
                           "note": "the same steps on ONE stream as ONE chain (no overlap between steps or between the two losses): what a training step that needs each loss before the next op would see"},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": npx_global / (e2e_ms * 1e-3) / 1e6, "unit": "Mpix/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "steps": e2e_steps,
                    "one_step_at_a_time": {"ms_per_step": e2e_sync_ms, "value": npx_global / (e2e_sync_ms * 1e-3) / 1e6},
                    "pipelining": "two steps in flight (ctd_host_end_batch_async / ctd_host_wait_batch): the uploads of step k + 1 run under the downloads of step k; every step's copies are inside the timed region",
                    "api": "ctd_host_begin_batch; ctd_host_lcn_f32 + 2x ctd_host_photometric_fwd_bwd_masked_f32 (loss scalars + d loss / d es; loss maps stay on the device, mask = the batch's own LCN std); ctd_host_end_batch_async, then ctd_host_wait_batch for the step before -- pinned host buffers; es / ta / grad_out uploaded once"},
            "roofline": roofline, "ops": ops,
            "separate_calls": {"ms_per_step": sep_ms_per_step, "value": npx_global / (sep_ms_per_step * 1e-3) / 1e6, "steps": sep_steps,
                               "note": "same chain, forward and backward of both losses as separate calls (torch autograd path)"}}
    if strong_block is not None:
        line["strong"] = strong_block
    if world == 1 and not args.no_extra:
        # the other ops of the path (configs[2], configs[3]) and the reference's OWN CUDA extension on the same GPU and buffers
        try:
            del sets, host_sets
            torch.cuda.empty_cache()
            from tools import bench_ops
            extra = bench_ops.run("xcorrvol,proj_nn,crosscheck,config4,nn,gpu_reference", iters=10, batch=B, device_index=local_rank, verbose=False)
            for n in ("xcorrvol_D128_bs9", "xcorrvol_D128_bs5", "proj_nn_ps3_12pairs", "proj_nn_ps5_12pairs", "config4_geometric_step_4frames", "nn_16384x16384"):
                if n in extra["ops"]:
                    ops[n] = dict(extra["ops"][n], in_step=False, ms=extra["ops"][n]["ms_median"])
            for n, v in extra["ops"].items():
                if n.startswith("crosscheck_"):
                    ops[n] = dict(v, in_step=False, ms=v["ms_median"], note="working set below L2: not an HBM figure")
            gr = extra.get("gpu_reference")
            if isinstance(gr, dict) and "unavailable" not in gr:
                mine = {"lcn_fwd": op_ms["lcn_fwd"], "sad_fwd": op_ms["sad_fwd"], "sad_bwd": op_ms["sad_bwd"],
                        "census_sad_fwd": op_ms["census_sad_fwd"], "census_sad_bwd": op_ms["census_sad_bwd"]}
                for n, v in gr.items():
                    m = mine.get(n, ops.get(n, {}).get("ms"))
                    if m:
                        v["this_ms"], v["ratio"] = m, v["ms"] / m
                line["gpu_reference"] = {"what": "the reference's own CUDA extension (torchext/ext/ext_cuda.cpp + ext_kernel.cu, unmodified, built for sm_100 into oracle/_ref) and its torch LCN on this GPU, same buffers, stream launches on the legacy stream as the reference issues them; ms per call at batch %d" % B,
                                         "ops": gr}
            else:
                line["gpu_reference"] = gr
        except Exception as e:
            line["gpu_reference"] = {"unavailable": "extra op timings failed: %s" % e}
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_leg()
    emit_line(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_IMAGES = 8  # six [8,1,480,640] float32 maps = 59 MB: the dump stays under 64 MB at any batch


def dump_outputs(out_dir, d):
    """What the last timed step hands its caller, as float32 .npy files in out_dir: LCN's two outputs, the loss map
    and d loss / d es of both losses (images 0..7 of the batch; a larger batch repeats those frames), and each
    loss's masked-mean terms over the whole batch (sum(std * loss), sum(std)).  Inputs are seeded, so two builds run
    with the same arguments can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    n = DUMP_IMAGES
    arrays = {"lcn": d["lcn"][:n], "lcn_std": d["std"][:n], "sad_loss": d["out_sad"][:n], "sad_grad": d["gi_sad"][:n],
              "census_sad_loss": d["out_cs"][:n], "census_sad_grad": d["gi_cs"][:n],
              "sad_masked_sums": d["sums"][0], "census_sad_masked_sums": d["sums"][1]}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float32))


def run_strong_block(args, rank, world, dev, sync_all):
    """BASELINE configs[4] as stated: a FIXED global batch of 64 frames (16 tracks of 4 frames) split over the ranks by
    shard_range, the ops of configs 2 and 4 -- LCN, sad and census_sad forward+backward with their masked sums, ProjNN
    (patch 3) in both directions for the 6 frame pairs of every track and CrossCheck in both directions -- and ONE packed
    all-reduce of the loss scalars per step.  Device-resident inputs on two rotating sets; returns the block for the JSON
    line (rank 0) after the max-over-ranks timing."""
    import torch
    import torch.distributed as dist
    from connecting_the_dots_b200 import _lib, synth, shard_range
    GB, T = 64, 4
    lo, hi = shard_range(GB // T, rank, world)     # whole tracks per rank
    ntr = hi - lo
    if ntr <= 0:
        return {"unavailable": "more ranks than tracks"}
    B = ntr * T
    npx = B * H * W
    base = synth.make_batch(8, H, W)
    xyz, K, poses = synth.make_clouds(T, H, W)
    pairs = [(i, j) for i in range(T) for j in range(T) if i != j]
    rev = [pairs.index((j, i)) for i, j in pairs]
    x0_1 = np.stack([synth.transform(xyz[i], poses[j]) for i, j in pairs])
    x1_1 = np.stack([xyz[j] for i, j in pairs])
    nq = len(pairs) * ntr
    NS = 2
    sets = []
    for s in range(NS):
        d = {k: torch.from_numpy(np.ascontiguousarray(np.roll(np.concatenate([base[k]] * ((B + 7) // 8))[:B], 3 * s + rank, axis=2))).to(dev) for k in ("im", "es", "ta", "go")}
        for k in ("lcn", "std", "out_sad", "gi_sad", "out_cs", "gi_cs"):
            d[k] = torch.empty(B, 1, H, W, device=dev)
        d["x0"] = torch.from_numpy(np.ascontiguousarray(np.roll(x0_1, s, axis=2))).to(dev).repeat(ntr, 1, 1, 1)
        d["x1"] = torch.from_numpy(np.ascontiguousarray(np.roll(x1_1, s, axis=2))).to(dev).repeat(ntr, 1, 1, 1)
        d["idx"] = torch.empty(nq, H, W, dtype=torch.int64, device=dev)
        d["idx_rev"] = torch.empty_like(d["idx"])
        d["m"] = torch.empty(nq * H * W, dtype=torch.uint8, device=dev)
        d["sums"] = torch.zeros(2, 2, device=dev)
        sets.append(d)
    Kd = torch.from_numpy(K).to(dev)
    # reverse pair of query p inside its own track (indices are per-image local after subtracting the image offset)
    rev_t = torch.tensor([12 * (p // 12) + rev[p % 12] for p in range(nq)], device=dev)
    rebase = ((torch.arange(nq, device=dev, dtype=torch.int64) - rev_t.to(torch.int64)) * (H * W)).view(nq, 1, 1)
    zero = torch.zeros(1, 1, 1, dtype=torch.int64, device=dev)

    def step_body(d, st_):
        p = {n: t.data_ptr() for n, t in d.items()}
        _lib.call("ctd_lcn_f32", p["im"], p["lcn"], p["std"], B, H, W, LCN_R, LCN_EPS, st_)
        _lib.call("ctd_photometric_fwd_bwd_masked_f32", p["es"], p["ta"], p["go"], p["std"], p["out_sad"], p["gi_sad"], p["sums"], B, 1, H, W, BS, 1, EPS, st_)
        _lib.call("ctd_photometric_fwd_bwd_masked_f32", p["es"], p["ta"], p["go"], p["std"], p["out_cs"], p["gi_cs"], p["sums"] + 8, B, 1, H, W, BS, 3, EPS, st_)
        _lib.call("ctd_proj_nn_f32", p["x0"], p["x1"], Kd.data_ptr(), p["idx"], nq, H, W, 3, st_)
        # ProjNN's indices are flat over the launch batch; CrossCheck pairs query p with its reverse query: re-base the
        # reverse query's indices onto p's image offsets (two elementwise torch kernels, inside the timed step)
        torch.index_select(d["idx"], 0, rev_t, out=d["idx_rev"])
        d["idx_rev"].add_(torch.where(d["idx_rev"] >= 0, rebase, zero))
        _lib.call("ctd_crosscheck", p["idx"], p["idx_rev"], p["m"], nq * H * W, nq * H * W, st_)

    cur = torch.cuda.current_stream(dev)
    step_body(sets[0], cur.cuda_stream)
    torch.cuda.synchronize(dev)
    graphs = []
    try:
        for d in sets:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                step_body(d, torch.cuda.current_stream(dev).cuda_stream)
            graphs.append(g)
    except Exception as e:
        print("bench: strong block: graph capture failed (%s); stream launches" % e, file=sys.stderr)
        graphs = []
        torch.cuda.synchronize(dev)
    comm = torch.cuda.Stream(dev) if world > 1 else None

    def run_steps(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        e0.record(cur)
        done = None
        for k in range(n):
            d = sets[k % NS]
            if done is not None and k % NS == 0:
                cur.wait_event(done)
            if graphs:
                graphs[k % NS].replay()
            else:
                step_body(d, cur.cuda_stream)
            if world > 1:
                comm.wait_stream(cur)
                with torch.cuda.stream(comm):
                    dist.all_reduce(d["sums"])   # 4 floats: the packed scalars of the step
                    done = comm.record_event()
        if world > 1:
            cur.wait_stream(comm)
        e1.record(cur)
        sync_all()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / n

    run_steps(3)
    n = max(4, min(args.steps, 10))
    ms = run_steps(n)
    valid = float((sets[(n - 1) % NS]["m"] > 0).float().mean())
    for d in sets:
        d.clear()
    del sets
    torch.cuda.empty_cache()
    return {"what": "BASELINE configs[4]: global batch 64 (16 tracks x 4 frames) split over the ranks; LCN + sad f+b + census_sad f+b (fused, masked sums) on the frames, ProjNN patch 3 both ways for the 6 frame pairs of each track + CrossCheck; one packed 4-float all-reduce per step",
            "global_batch": GB, "batch_per_gpu": B, "proj_nn_queries_per_gpu": nq, "n_gpus": world, "steps": n, "ms_per_step": ms,
            "value": GB * H * W / (ms * 1e-3) / 1e6, "unit": "Mpix/s (frames)", "scaling": "strong",
            "crosscheck_mutual_fraction": valid,
            "l2_policy": "two rotating input/output sets, %.0f MB per set per GPU" % ((10 * npx * 4 + nq * H * W * (24 + 16 + 1)) / 1e6)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=("b200", "reference"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time plain stream launches instead of CUDA graph replays")
    ap.add_argument("--pipeline", type=int, default=4, help="steps in flight (replayed on that many alternating streams, at most one per buffer set); 1 = one stream")
    ap.add_argument("--fork", type=int, default=1,
                    help="the two losses as parallel graph branches behind LCN (1: sad on the side stream, 2: census; 0: one chain)")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="run the MAIN figure as strong scaling: split this many images over the ranks instead of 8 per GPU")
    ap.add_argument("--census-sym", type=int, default=-1, help="A/B runs: ctd_set_option('census_sym', v) before the benchmark (0 gather kernels, 1 pair-symmetric kernel everywhere, 2 automatic = library default)")
    ap.add_argument("--no-strong", action="store_true", help="skip the `strong` block (BASELINE configs[4]: global batch 64 over the ranks)")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra op timings (XCorrVol, ProjNN, ...) and the reference CUDA extension leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the B200 path's outputs; the reference arm times a CPU sample and keeps none")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl != "reference" and world == 1 and args.gpus > 1:
        # plain `python bench.py --gpus N`: re-launch under torchrun, one rank per GPU (before stdout is re-pointed)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(29400 + os.getpid() % 500), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    run_b200_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
