#!/usr/bin/env python
"""Per-kernel device times of one ctd_sgm_f32 call (torch.profiler, CUDA activities) at batch 8 x 480x640, D = 128, on the
xcorrvol block-9 volume of the bench's synthetic frames, with 4 and 8 paths and with and without the fused winner-take-all.
Prints one JSON object with the GPU's name and power limit read in the same run.

    python tools/experiments/sgm_kernels.py > profiles/r05_sgm_kernels.json
"""
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from connecting_the_dots_b200 import _lib, synth  # noqa: E402
from bench_ops import device_info  # noqa: E402

B, H, W, D, REPS = 8, 480, 640, 128, 5


def main():
    d = synth.make_batch(B)
    a, b = torch.from_numpy(d["ta"]).cuda(), torch.from_numpy(d["pat_lcn"]).cuda()
    st = torch.cuda.current_stream().cuda_stream
    vol = torch.empty(B, D, H, W, device="cuda")
    _lib.call("ctd_xcorrvol_f32", a.data_ptr(), b.data_ptr(), vol.data_ptr(), B, 1, H, W, D, 9, st)
    agg = torch.empty_like(vol)
    disp, score = torch.empty(B, 1, H, W, device="cuda"), torch.empty(B, 1, H, W, device="cuda")
    out = {"batch": B, "height": H, "width": W, "n_disps": D, "device": device_info(0), "us_per_call": {}}
    for paths in (4, 8):
        for wta in (1, 0):
            def run():
                _lib.call("ctd_sgm_f32", vol.data_ptr(), agg.data_ptr(), disp.data_ptr() if wta else None,
                          score.data_ptr() if wta else None, B, D, H, W, 0.2, 2.0, paths, 1, st)
            for _ in range(3):
                run()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as p:
                for _ in range(REPS):
                    run()
                torch.cuda.synchronize()
            # one row per kernel instance; the line kernel runs once per vertical or diagonal path, so its row is the sum
            rows = {}
            for e in p.key_averages():
                if e.self_device_time_total > 0:
                    m = re.search(r"(sgm_\w+<[^>]*>)", e.key)
                    rows[m.group(1) if m else e.key[:80]] = {"us_per_call": round(e.self_device_time_total / REPS, 1),
                                                             "launches_per_call": e.count // REPS}
            out["us_per_call"]["paths%d_wta%d" % (paths, wta)] = rows
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
