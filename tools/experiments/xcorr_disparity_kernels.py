#!/usr/bin/env python
"""Per-kernel device times of one ctd_xcorr_disparity_f32 call (torch.profiler, CUDA activities) at batch 8 x 480x640,
D = 128, blocks 9 and 5, with and without sub-pixel refinement, on the bench's synthetic LCN'd frames.  Prints one JSON
object with the GPU's name and power limit read in the same run.

    python tools/experiments/xcorr_disparity_kernels.py > profiles/r04_xcorr_disparity_kernels.json
"""
import json
import os
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
    disp, score = torch.empty(B, 1, H, W, device="cuda"), torch.empty(B, 1, H, W, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    out = {"batch": B, "height": H, "width": W, "n_disps": D, "device": device_info(0), "us_per_call": {}}
    for bs in (9, 5):
        for sub in (1, 0):
            def run():
                _lib.call("ctd_xcorr_disparity_f32", a.data_ptr(), b.data_ptr(), disp.data_ptr(), score.data_ptr(), B, 1, H, W, D,
                          bs, sub, st)
            for _ in range(3):
                run()
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as p:
                for _ in range(REPS):
                    run()
                torch.cuda.synchronize()
            rows = {e.key.split("(")[0]: round(e.self_device_time_total / REPS, 1)
                    for e in p.key_averages() if e.self_device_time_total > 0}
            out["us_per_call"]["bs%d_subpixel%d" % (bs, sub)] = rows
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
