#!/usr/bin/env python
"""Per-kernel device times of one ctd_speckle_filter_f32 call (torch.profiler, CUDA activities), max_size 200, max_diff 1, at
batch 8 and 64 x 480x640, on three inputs: the census block-9 integer disparities of the bench's synthetic frames after
disparity_check(1, 0), the census block-1 -> sgm_disparity (8 paths) integer disparities, and a snake (one-pixel path
through every other row, the longest component an image holds).  Batch 64 repeats the 8 frames.  Prints one JSON object
with the GPU's name and power limit read in the same run.

    python tools/experiments/speckle_kernels.py > profiles/r08_speckle_kernels.json
"""
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

import connecting_the_dots_b200 as ctd  # noqa: E402
from connecting_the_dots_b200 import synth  # noqa: E402
from bench_ops import device_info  # noqa: E402

H, W, REPS = 480, 640, 10


def snake(B):
    d = np.where(np.arange(H)[:, None] % 2 == 0, 0.0, 10.0) * np.ones((1, W))
    d[1::4, W - 1] = 0.0
    d[3::4, 0] = 0.0
    return torch.from_numpy(np.ascontiguousarray(np.broadcast_to(d, (B, 1, H, W)))).float().cuda()


def main():
    tx = ctd.torchext
    d = synth.make_batch(8)
    a, b = torch.from_numpy(d["ta"]).cuda(), torch.from_numpy(d["pat_lcn"]).cuda()
    bm, _, ok = tx.disparity_check(tx.census_vol(a, b, 128, (7, 9), 9), 1, 0.0, subpixel=False)
    sgm = tx.sgm_disparity(tx.census_vol(a, b, 128, (7, 9), 1), 6, 400, 8, subpixel=False)[0]
    res = {"reps": REPS, "unit": "us per call", "device": device_info(0)}
    for B in (8, 64):
        r = B // 8
        for name, disp, valid in (("census_bs9_checked", bm.repeat(r, 1, 1, 1), ok.repeat(r, 1, 1, 1)),
                                  ("census_bs1_sgm", sgm.repeat(r, 1, 1, 1), None), ("snake", snake(B), None)):
            for _ in range(3):
                tx.speckle_filter(disp, valid, 200, 1.0)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as p:
                for _ in range(REPS):
                    tx.speckle_filter(disp, valid, 200, 1.0)
                torch.cuda.synchronize()
            ks = {}
            for e in p.events():
                m = re.search(r"speckle_(tiles|merge|sizes|mark)", e.name)
                if m:
                    ks[m.group(1)] = ks.get(m.group(1), 0.0) + e.device_time / REPS
            ks["total"] = sum(ks.values())
            res["b%d_%s" % (B, name)] = {k: round(v, 2) for k, v in ks.items()}
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
