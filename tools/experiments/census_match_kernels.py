#!/usr/bin/env python
"""Per-kernel device times of the census matching calls (torch.profiler, CUDA activities) at batch 8 x 480x640, D = 128, on
the bench's synthetic frames (ta against pat_lcn), 7x9 window: ctd_census_vol_f32 at block 1 and 9 and
ctd_census_disparity_f32 at block 9 and 1 (sub-pixel on).  Each kernel's time is set against its traffic floor (from
shapes, tools/bench_ops.census_traffic) at the HBM bandwidth DESIGN section 3 measured.  Prints one JSON object with the
GPU's name and power limit read in the same run.

    python tools/experiments/census_match_kernels.py > profiles/r06_census_match_kernels.json
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
from bench_ops import PEAK, census_traffic, device_info  # noqa: E402

B, H, W, D, REPS = 8, 480, 640, 128, 5


def main():
    d = synth.make_batch(B)
    a, b = torch.from_numpy(d["ta"]).cuda(), torch.from_numpy(d["pat_lcn"]).cuda()
    st = torch.cuda.current_stream().cuda_stream
    vol = torch.empty(B, D, H, W, device="cuda")
    disp, score = torch.empty(B, 1, H, W, device="cuda"), torch.empty(B, 1, H, W, device="cuda")
    npx = B * H * W
    floors = census_traffic(B, 1, H, W, D)
    out = {"batch": B, "height": H, "width": W, "n_disps": D, "window": [7, 9], "peak_gbs": PEAK, "device": device_info(0),
           "floor_bytes": dict(floors, transform_per_input=12 * npx), "us_per_call": {}}
    calls = {
        "vol_bs1": lambda: _lib.call("ctd_census_vol_f32", a.data_ptr(), b.data_ptr(), vol.data_ptr(), B, 1, H, W, D, 7, 9, 1, st),
        "vol_bs9": lambda: _lib.call("ctd_census_vol_f32", a.data_ptr(), b.data_ptr(), vol.data_ptr(), B, 1, H, W, D, 7, 9, 9, st),
        "disparity_bs9": lambda: _lib.call("ctd_census_disparity_f32", a.data_ptr(), b.data_ptr(), disp.data_ptr(), score.data_ptr(),
                                           B, 1, H, W, D, 7, 9, 9, 1, st),
        "disparity_bs1": lambda: _lib.call("ctd_census_disparity_f32", a.data_ptr(), b.data_ptr(), disp.data_ptr(), score.data_ptr(),
                                           B, 1, H, W, D, 7, 9, 1, 1, st),
    }
    for name, run in calls.items():
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as p:
            for _ in range(REPS):
                run()
            torch.cuda.synchronize()
        rows = {}
        for e in p.key_averages():
            if e.self_device_time_total > 0:
                m = re.search(r"(census_\w+<[^>]*>)", e.key)
                key = m.group(1) if m else e.key[:80]
                us = e.self_device_time_total / REPS
                row = {"us_per_call": round(us, 1), "launches_per_call": e.count // REPS}
                # traffic floors: the transform reads 4 B and writes 8 B per pixel (two launches a call); the match kernel
                # writes the volume (4D B/px) or disp and score (8 B/px) and reads the descriptors once (16 B/px)
                if "transform" in key:
                    row["floor_bytes"] = 12 * npx * (e.count // REPS)
                elif "census_match" in key:
                    row["floor_bytes"] = (4 * D * npx if name.startswith("vol") else 8 * npx) + 16 * npx
                if "floor_bytes" in row:
                    row["frac_floor_at_peak"] = round(row["floor_bytes"] / (us * 1e-6) / 1e9 / PEAK, 3)
                rows[key] = row
        out["us_per_call"][name] = rows
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
