"""Generate tests/golden/xcorrvol_full.npz: BASELINE configs[2] at ITS OWN SIZE from the UNMODIFIED reference.

One 480x640 synthetic LCN'd pair (frame 0 of connecting_the_dots_b200.synth.make_batch(8): in0 = the LCN'd IR image,
in1 = the LCN'd dot pattern), D = 128 disparities, block 9 and block 5, evaluated by the reference's own CPU extension
(oracle/_ref/ctd_ref_ext_cpu.so: xcorrvol_cpu, ext_cpu.cpp:88-105, ~17 s + ~6 s).  The full volume is 157 MB per
block size, so the fixture keeps 16 of the 480 rows (image border rows, rows next to them, interior rows), 64 of the
640 columns and all 128 disparities: 0.52 MB per block size.  The columns are the 9 at each border (the window leaves
the image), two on each side of the kernels' 128-column CTA edges, 16 seeded columns in 9..125 (x - d < 0 for many d:
the in1 window is clamped) and 14 seeded columns elsewhere.  The GPU test runs the batched B = 8 call and compares
image 0 at those rows and columns (tests/test_gpu_ops.py: test_xcorrvol_full_size_golden).

    python tests/golden/make_golden_full.py      # in the build container only (/root/reference is not on the GPU box)
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import build_ref  # noqa: E402
from connecting_the_dots_b200 import synth  # noqa: E402

ROWS = np.array([0, 1, 3, 4, 5, 37, 101, 165, 229, 240, 293, 357, 421, 474, 476, 479])
EDGES = np.array([c + o for c in (128, 256, 384, 512) for o in (-2, -1, 0, 1)])   # xcorrvol.cu: 128 columns per CTA
_rs = np.random.RandomState(0)
COLS = np.unique(np.concatenate([np.arange(9), _rs.choice(np.arange(9, 126), 16, replace=False), EDGES,
                                 _rs.choice(np.setdiff1d(np.arange(130, 631), EDGES), 14, replace=False), np.arange(631, 640)]))


def main():
    build_ref.build()
    ref = build_ref.load_ref()
    assert ref is not None, "reference extension not built"
    torch.set_num_threads(1)
    d = synth.make_batch(8, 480, 640)
    in0 = np.ascontiguousarray(d["ta"][0])       # [1,480,640]
    in1 = np.ascontiguousarray(d["pat_lcn"][0])
    out = {"rows": ROWS, "cols": COLS, "in0_sum": np.float64(in0.astype(np.float64).sum()), "in1_sum": np.float64(in1.astype(np.float64).sum()),
           "in0_row240": in0[0, 240].copy(), "in1_row240": in1[0, 240].copy()}
    for bs in (9, 5):
        vol = ref.xcorrvol_cpu(torch.from_numpy(in0), torch.from_numpy(in1), 128, bs).numpy()   # [128,480,640]
        out["bs%d" % bs] = np.ascontiguousarray(vol[:, ROWS][:, :, COLS])
        print("bs", bs, "done", vol.shape, float(np.abs(vol).max()), flush=True)
    np.savez_compressed(os.path.join(HERE, "xcorrvol_full.npz"), **out)


if __name__ == "__main__":
    main()
