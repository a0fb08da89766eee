#!/usr/bin/env python
"""Error of the fp32 SSIM kernels against the float64 restatement (max |got - ref| / max |ref|, the repo comparator's
figure) on three kinds of input: randn pairs, raw IR frames in [0, 1] with clipped flat regions, and frames whose mean
is far above their local contrast (10 +- 0.1, the case DESIGN section 4.11 does not guarantee 1e-5 for).  Prints one
JSON object.

    python tools/experiments/ssim_error.py"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import connecting_the_dots_b200 as ctd  # noqa: E402
from connecting_the_dots_b200 import synth  # noqa: E402


def rel(a, b):
    return float((a.double() - b).abs().max() / b.abs().max())


def main():
    tx = ctd.torchext
    dev = "cuda:0"
    rng = np.random.RandomState(0)
    d = synth.make_batch(2)
    im = d["im"]
    x = rng.randn(2, 1, 480, 640).astype(np.float32)
    inputs = {
        "randn": (x, (x + 0.5 * rng.randn(*x.shape)).astype(np.float32)),
        "ir_0_1": (im, np.ascontiguousarray(np.roll(im, 2, axis=3))),
        "offset_10_pm_0.1": ((10 + 0.1 * (2 * im - 1)).astype(np.float32),
                             (10 + 0.1 * (2 * np.roll(im, 2, axis=3) - 1)).astype(np.float32)),
    }
    go = torch.from_numpy(d["go"]).to(dev)
    res = {"device": torch.cuda.get_device_name(0), "shape": [2, 1, 480, 640]}
    for name, (es, ta) in inputs.items():
        for bs in (3, 9):
            e = torch.from_numpy(es).to(dev).requires_grad_(True)
            t = torch.from_numpy(ta).to(dev)
            out = tx.ssim_loss(e, t, bs)
            (g,) = torch.autograd.grad(out, e, go)
            e64 = e.detach().double().requires_grad_(True)
            ref = tx.ssim_loss_pytorch(e64, t.double(), bs)
            (gref,) = torch.autograd.grad(ref, e64, go.double())
            res["%s_bs%d" % (name, bs)] = {"fwd": rel(out.detach(), ref.detach()), "bwd": rel(g, gref)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
