"""A/B timings of the census kernels at the bench size, every entry point: pair-symmetric (census_sym.cu), tile
(photometric.cu) and the automatic dispatch.  python tools/experiments/census_sym_ab.py [batch]"""
import os, sys, json
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np, torch
from connecting_the_dots_b200 import _lib, synth
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_ops import timeit
B = int(sys.argv[1]) if len(sys.argv) > 1 else 8
H, W = 480, 640
dev = torch.device("cuda", 0)
base = synth.make_batch(min(B, 8), H, W)
if B > 8:
    base = {k: np.concatenate([v] * ((B + 7) // 8))[:B] for k, v in base.items()}
NS = 5 if B <= 8 else 2
sets = []
for s in range(NS):
    d = {k: torch.from_numpy(np.ascontiguousarray(np.roll(base[k], 5 * s, axis=2))).to(dev) for k in ("es", "ta", "go", "std")}
    d["o1"], d["o2"], d["sums"] = torch.empty(B, 1, H, W, device=dev), torch.empty(B, 1, H, W, device=dev), torch.zeros(2, device=dev)
    sets.append(d)
res = {}
for label, opts in (("sym", {"census_sym": 1}), ("tile", {"census_sym": 0}), ("auto", {})):
    for k, v in opts.items():
        _lib.set_option(k, v)
    for ty in (2, 3):
        def fwd(i, st):
            d = sets[i % NS]
            _lib.call("ctd_photometric_fwd_f32", d["es"].data_ptr(), d["ta"].data_ptr(), d["o1"].data_ptr(), B, 1, H, W, 9, ty, 0.5, st)
        def bwd(i, st):
            d = sets[i % NS]
            _lib.call("ctd_photometric_bwd_f32", d["es"].data_ptr(), d["ta"].data_ptr(), d["go"].data_ptr(), d["o2"].data_ptr(), B, 1, H, W, 9, ty, 0.5, st)
        def fused(i, st):
            d = sets[i % NS]
            _lib.call("ctd_photometric_fwd_bwd_masked_f32", d["es"].data_ptr(), d["ta"].data_ptr(), d["go"].data_ptr(), d["std"].data_ptr(),
                      d["o1"].data_ptr(), d["o2"].data_ptr(), d["sums"].data_ptr(), B, 1, H, W, 9, ty, 0.5, st)
        for name, f in (("fwd", fwd), ("bwd", bwd), ("fused_masked", fused)):
            res["%s_t%d_%s" % (label, ty, name)] = round(timeit(f, 10)[0] * 1e3, 1)
    _lib.set_option("census_sym", 2)
print(json.dumps(res, indent=1))
