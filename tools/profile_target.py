import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from connecting_the_dots_b200 import _lib, synth
H, W, B = 480, 640, 8
base = synth.make_batch(B, H, W)
d = {k: torch.from_numpy(base[k]).cuda() for k in ("im", "es", "ta", "go", "std", "pat_lcn")}
o = [torch.empty(B, 1, H, W, device="cuda") for _ in range(6)]
ws = torch.zeros(int(_lib.lib().ctd_masked_sums_workspace_bytes()), dtype=torch.uint8, device="cuda")
sums = torch.zeros(2, device="cuda")
st = torch.cuda.current_stream().cuda_stream
p = {k: v.data_ptr() for k, v in d.items()}
for rnd in range(2):
    _lib.call("ctd_lcn_f32", p["im"], o[0].data_ptr(), o[1].data_ptr(), B, H, W, 5, 0.05, st)
    _lib.call("ctd_photometric_fwd_f32", p["es"], p["ta"], o[2].data_ptr(), B, 1, H, W, 9, 1, 0.5, st)
    _lib.call("ctd_photometric_bwd_f32", p["es"], p["ta"], p["go"], o[3].data_ptr(), B, 1, H, W, 9, 1, 0.5, st)
    _lib.call("ctd_photometric_fwd_f32", p["es"], p["ta"], o[4].data_ptr(), B, 1, H, W, 9, 3, 0.5, st)
    _lib.call("ctd_photometric_bwd_f32", p["es"], p["ta"], p["go"], o[5].data_ptr(), B, 1, H, W, 9, 3, 0.5, st)
    _lib.call("ctd_photometric_fwd_bwd_masked_f32", p["es"], p["ta"], p["go"], p["std"], o[2].data_ptr(), o[3].data_ptr(), sums.data_ptr(),
              B, 1, H, W, 9, 1, 0.5, st)
    _lib.call("ctd_photometric_fwd_bwd_masked_f32", p["es"], p["ta"], p["go"], p["std"], o[4].data_ptr(), o[5].data_ptr(), sums.data_ptr(),
              B, 1, H, W, 9, 3, 0.5, st)
    _lib.call("ctd_masked_sums_f32", o[4].data_ptr(), p["std"], B * H * W, sums.data_ptr(), ws.data_ptr(), st)
    torch.cuda.synchronize()
