"""nn.Module layer of the drop-in torchext package.

CoordConv2d is the one module the reference ships (torchext/modules.py:7-27).  The others are thin
nn.Module faces of the ops for callers that want modules (BASELINE.json's naming); `LCN` is a drop-in
for model.networks.LCN (model/networks.py:507-533): same constructor, forward returns (lcn, std)."""
import torch

from .functions import *  # noqa: F401,F403
from . import functions as F


class CoordConv2d(torch.nn.Module):
    """Conv2d over the input with two extra channels holding the pixel coordinates in [-1, 1]."""

    def __init__(self, channels_in, channels_out, kernel_size, stride, padding):
        super().__init__()
        self.conv = torch.nn.Conv2d(channels_in + 2, channels_out, kernel_size=kernel_size, padding=padding, stride=stride)
        self.uv = None

    def _grid(self, x):
        h, w = x.shape[2], x.shape[3]
        if self.uv is None or self.uv.shape[2:] != (h, w) or self.uv.device != x.device:
            u = torch.linspace(-1, 1, w, device=x.device, dtype=torch.float32).view(1, 1, 1, w).expand(1, 1, h, w)
            v = torch.linspace(-1, 1, h, device=x.device, dtype=torch.float32).view(1, 1, h, 1).expand(1, 1, h, w)
            self.uv = torch.cat((u, v), dim=1)
        return self.uv

    def forward(self, x):
        uv = self._grid(x).expand(x.shape[0], -1, -1, -1)
        return self.conv(torch.cat((x, uv), dim=1))


class PhotometricLoss(torch.nn.Module):
    def __init__(self, block_size=9, type="census_sad", eps=0.5):
        super().__init__()
        self.block_size, self.type, self.eps = block_size, type, eps

    def forward(self, es, ta):
        return F.photometric_loss(es, ta, self.block_size, self.type, self.eps)


class SSIMLoss(torch.nn.Module):
    """forward(es, ta) -> ssim_loss map [B,1,H,W]."""

    def __init__(self, block_size=3, c1=F.SSIM_C1, c2=F.SSIM_C2):
        super().__init__()
        self.block_size, self.c1, self.c2 = block_size, c1, c2

    def forward(self, es, ta):
        return F.ssim_loss(es, ta, self.block_size, self.c1, self.c2)


class XCorrVol(torch.nn.Module):
    def __init__(self, n_disps=128, block_size=9):
        super().__init__()
        self.n_disps, self.block_size = n_disps, block_size

    def forward(self, in0, in1):
        return F.xcorrvol(in0, in1, self.n_disps, self.block_size)


class XCorrDisparity(torch.nn.Module):
    """forward(in0, in1) -> (disp, score) of xcorr_disparity: the winner-take-all disparity of XCorrVol's volume."""

    def __init__(self, n_disps=128, block_size=9, subpixel=True):
        super().__init__()
        self.n_disps, self.block_size, self.subpixel = n_disps, block_size, subpixel

    def forward(self, in0, in1):
        return F.xcorr_disparity(in0, in1, self.n_disps, self.block_size, self.subpixel)


class SGMDisparity(torch.nn.Module):
    """forward(in0, in1) -> (disp, score): xcorrvol(in0, in1, n_disps, block_size), then sgm_disparity over it.  The
    default penalties (p1 = 0.2, p2 = 2.0 on the correlation scale, 8 paths) were tuned on two synthetic frames only."""

    def __init__(self, n_disps=128, block_size=9, p1=0.2, p2=2.0, paths=8, subpixel=True):
        super().__init__()
        self.n_disps, self.block_size, self.p1, self.p2, self.paths, self.subpixel = n_disps, block_size, p1, p2, paths, subpixel

    def forward(self, in0, in1):
        return F.sgm_disparity(F.xcorrvol(in0, in1, self.n_disps, self.block_size), self.p1, self.p2, self.paths, self.subpixel)


class CensusDisparity(torch.nn.Module):
    """forward(in0, in1) -> (disp, score) of census_disparity: the winner-take-all disparity of census_vol's volume."""

    def __init__(self, n_disps=128, window=(7, 9), block_size=9, subpixel=True):
        super().__init__()
        self.n_disps, self.window, self.block_size, self.subpixel = n_disps, tuple(window), block_size, subpixel

    def forward(self, in0, in1):
        return F.census_disparity(in0, in1, self.n_disps, self.window, self.block_size, self.subpixel)


class CensusSGMDisparity(torch.nn.Module):
    """forward(in0, in1) -> (disp, score): census_vol(in0, in1, n_disps, window, block_size), then sgm_disparity over it.
    The default penalties (p1 = 6, p2 = 400 in Hamming units, 8 paths) were tuned on two synthetic frames only: a CPU sweep
    of the definition over p1 in 3..16 and p2 in 100..1000 on synth.make_batch(2) put 0.911 (8 paths) and 0.913 (4 paths)
    of the interior pixels within 2 px of the ground truth, against 0.849 and 0.789 at p1 = 10, p2 = 120."""

    def __init__(self, n_disps=128, window=(7, 9), block_size=1, p1=6, p2=400, paths=8, subpixel=True):
        super().__init__()
        self.n_disps, self.window, self.block_size = n_disps, tuple(window), block_size
        self.p1, self.p2, self.paths, self.subpixel = p1, p2, paths, subpixel

    def forward(self, in0, in1):
        vol = F.census_vol(in0, in1, self.n_disps, self.window, self.block_size)
        return F.sgm_disparity(vol, self.p1, self.p2, self.paths, self.subpixel)


class DisparityCheck(torch.nn.Module):
    """forward(vol) -> (disp, score, valid) of disparity_check: the winner-take-all disparity of a score volume and the
    mask of pixels that pass the left-right consistency and uniqueness checks.
    DisparityCheck()(sgm_aggregate(census_vol(in0, in1, 128), 6, 400)) is a full classical stereo pipeline."""

    def __init__(self, max_diff=1, uniqueness=0.0, subpixel=True):
        super().__init__()
        self.max_diff, self.uniqueness, self.subpixel = max_diff, uniqueness, subpixel

    def forward(self, vol):
        return F.disparity_check(vol, self.max_diff, self.uniqueness, self.subpixel)


class CrossCheck(torch.nn.Module):
    def forward(self, in0, in1):
        return F.crosscheck(in0, in1)


class NN(torch.nn.Module):
    def forward(self, in0, in1):
        return F.nn(in0, in1)


class ProjNN(torch.nn.Module):
    def __init__(self, patch_size=3):
        super().__init__()
        self.patch_size = patch_size

    def forward(self, xyz0, xyz1, K):
        return F.proj_nn(xyz0, xyz1, K, self.patch_size)


class LCN(torch.nn.Module):
    """Drop-in for model.networks.LCN(radius, epsilon): forward(data) -> (lcn, std)."""

    def __init__(self, radius=5, epsilon=0.05):
        super().__init__()
        self.radius, self.epsilon = radius, epsilon

    def forward(self, data):
        return F.lcn(data, self.radius, self.epsilon)
