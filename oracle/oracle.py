"""TEST INFRASTRUCTURE ONLY: numpy front-end of the plain-C oracle (oracle/ctd_oracle.c).

Argument meaning and return shapes mirror the reference's CPU entry points
(torchext/ext/ext_cpu.cpp:14-184) so tests read like calls into the reference.  Only
tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import this module.
"""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libctd_oracle.so")

LOSS_TYPES = {"mse": 0, "sad": 1, "census_mse": 2, "census_sad": 3}  # ext.h:196-199

_lib = None


def build():
    """Path of a libctd_oracle.so built from the current sources: the in-tree one, (re)built with the committed
    Makefile if it is missing or stale.  In a read-only tree a missing or stale library is built in a temporary
    directory instead (removed at exit)."""
    names = ("ctd_oracle.c", "ctd_oracle_impl.h", "Makefile")
    if os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(os.path.join(HERE, f)) for f in names):
        return LIB_PATH
    where = HERE
    if not os.access(HERE, os.W_OK):
        where = tempfile.mkdtemp(prefix="ctd_oracle_")
        atexit.register(shutil.rmtree, where, True)
        for f in names:
            shutil.copy(os.path.join(HERE, f), where)
    subprocess.run(["make", "-C", where, "libctd_oracle.so"], check=True, capture_output=True)
    return os.path.join(where, "libctd_oracle.so")


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _real(a, *more):
    a = np.ascontiguousarray(a)
    if a.dtype not in (np.float32, np.float64):
        raise NotImplementedError("oracle: float32/float64 only, got %s" % a.dtype)
    rest = [np.ascontiguousarray(m, dtype=a.dtype) for m in more]
    return (a, *rest, "_f32" if a.dtype == np.float32 else "_f64")


def _type_id(t):
    return LOSS_TYPES[t.lower()] if isinstance(t, str) else int(t)


def photometric_loss_forward(es, ta, block_size, type, eps):
    """ext_cpu.cpp:110-145.  es, ta [B,C,H,W] -> [B,1,H,W]."""
    es, ta, sfx = _real(es, ta)
    B, C, H, W = es.shape
    out = np.empty((B, 1, H, W), es.dtype)
    getattr(lib(), "ctdo_photometric_fwd" + sfx)(
        _p(es), _p(ta), _p(out), B, C, H, W, int(block_size), _type_id(type), ctypes.c_float(eps))
    return out


def photometric_loss_backward(es, ta, grad_out, block_size, type, eps):
    """ext_cpu.cpp:147-184.  grad_out [B,1,H,W] -> grad_in [B,C,H,W] (w.r.t. es only)."""
    es, ta, go, sfx = _real(es, ta, grad_out)
    B, C, H, W = es.shape
    gi = np.empty((B, C, H, W), es.dtype)
    getattr(lib(), "ctdo_photometric_bwd" + sfx)(
        _p(es), _p(ta), _p(go), _p(gi), B, C, H, W, int(block_size), _type_id(type), ctypes.c_float(eps))
    return gi


def xcorrvol(in0, in1, n_disps, block_size):
    """ext_cpu.cpp:88-105.  in0, in1 [C,H,W] -> [n_disps,H,W]."""
    in0, in1, sfx = _real(in0, in1)
    C, H, W = in0.shape
    out = np.empty((n_disps, H, W), in0.dtype)
    L = ctypes.c_long
    getattr(lib(), "ctdo_xcorrvol" + sfx)(_p(in0), _p(in1), _p(out), L(C), L(H), L(W), L(n_disps), L(block_size))
    return out


def proj_nn(xyz0, xyz1, K, patch_size):
    """ext_cpu.cpp:59-85.  xyz0, xyz1 [B,H,W,3], K [3,3] -> int64 [B,H,W]."""
    xyz0, xyz1, K, sfx = _real(xyz0, xyz1, K)
    B, H, W, _ = xyz0.shape
    out = np.empty((B, H, W), np.int64)
    L = ctypes.c_long
    getattr(lib(), "ctdo_proj_nn" + sfx)(_p(xyz0), _p(xyz1), _p(K), _p(out), L(B), L(H), L(W), L(patch_size))
    return out


def nn(in0, in1):
    """ext_cpu.cpp:14-36.  in0 [N0,3], in1 [N1,3] -> int64 [N0]."""
    in0, in1, sfx = _real(in0, in1)
    out = np.empty((in0.shape[0],), np.int64)
    L = ctypes.c_long
    getattr(lib(), "ctdo_nn" + sfx)(_p(in0), _p(in1), _p(out), L(in0.shape[0]), L(in1.shape[0]))
    return out


def crosscheck(in0, in1):
    """ext_cpu.cpp:39-56.  in0 int64 [N0], in1 int64 [N1] -> uint8 [N0]."""
    in0 = np.ascontiguousarray(in0, dtype=np.int64)
    in1 = np.ascontiguousarray(in1, dtype=np.int64)
    out = np.empty((in0.shape[0],), np.uint8)
    L = ctypes.c_long
    lib().ctdo_crosscheck(_p(in0), _p(in1), _p(out), L(in0.shape[0]), L(in1.shape[0]))
    return out


def lcn(x, radius, epsilon):
    """model/networks.py:507-533.  x [N,1,H,W] -> (lcn, std), both [N,1,H,W]."""
    (x, sfx) = _real(x)
    N, C, H, W = x.shape
    assert C == 1, "LCN is single-channel (networks.py:514)"
    o = np.empty_like(x)
    s = np.empty_like(x)
    L = ctypes.c_long
    e = ctypes.c_float(epsilon) if x.dtype == np.float32 else ctypes.c_double(epsilon)
    getattr(lib(), "ctdo_lcn" + sfx)(_p(x), _p(o), _p(s), L(N), L(H), L(W), L(radius), e)
    return o, s


def lcn_cython(img, kernel_size=4, epsilon=0.01):
    """data/lcn/lcn.pyx:16-58 normalize(img [M,N] float32, kernel_size, epsilon) -> (lcn, std)."""
    img = np.ascontiguousarray(img, dtype=np.float32)
    M, N = img.shape
    o, s = np.empty_like(img), np.empty_like(img)
    L = ctypes.c_long
    lib().ctdo_lcn_cython_f32(_p(img), _p(o), _p(s), L(M), L(N), L(kernel_size), ctypes.c_float(epsilon))
    return o, s
