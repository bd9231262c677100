"""ctypes binding of ``oracle/_ref/libbev_pool_ref.so`` -- the reference's OWN
``bev_pool_cuda.cu`` compiled for sm_100a by ``oracle/Makefile`` (GPU box only).

TEST INFRASTRUCTURE ONLY -- see ``oracle/__init__.py``.  Used by
``tests/golden/gen_golden_ref_kernel.py`` to record the outputs the ``-m gpu``
parity tests compare the CUDA path with (the unmodified reference kernels on
identical inputs) and by ``bench.py`` for the "reference CUDA kernel on this
B200" line.
The reference launches on the legacy default stream
(bev_pool_cuda.cu:124, 133); callers synchronise around it.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_ref", "libbev_pool_ref.so")
_lib = None


def available():
    return os.path.exists(LIB_PATH)


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(LIB_PATH)
        _lib.ref_bev_pool_v2.restype = ctypes.c_int
        _lib.ref_bev_pool_v2.argtypes = [ctypes.c_int, ctypes.c_int] + \
            [ctypes.c_void_p] * 8
        _lib.ref_bev_pool_v2_grad.restype = ctypes.c_int
        _lib.ref_bev_pool_v2_grad.argtypes = [ctypes.c_int, ctypes.c_int] + \
            [ctypes.c_void_p] * 10
    return _lib


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


def bev_pool_v2_kernel(depth, feat, ranks_depth, ranks_feat, ranks_bev,
                       interval_starts, interval_lengths, out):
    """bev_pool_v2_forward (bev_pool.cpp:28-55): kernel only, `out` is the
    caller-zeroed (B,Z,Y,X,C) volume."""
    rc = lib().ref_bev_pool_v2(
        feat.shape[-1], interval_lengths.shape[0], _p(depth), _p(feat),
        _p(ranks_depth), _p(ranks_feat), _p(ranks_bev), _p(interval_starts),
        _p(interval_lengths), _p(out))
    if rc:
        raise RuntimeError(f"reference kernel launch failed: cuda error {rc}")
    return out


def bev_pool_v2(depth, feat, ranks_depth, ranks_feat, ranks_bev,
                bev_feat_shape, interval_starts, interval_lengths):
    """The reference op as shipped (bev_pool.py:15-39, 84-90):
    new_zeros + kernel + permute(0,4,1,2,3).contiguous()."""
    # the reference kernel runs on the legacy default stream
    torch.cuda.current_stream().synchronize()
    out = feat.new_zeros(bev_feat_shape)
    torch.cuda.current_stream().synchronize()
    bev_pool_v2_kernel(depth, feat, ranks_depth, ranks_feat, ranks_bev,
                       interval_starts, interval_lengths, out)
    torch.cuda.synchronize()
    return out.permute(0, 4, 1, 2, 3).contiguous()


def bev_pool_v2_grad(out_grad, depth, feat, ranks_depth, ranks_feat, ranks_bev,
                     interval_starts_bp, interval_lengths_bp):
    """bev_pool_v2_backward (bev_pool.cpp:72-102)."""
    depth_grad = depth.new_zeros(depth.shape)
    feat_grad = feat.new_zeros(feat.shape)
    torch.cuda.synchronize()
    rc = lib().ref_bev_pool_v2_grad(
        feat.shape[-1], interval_lengths_bp.shape[0], _p(out_grad), _p(depth),
        _p(feat), _p(ranks_depth), _p(ranks_feat), _p(ranks_bev),
        _p(interval_starts_bp), _p(interval_lengths_bp), _p(depth_grad),
        _p(feat_grad))
    if rc:
        raise RuntimeError(f"reference kernel launch failed: cuda error {rc}")
    torch.cuda.synchronize()
    return depth_grad, feat_grad
