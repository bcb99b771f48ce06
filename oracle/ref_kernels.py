"""The reference's OWN CUDA kernels as a checker (TEST INFRASTRUCTURE ONLY).

``oracle/ref_ops/build.sh`` compiles /root/reference/ops/{correlation,backward_warp,forward_warp,
downsample}_op.cu.cc for sm_100a exactly as they lie in the reference tree -- nothing is copied --
against stand-in headers (oracle/tf_stub) for the handful of TensorFlow declarations those files
include, and links them with a C wrapper (oracle/ref_ops/wrapper.cu) into oracle/_ref/libref_ops.so.
The op-registration files (*_op.cc) need the whole TensorFlow op framework and are not built; by
the letter of the task the reference is therefore "unbuildable", what IS built are its GPU kernels
and their launchers, which is where the arithmetic lives.

Used by tests/golden/make_reference_kernels.py (which stores their outputs for
tests/test_reference_kernels.py) and tools/bench_reference_kernels.py.

All functions take / return float32 CUDA tensors in the reference's layouts (correlation NCHW, the
warps and downsample NHWC) and synchronise before returning; the kernels run on the legacy default
stream like in the reference (its correlation launches ignore the TF stream).
"""
import ctypes
import os
import subprocess

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_ref", "libref_ops.so")
_lib = None


def build():
    """(Re)build when the reference tree is present and fail loudly if that leaves no library; where
    the tree is absent, a library built on another machine must have been copied to LIB_PATH."""
    subprocess.check_call(["bash", os.path.join(HERE, "ref_ops", "build.sh")])
    if not available():
        raise RuntimeError("%s is missing: oracle/ref_ops/build.sh builds it from the reference tree "
                           "(UNFLOW_REFERENCE)" % LIB_PATH)


def available():
    return os.path.exists(LIB_PATH)


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(LIB_PATH)
    return _lib


def correlation_out_shape(C, H, W, kernel_size=1, max_displacement=20, pad=20, stride_1=1, stride_2=2):
    """(channels, height, width) from the reference's CorrelationState (host code, runs anywhere)."""
    out = (ctypes.c_int * 3)()
    lib().ref_correlation_out_shape(C, H, W, kernel_size, max_displacement, pad, stride_1, stride_2, out)
    return tuple(out)


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


def _check(rc, what):
    torch.cuda.synchronize()
    if rc != 0:
        raise RuntimeError("reference kernel %s: CUDA error" % what)


def correlation(in0, in1, kernel_size=1, max_displacement=20, pad=20, stride_1=1, stride_2=2):
    """-> (volume [B,D*D,oh,ow], padded_0, padded_1) like the reference op's three outputs."""
    B, C, H, W = in0.shape
    oc, oh, ow = correlation_out_shape(C, H, W, kernel_size, max_displacement, pad, stride_1, stride_2)
    in0, in1 = in0.contiguous(), in1.contiguous()
    out = torch.empty(B, oc, oh, ow, device=in0.device)
    p0 = torch.empty(B, H + 2 * pad, W + 2 * pad, C, device=in0.device)
    p1 = torch.empty_like(p0)
    torch.cuda.synchronize()
    _check(lib().ref_correlation_fwd(_p(in0), _p(in1), _p(out), _p(p0), _p(p1), B, C, H, W, kernel_size,
                                     max_displacement, pad, stride_1, stride_2), "Correlation")
    return out, p0, p1


def correlation_grad(gout, padded0, padded1, shape, kernel_size=1, max_displacement=20, pad=20, stride_1=1, stride_2=2):
    B, C, H, W = shape
    g0 = torch.zeros(B, C, H, W, device=gout.device)
    g1 = torch.zeros(B, C, H, W, device=gout.device)
    torch.cuda.synchronize()
    _check(lib().ref_correlation_bwd(_p(gout.contiguous()), _p(padded0), _p(padded1), _p(g0), _p(g1), B, C, H, W,
                                     kernel_size, max_displacement, pad, stride_1, stride_2), "CorrelationGrad")
    return g0, g1


def backward_warp(images, flows):
    B, H, W, C = images.shape
    out = torch.empty_like(images)
    torch.cuda.synchronize()
    _check(lib().ref_backward_warp_fwd(_p(images.contiguous()), _p(flows.contiguous()), _p(out), B, H, W, C), "BackwardWarp")
    return out


def backward_warp_grad(grad, images, flows):
    B, H, W, C = images.shape
    dflow = torch.empty(B, H, W, 2, device=images.device)
    torch.cuda.synchronize()
    _check(lib().ref_backward_warp_bwd(_p(grad.contiguous()), _p(images.contiguous()), _p(flows.contiguous()), _p(dflow),
                                       B, H, W, C), "BackwardWarpGrad")
    return dflow


def forward_warp(flows):
    B, H, W, _ = flows.shape
    out = torch.empty(B, H, W, 1, device=flows.device)
    torch.cuda.synchronize()
    _check(lib().ref_forward_warp_fwd(_p(flows.contiguous()), _p(out), B, H, W), "ForwardWarp")
    return out


def forward_warp_grad(grad, flows):
    B, H, W, _ = flows.shape
    dflow = torch.empty(B, H, W, 2, device=flows.device)
    torch.cuda.synchronize()
    _check(lib().ref_forward_warp_bwd(_p(grad.contiguous()), _p(flows.contiguous()), _p(dflow), B, H, W), "ForwardWarpGrad")
    return dflow


def downsample(images, scale):
    B, H, W, C = images.shape
    out = torch.empty(B, H // scale, W // scale, C, device=images.device)
    torch.cuda.synchronize()
    _check(lib().ref_downsample(_p(images.contiguous()), _p(out), B, H, W, C, scale), "Downsample")
    return out
