"""The reference's own CUDA kernels as ground truth for the four custom ops.  Their outputs on the
inputs below are stored in tests/golden/reference_kernels.npz (made on a B200 by
tests/golden/make_reference_kernels.py from oracle/_ref/libref_ops.so, the reference kernels compiled
against stand-in TensorFlow headers: oracle/ref_kernels.py).

* CPU part: the correlation geometry of the reference's ``CorrelationState`` host code -- compared
  with the oracle and with the product's C ABI.
* GPU part: the oracle's C restatement and the product's kernels are compared with the reference
  kernels' outputs -- forward and gradients of all four ops, including displacement > 0 / C > 1 /
  K = 3 / strides, which the reference's own KATs never exercise (test/ops/correlation.py:30-89).
  Outputs above golden_data.SAMPLE elements are compared on a fixed sample; the product is also
  held to the oracle on every element."""
import ctypes
import itertools
import os

import numpy as np
import pytest
import torch

import golden_data
from oracle import ops as oops

GEOMETRY = list(itertools.product((48, 37), (160, 64), (1, 3), (20, 4, 0), (20, 4, 0), (1, 2), (1, 2)))
CORRELATION_CASES = [(2, 32, 12, 20, dict(kernel_size=1, max_displacement=4, pad=4, stride_1=1, stride_2=2)),
                     (1, 16, 10, 14, dict(kernel_size=3, max_displacement=3, pad=4, stride_1=2, stride_2=1)),
                     (1, 256, 48, 160, dict(kernel_size=1, max_displacement=20, pad=20, stride_1=1, stride_2=2))]


def load_golden():
    with np.load(os.path.join(golden_data.GOLDEN, "reference_kernels.npz")) as z:
        return {k: z[k] for k in z.files}


def correlation_inputs(B, C, H, W, out_shape):
    g = torch.Generator().manual_seed(C + H)
    a, b = torch.randn(B, C, H, W, generator=g), torch.randn(B, C, H, W, generator=g)
    return a, b, torch.randn(tuple(out_shape), generator=g)


def warp_inputs():
    g = torch.Generator().manual_seed(3)
    im = torch.rand(2, 18, 26, 3, generator=g)
    fl = torch.randn(2, 18, 26, 2, generator=g) * 4
    go_backward = torch.randn(2, 18, 26, 3, generator=g)
    go_forward = torch.randn(2, 18, 26, 1, generator=g)
    x = torch.rand(2, 16, 24, 3, generator=g)
    return dict(im=im, fl=fl, go_backward=go_backward, go_forward=go_forward, x=x)


def checked_inputs(G, prefix, inputs):
    for name, t in inputs.items():
        golden_data.check_digest(prefix + name, t, G[prefix + name + '_sha256'])
    return inputs


def _close(a, b, tol=1e-5):
    a, b = a.detach().cpu(), b.detach().cpu()
    scale = max(float(b.abs().max()), 1e-12)
    assert float((a - b).abs().max()) <= tol * scale, float((a - b).abs().max()) / scale


def _close_ref(G, got, key, tol=1e-5):
    """``got`` against the reference kernels' output ``key``: on the stored sample, scaled by the
    largest magnitude of the whole output."""
    assert tuple(got.shape) == tuple(G[key + '_shape']), (key, tuple(got.shape))
    got = torch.from_numpy(golden_data.sample(got))
    want = torch.from_numpy(G[key + '_sample'])
    scale = max(float(G[key + '_absmax']), 1e-12)
    assert float((got - want).abs().max()) <= tol * scale, (key, float((got - want).abs().max()) / scale)


def test_correlation_geometry_from_the_reference_host_code():
    from unflow_b200 import _native
    lib = _native.lib()
    G = load_golden()
    n = 0
    for (H, W, ks, md, pad, s1, s2), want in zip(GEOMETRY, G['geometry']):
        want = tuple(int(v) for v in want)
        oc, oh, ow = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        rc = oops.lib().oracle_correlation_shape(H, W, ks, md, pad, s1, s2, ctypes.byref(oc), ctypes.byref(oh), ctypes.byref(ow))
        c2, h2, w2 = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        rc2 = lib.unflow_correlation_out_shape(H, W, ks, md, pad, s1, s2, ctypes.byref(c2), ctypes.byref(h2),
                                               ctypes.byref(w2))
        shape = (c2.value, h2.value, w2.value)
        if want[1] <= 0 or want[2] <= 0:            # the reference op rejects these (correlation_op.cc:60-61)
            assert rc != 0 and rc2 != 0
            continue
        n += 1
        assert rc == 0 and (oc.value, oh.value, ow.value) == want, (H, W, ks, md, pad, s1, s2)
        assert rc2 == 0 and tuple(shape) == want, (H, W, ks, md, pad, s1, s2)
    assert len(G['geometry']) == len(GEOMETRY) and n > 100


@pytest.mark.gpu
@pytest.mark.parametrize("B,C,H,W,attrs", CORRELATION_CASES)
def test_correlation_kernels(B, C, H, W, attrs):
    from unflow_b200.e2eflow import ops
    G = load_golden()
    p = 'corr%d_' % CORRELATION_CASES.index((B, C, H, W, attrs))
    a, b, go = correlation_inputs(B, C, H, W, G[p + 'out_shape'])
    checked_inputs(G, p, dict(a=a, b=b, go=go))
    want = oops.correlation(a, b, **attrs)
    _close_ref(G, want, p + 'out')
    ao, bo = a.clone().requires_grad_(True), b.clone().requires_grad_(True)
    oops.correlation(ao, bo, **attrs).backward(go)
    _close_ref(G, ao.grad, p + 'g0')
    _close_ref(G, bo.grad, p + 'g1')
    ac, bc = a.cuda().requires_grad_(True), b.cuda().requires_grad_(True)
    out = ops.correlation(ac, bc, **attrs)
    _close_ref(G, out, p + 'out')
    _close(out, want, 2e-5)
    out.backward(go.cuda())
    _close_ref(G, ac.grad, p + 'g0', 2e-5)
    _close_ref(G, bc.grad, p + 'g1', 2e-5)
    _close(ac.grad, ao.grad, 3e-5)
    _close(bc.grad, bo.grad, 3e-5)


@pytest.mark.gpu
def test_warp_and_downsample_kernels():
    from unflow_b200.e2eflow import ops
    G = load_golden()
    i = checked_inputs(G, 'warp_', warp_inputs())
    im, fl = i['im'], i['fl']
    _close_ref(G, oops.backward_warp(im, fl), 'backward_warp')
    _close_ref(G, ops.backward_warp(im.cuda(), fl.cuda()), 'backward_warp')
    go = i['go_backward']
    fo = fl.clone().requires_grad_(True)
    oops.backward_warp(im, fo).backward(go)
    _close_ref(G, fo.grad, 'backward_warp_grad')
    fc = fl.cuda().requires_grad_(True)
    ops.backward_warp(im.cuda(), fc).backward(go.cuda())
    _close_ref(G, fc.grad, 'backward_warp_grad', 2e-5)

    _close_ref(G, oops.forward_warp(fl), 'forward_warp', 1e-4)          # float atomics: order-dependent rounding
    _close_ref(G, ops.forward_warp(fl.cuda()), 'forward_warp', 1e-4)
    go = i['go_forward']
    fo = fl.clone().requires_grad_(True)
    oops.forward_warp(fo).backward(go)
    _close_ref(G, fo.grad, 'forward_warp_grad', 1e-4)
    fc = fl.cuda().requires_grad_(True)
    ops.forward_warp(fc).backward(go.cuda())
    _close_ref(G, fc.grad, 'forward_warp_grad', 1e-4)

    x = i['x']
    for scale in (2, 4):
        _close_ref(G, oops.downsample(x, scale), 'downsample%d' % scale)
        _close_ref(G, ops.downsample(x.cuda(), scale), 'downsample%d' % scale)
