#!/usr/bin/env python
"""Run the reference's own CUDA kernels (oracle/_ref/libref_ops.so, see oracle/ref_kernels.py) on the
inputs of tests/test_reference_kernels.py and store what they return in
tests/golden/reference_kernels.npz: the correlation geometry of its host code, and for every kernel
output its shape, largest magnitude and a fixed sample (tests/golden_data.py).  The inputs are stored
as their SHA-256 only; the test draws them again from the same seeds.

    bash oracle/ref_ops/build.sh                      (needs the reference tree)
    python tests/golden/make_reference_kernels.py [OUT.npz]     (needs a GPU)

Before writing, the oracle (oracle/oracle_ops.c) is held to the reference kernels on every element,
with the tolerances of the test."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import golden_data  # noqa: E402
import test_reference_kernels as T  # noqa: E402
from oracle import ops as oops  # noqa: E402
from oracle import ref_kernels as RK  # noqa: E402


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "reference_kernels.npz")
    RK.build()
    out = {'geometry': np.array([RK.correlation_out_shape(256, *g) for g in T.GEOMETRY], dtype=np.int32)}

    def store(key, ref, oracle, tol=1e-5):
        T._close(oracle, ref, tol)
        ref = ref.detach().cpu()
        out[key + '_shape'] = np.array(ref.shape)
        out[key + '_absmax'] = np.float32(ref.abs().max())
        out[key + '_sample'] = golden_data.sample(ref)

    def inputs(prefix, named):
        for name, t in named.items():
            out[prefix + name + '_sha256'] = np.array(golden_data.digest(t))

    for i, (B, C, H, W, attrs) in enumerate(T.CORRELATION_CASES):
        p = 'corr%d_' % i
        shape = (B,) + RK.correlation_out_shape(C, H, W, **attrs)
        a, b, go = T.correlation_inputs(B, C, H, W, shape)
        inputs(p, dict(a=a, b=b, go=go))
        out[p + 'out_shape'] = np.array(shape)
        ref, p0, p1 = RK.correlation(a.cuda(), b.cuda(), **attrs)
        store(p + 'out', ref, oops.correlation(a, b, **attrs))
        r0, r1 = RK.correlation_grad(go.cuda(), p0, p1, (B, C, H, W), **attrs)
        ao, bo = a.clone().requires_grad_(True), b.clone().requires_grad_(True)
        oops.correlation(ao, bo, **attrs).backward(go)
        store(p + 'g0', r0, ao.grad)
        store(p + 'g1', r1, bo.grad)

    i = T.warp_inputs()
    inputs('warp_', i)
    im, fl = i['im'], i['fl']
    store('backward_warp', RK.backward_warp(im.cuda(), fl.cuda()), oops.backward_warp(im, fl))
    fo = fl.clone().requires_grad_(True)
    oops.backward_warp(im, fo).backward(i['go_backward'])
    store('backward_warp_grad', RK.backward_warp_grad(i['go_backward'].cuda(), im.cuda(), fl.cuda()), fo.grad)
    store('forward_warp', RK.forward_warp(fl.cuda()), oops.forward_warp(fl), 1e-4)
    fo = fl.clone().requires_grad_(True)
    oops.forward_warp(fo).backward(i['go_forward'])
    store('forward_warp_grad', RK.forward_warp_grad(i['go_forward'].cuda(), fl.cuda()), fo.grad, 1e-4)
    for scale in (2, 4):
        store('downsample%d' % scale, RK.downsample(i['x'].cuda(), scale), oops.downsample(i['x'], scale))

    np.savez_compressed(path, **out)
    print("wrote %s: %d arrays, %.1f KB (%s)" % (path, len(out), os.path.getsize(path) / 1024.0,
                                               torch.cuda.get_device_name(0)))


if __name__ == "__main__":
    main()
