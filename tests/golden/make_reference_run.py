#!/usr/bin/env python
"""Run the reference's OWN Python source (unmodified, from /root/reference/src/e2eflow/core) under
the TensorFlow-API stand-in of tests/golden/tf_shim.py and store inputs + outputs as golden vectors
in tests/golden/reference_run.npz (seeded input images as their SHA-256, the full-resolution output
flows as a fixed sample: tests/golden_data.py).

    python tests/golden/make_reference_run.py          (needs /root/reference; run in the build container)

What this pins: the graph the reference builds -- op order, constants, masks, loss weights, pyramid
bookkeeping, variable scopes / names / shapes, gradient flow (stop_gradient, casts) -- for
``image_warp``, every loss term, ``compute_losses`` (all three occlusion modes), ``flownet`` (C, S,
stacked) and ``unsupervised_loss``.  What it does not pin: the arithmetic inside TensorFlow's own
primitives (SAME padding, legacy bilinear resize, grayscale weights, conv2d_transpose), which the
stand-in restates from the TF documentation, and the custom CUDA ops, which are served by
oracle/oracle_ops.c (pinned by the reference's known-answer tests, tests/golden/reference_kats.json).
tests/test_oracle_vs_reference_run.py compares the oracle with these vectors.
"""
import importlib
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
REF_SRC = os.environ.get("UNFLOW_REFERENCE_SRC", "/root/reference/src")

import golden_data  # noqa: E402
import tf_shim  # noqa: E402
from oracle import flownet as oflownet  # noqa: E402
from oracle import ops as oops  # noqa: E402
from unflow_b200 import synthetic as synth  # noqa: E402


def load_reference():
    """Import the reference's e2eflow.core modules with the stand-ins for tensorflow and for the
    compiled-op loader (e2eflow/ops.py JIT-compiles CUDA at import)."""
    tf = tf_shim.install()
    sys.path.insert(0, REF_SRC)
    pkg = importlib.import_module('e2eflow')
    assert os.path.realpath(os.path.dirname(pkg.__file__)).startswith(os.path.realpath(REF_SRC)), pkg.__file__
    ops = types.ModuleType('e2eflow.ops')
    wrap = lambda t: t.as_subclass(tf_shim.Tensor)
    ops.correlation = lambda first, second, **kw: wrap(oops.correlation(first.contiguous(), second.contiguous(), **kw))
    ops.backward_warp = lambda images, flows: wrap(oops.backward_warp(images, flows))
    ops.forward_warp = lambda flows: wrap(oops.forward_warp(flows))
    ops.downsample = lambda images, scale: wrap(oops.downsample(images, scale))
    sys.modules['e2eflow.ops'] = ops
    pkg.ops = ops
    mods = {n: importlib.import_module('e2eflow.core.' + n)
            for n in ('image_warp', 'losses', 'flownet', 'unsupervised', 'augment', 'spatial_transformer',
                      'flow_util', 'input')}
    mods['kitti_input'] = importlib.import_module('e2eflow.kitti.input')
    mods['util'] = importlib.import_module('e2eflow.util')
    for m in mods.values():
        assert os.path.realpath(m.__file__).startswith(os.path.realpath(REF_SRC)), m.__file__
    return tf, mods


def T(x, grad=False):
    t = torch.as_tensor(np.asarray(x), dtype=torch.float32).clone().requires_grad_(grad)
    return t.as_subclass(tf_shim.Tensor)


def N(t):
    return t.detach().cpu().numpy().astype(np.float32) if isinstance(t, torch.Tensor) else np.float32(t)


def checksum(variables):
    s = sum(float(v.double().sum()) for v in variables.values())
    a = sum(float(v.double().abs().sum()) for v in variables.values())
    return np.array([s, a], dtype=np.float64)


def main():
    tf, ref = load_reference()
    out = {}

    # ---- image_warp, individual loss terms, masks ---------------------------------------------
    im1, im2, ffw, fbw = synth.level_inputs(2, 20, 28, seed=5)
    out['L_im1'], out['L_im2'], out['L_ffw'], out['L_fbw'] = map(N, (im1, im2, ffw, fbw))
    tf_shim.STATE.reset({})
    a, f = T(im1, True), T(ffw, True)
    w = ref['image_warp'].image_warp(a, f)
    gsel = torch.linspace(-1, 1, w.numel()).reshape(w.shape)
    ga, gf = torch.autograd.grad((w * gsel).sum(), (a, f))
    out['warp_out'], out['warp_dim'], out['warp_dflow'] = N(w), N(ga), N(gf)
    L = ref['losses']
    out['border_mask'] = N(L.create_border_mask(T(im1), 0.1))
    out['outgoing_mask'] = N(L.create_outgoing_mask(T(ffw * 4)))
    occ = L.occlusion(T(ffw), T(fbw))
    out['occ_fw'], out['occ_bw'] = N(occ[0]), N(occ[1])
    mask = L.create_border_mask(T(im1), 0.1)
    for d in (1, 2, 3):
        out['ternary_d%d' % d] = N(L.ternary_loss(T(im1), T(im2), mask, max_distance=d))
    out['photometric'] = N(L.photometric_loss(T(im1) - T(im2), mask))
    out['gradient_loss'] = N(L.gradient_loss(T(im1), T(im2), mask))
    out['smoothness_1st'] = N(L.smoothness_loss(T(ffw)))
    out['smoothness_2nd'] = N(L.second_order_loss(T(ffw)))
    out['charbonnier_trunc'] = N(L.charbonnier_loss(T(ffw), mask, truncate=0.7, alpha=0.3, beta=2.0))

    # ---- compute_losses: every term, three occlusion modes, with / without border mask ----------
    weights = dict(ternary=1.0, smooth_2nd=3.0, fb=0.2, occ=12.4, photo=0.5, grad=0.25, smooth_1st=0.75, sym=0.3)
    for tag, mode, use_border, dist in (('fb', 'fb', True, 3), ('none', '', False, 1), ('disocc', 'disocc', True, 2)):
        fw, bw = T(ffw, True), T(fbw, True)
        border = L.create_border_mask(T(im1), 0.1) if use_border else None
        res = L.compute_losses(T(im1), T(im2), fw, bw, border_mask=border, mask_occlusion=mode,
                               data_max_distance=dist)
        assert sorted(res) == sorted(weights), sorted(res)
        total = 0.0
        for k in sorted(res):
            out['cl_%s_%s' % (tag, k)] = N(res[k])
            total = total + weights[k] * res[k]
        gfw, gbw = torch.autograd.grad(total, (fw, bw))
        out['cl_%s_dfw' % tag], out['cl_%s_dbw' % tag] = N(gfw), N(gbw)

    # ---- flownet: C, S and a stacked net, both directions -----------------------------------------
    for tag, spec, hw, seed in (('c', 'c', (64, 128), 21), ('s', 's', (64, 64), 22), ('cs', 'cs', (64, 64), 23)):
        variables = oflownet.init_variables(spec, False, seed=seed)
        tf_shim.STATE.reset({k: v for k, v in variables.items()})
        i1, i2, _ = synth.image_pair(1, hw[0], hw[1], seed=seed + 100)
        i1, i2 = i1 / 255.0 - 0.4, i2 / 255.0 - 0.4
        fw, bw = ref['flownet'].flownet(T(i1), T(i2), flownet_spec=spec, backward_flow=True)
        assert sorted(tf_shim.STATE.created) == sorted(variables), "variable names differ from the reference graph"
        out['fn_%s_im1' % tag], out['fn_%s_im2' % tag] = N(i1), N(i2)
        out['fn_%s_vars' % tag] = checksum(variables)
        for n, (nf, nb) in enumerate(zip(fw, bw)):
            for lvl, (a_, b_) in enumerate(zip(nf, nb)):
                out['fn_%s_net%d_fw%d' % (tag, n, lvl)] = N(a_)
                out['fn_%s_net%d_bw%d' % (tag, n, lvl)] = N(b_)

    # full-resolution variant (two more up-convolutions under the scope 'full_res')
    variables = oflownet.init_variables('s', True, seed=24)
    tf_shim.STATE.reset(dict(variables))
    i1, i2, _ = synth.image_pair(1, 64, 64, seed=124)
    i1, i2 = i1 / 255.0 - 0.4, i2 / 255.0 - 0.4
    fw, bw = ref['flownet'].flownet(T(i1), T(i2), flownet_spec='s', full_resolution=True, backward_flow=True)
    assert sorted(tf_shim.STATE.created) == sorted(variables) and len(fw[0]) == 7
    out['fn_sfull_im1'], out['fn_sfull_im2'], out['fn_sfull_vars'] = N(i1), N(i2), checksum(variables)
    for lvl in range(7):
        out['fn_sfull_fw%d' % lvl], out['fn_sfull_bw%d' % lvl] = N(fw[0][lvl]), N(bw[0][lvl])

    # ---- unsupervised_loss: value, output flows, gradient norms ---------------------------------
    for tag, spec, hw, seed, extra in (('c', 'c', (128, 128), 31, {}), ('s', 's', (128, 128), 32, {'pyramid_loss': False}),
                                       ('cs', 'cs', (128, 128), 33, {'train_all': True})):
        params = dict(synth.KITTI_PARAMS, flownet=spec, **extra)
        variables = oflownet.init_variables(spec, False, seed=seed)
        leaves = {k: v.clone().requires_grad_(True) for k, v in variables.items()}
        tf_shim.STATE.reset(leaves)
        i1, i2, _ = synth.image_pair(1, hw[0], hw[1], seed=seed + 100)
        loss, ffw_, fbw_ = ref['unsupervised'].unsupervised_loss((T(i1), T(i2)), params, synth.KITTI_NORMALIZATION,
                                                                 augment=False, return_flow=True)
        names = sorted(leaves)
        grads = torch.autograd.grad(loss, [leaves[k] for k in names], allow_unused=True)
        out['ul_%s_im1' % tag], out['ul_%s_im2' % tag] = N(i1), N(i2)
        out['ul_%s_vars' % tag] = checksum(variables)
        out['ul_%s_loss' % tag] = N(loss)
        out['ul_%s_flow_fw' % tag], out['ul_%s_flow_bw' % tag] = N(ffw_), N(fbw_)
        out['ul_%s_grad_names' % tag] = np.array(names)
        out['ul_%s_grad_norms' % tag] = np.array([0.0 if g is None else float(g.double().norm()) for g in grads])
        for k, g in zip(names, grads):          # the small gradients in full
            if g is not None and g.numel() <= 4096:
                out['ul_%s_grad/%s' % (tag, k)] = N(g)

    # ---- augmentation (SURVEY.md 8f N4): the random draws are recorded and stored as inputs -------
    a1, a2, _ = synth.image_pair(3, 24, 36, seed=41)
    a1, a2 = a1 / 255.0, a2 / 255.0
    amask = ref['losses'].create_border_mask(T(a1), 0.1)
    out['aug_im1'], out['aug_im2'], out['aug_mask'] = N(a1), N(a2), N(amask)
    theta = torch.tensor([[1.05, 0.1, 0.02, -0.08, 0.93, -0.03], [0.9, 0.0, 0.0, 0.0, 1.1, 0.0],
                          [-1.0, 0.2, 0.1, 0.15, 1.0, 0.05]])
    out['aug_theta'] = N(theta)
    out['aug_transformer'] = N(ref['spatial_transformer'].transformer(T(a1), T(theta), (20, 30)))
    tf_shim.STATE.reset({})
    tf_shim.STATE.rng.manual_seed(1)
    res = ref['augment'].random_affine([T(a1), T(a2), amask], horizontal_flipping=True, min_scale=0.9, max_scale=1.1,
                                       max_translation_x=0.1, max_translation_y=0.05, max_rotation=10.0)
    for name, d in zip(('tx', 'ty', 'rot', 'scale', 'flip'), tf_shim.STATE.draws):
        out['aug_affine_' + name] = N(d)
    assert len(tf_shim.STATE.draws) == 5
    for i, r in enumerate(res):
        out['aug_affine_out%d' % i] = N(r)
    tf_shim.STATE.reset({})
    tf_shim.STATE.rng.manual_seed(8)
    res = ref['augment'].random_photometric([T(a1), T(a2)], noise_stddev=0.04, min_contrast=-0.3, max_contrast=0.3,
                                            brightness_stddev=0.02, min_colour=0.9, max_colour=1.1,
                                            min_gamma=0.7, max_gamma=1.5)
    for name, d in zip(('contrast', 'gamma', 'colour', 'noise', 'brightness'), tf_shim.STATE.draws):
        out['aug_photo_' + name] = N(d)
    assert len(tf_shim.STATE.draws) == 5
    out['aug_photo_out0'], out['aug_photo_out1'] = N(res[0]), N(res[1])

    # ---- evaluation utilities (SURVEY.md 8f N3): flow_util.py, the resize helpers of input.py -----
    FU, IN = ref['flow_util'], ref['input']
    g = torch.Generator().manual_seed(51)
    fl = torch.randn(2, 12, 16, 2, generator=g) * 6
    fl[0, 0, 0] = 0.0                                   # atan2(0, 0) -> NaN hue in the reference
    fl[0, 0, 1] = torch.tensor([0.0, 2.0])
    fl[0, 0, 2] = torch.tensor([0.0, -2.0])
    fl[0, 0, 3] = torch.tensor([-3.0, 0.0])
    gt = fl + torch.randn(2, 12, 16, 2, generator=g) * 2
    mocc = (torch.rand(2, 12, 16, 1, generator=g) > 0.2).float()
    mnoc = mocc * (torch.rand(2, 12, 16, 1, generator=g) > 0.3).float()
    out['fu_flow'], out['fu_gt'], out['fu_mocc'], out['fu_mnoc'] = N(fl), N(gt), N(mocc), N(mnoc)
    out['fu_color'] = N(FU.flow_to_color(T(fl)))
    out['fu_color_mask_max'] = N(FU.flow_to_color(T(fl), T(mocc), max_flow=10.0))
    out['fu_error_log'] = N(FU.flow_error_image(T(fl), T(gt), T(mocc), T(mnoc)))
    out['fu_error_lin'] = N(FU.flow_error_image(T(fl), T(gt), T(mocc), T(mnoc), log_colors=False))
    out['fu_error_log_nonoc'] = N(FU.flow_error_image(T(fl), T(gt), T(mocc)))
    out['fu_aee'] = N(FU.flow_error_avg(T(gt), T(fl), T(mocc)))
    out['fu_outlier_pct'] = N(FU.outlier_pct(T(gt), T(fl), T(mocc)))
    out['fu_outlier_ratio_abs'] = N(FU.outlier_ratio(T(gt), T(fl), T(mnoc), threshold=2.0, relative=None))
    img = torch.rand(1, 14, 20, 3, generator=g) * 255
    out['in_img'] = N(img)
    out['in_resize_input'] = N(IN.resize_input(T(img.reshape(-1)), 10, 16, 14, 20))
    out['in_resize_output_crop'] = N(IN.resize_output_crop(T(img), 10, 24, 3))
    out['in_resize_output'] = N(IN.resize_output(T(img), 7, 30, 3))
    out['in_resize_output_flow'] = N(IN.resize_output_flow(T(fl[:1]), 18, 8, 2))
    out['in_frame_nums'] = np.array([IN.frame_name_to_num(n) for n in ('0000000000.png', '0000000120.png', '7.png')])

    # ---- input pipeline (SURVEY.md 8f N4): which files are paired, in which order ------------------
    import json
    import tempfile
    listing = {}
    with tempfile.TemporaryDirectory() as root:
        tree = {'raw/a/image_02/data': [0, 1, 2, 3, 5, 6], 'raw/a/image_03/data': [0, 1, 2],
                'raw/b/image_02/data': [10, 11, 12, 14], 'raw/b/image_03/data': [7, 8]}
        for d, nums in tree.items():
            os.makedirs(os.path.join(root, d))
            for n in nums:
                open(os.path.join(root, d, '%010d.png' % n), 'w').close()
        for sub, names in (('data_stereo_flow/training/colored_0', ['%06d_%d.png' % (i, j) for i in range(5) for j in (10, 11)]),
                           ('data_stereo_flow/training/flow_occ', ['%06d_10.png' % i for i in range(5)]),
                           ('data_stereo_flow/training/flow_noc', ['%06d_10.png' % i for i in range(5)])):
            os.makedirs(os.path.join(root, sub))
            for n in names:
                open(os.path.join(root, sub, n), 'w').close()

        class Data:
            current_dir = root

            def get_raw_dirs(self):
                return [os.path.join(root, d) for d in sorted(tree)]

        rel = lambda files: [os.path.relpath(f, root) for f in files]
        KI = ref['kitti_input'].KITTIInput
        cases = {'plain': dict(kw={}, call=dict(swap_images=False)),
                 'skipped_swap_shift3': dict(kw=dict(skipped_frames=True), call=dict(swap_images=True, shift=3)),
                 'skipped_shift4_seed5': dict(kw=dict(skipped_frames=True), call=dict(swap_images=False, shift=4, seed=5)),
                 'skip01': dict(kw={}, call=dict(swap_images=False, skip=[0, 1]))}
        for tag, c in cases.items():
            tf_shim.STATE.reset({})
            tf_shim.STATE.decode_shape = (4, 6, 3)
            inp = KI(Data(), batch_size=2, dims=(4, 6), normalize=False, **c['kw'])
            inp.input_raw(needs_crop=False, **c['call'])
            first, second = tf_shim.STATE.queues[:2]
            listing['raw_' + tag] = [rel(first), rel(second)]
        for tag, hold in (('all', None), ('hold3', 3)):
            tf_shim.STATE.reset({})
            inp = KI(Data(), batch_size=1, dims=(4, 6), normalize=False)
            inp.input_train_2012(hold)
            q = tf_shim.STATE.queues
            listing['train2012_' + tag] = [rel(x) for x in q[:4]]      # frame 1, frame 2, flow_occ, flow_noc
    out['input_listing_json'] = np.array(json.dumps(listing))
    ini = ("[dirs]\nlog = ../log\ndata = /data\n[run]\nbatch_size = 4\ngpu_list = 0,1\ndevelopment = False\n"
           "dataset = kitti\n[train]\nlearning_rate = 1.0e-4\ndecay_interval = 100000\nflownet = CSS\n"
           "pyramid_loss = True\nmask_occlusion = fb\nternary_weight = 1.0\nnum_iters = 500000\n"
           "[train_kitti_ft]\nmanual_decay_iters = 45000,20000\nmanual_decay_lrs = 0.5e-5,0.25e-5\nheight = 320\n")
    with tempfile.TemporaryDirectory() as d:
        path_ini = os.path.join(d, 'config.ini')
        open(path_ini, 'w').write(ini)
        cfg = ref['util'].config_dict(path_ini)
        ft = dict(cfg['train'])
        ft.update(cfg['train_kitti_ft'])
        ref['util'].convert_input_strings(ft, cfg['dirs'])
    out['config_ini'] = np.array(ini)
    out['config_json'] = np.array(json.dumps({'config': cfg, 'kitti_ft': ft}, sort_keys=True))

    # ---- learning-rate schedule: the reference computes it inline in Trainer.train (train.py:224-244);
    # those source lines are cut out and executed as they are -----------------------------------
    import textwrap
    src = open(os.path.join(REF_SRC, 'e2eflow', 'core', 'train.py')).read().split('\n')
    first = next(i for i, l in enumerate(src) if 'decay_iters = local_i + iter_offset' in l)
    last = next(i for i in range(first, len(src)) if 'feed_dict = {learning_rate_' in src[i])
    block = textwrap.dedent('\n'.join(src[first + 1:last]))
    assert "learning_rate = self.params['learning_rate'] / (2 ** decay)" in block

    def reference_lr(params, decay_iters):
        scope = {'self': types.SimpleNamespace(params=params), 'decay_iters': decay_iters}
        exec(block, scope)
        return scope['learning_rate']

    schedules = {'halving': dict(learning_rate=1.0e-4, decay_interval=100000, decay_after=300000),
                 'halving_from_start': dict(learning_rate=2.0e-4, decay_interval=50000),
                 'manual': dict(learning_rate=1.0e-4, decay_interval=100000, manual_decay_iters=[45000, 20000, 5000],
                                manual_decay_lrs=[0.5e-5, 0.25e-5, 0.1e-5])}
    probes = [0, 1, 44999, 45000, 45001, 49999, 50000, 65000, 65001, 70000, 99999, 100000, 299999, 300000, 300001,
              399999, 400000, 500000, 750000]
    out['lr_probes'] = np.array(probes)
    out['lr_schedules_json'] = np.array(json.dumps(schedules))
    for name, prm in schedules.items():
        out['lr_' + name] = np.array([reference_lr(prm, it) for it in probes], dtype=np.float64)

    # ---- restore_networks (train.py:23-37): which finetune sources are loaded -----------------------
    first = next(i for i, l in enumerate(src) if l.startswith('def restore_networks('))
    last = next(i for i in range(first, len(src)) if 'saver = tf.train.Saver(variables_to_save' in src[i])
    block = textwrap.dedent('\n'.join(src[first + 1:last]))
    plans = {}
    for spec in ('C', 'CS', 'CSS'):
        for train_all in (None, True):
            for n_ft in range(0, len(spec) + 1):
                for has_ckpt in (False, True):
                    scope = {'params': {'flownet': spec, 'train_all': train_all, 'finetune': ['ex%d' % i for i in range(n_ft)]},
                             'ckpt': object() if has_ckpt else None,
                             'slim': types.SimpleNamespace(get_variables_to_restore=lambda include=None: include)}
                    exec(block, scope)
                    plans['%s|%s|%d|%d' % (spec, bool(train_all), n_ft, int(has_ckpt))] = {
                        'external': scope['restore_external_nets'], 'net_names': scope['net_names']}
    out['restore_plans_json'] = np.array(json.dumps(plans))

    out = golden_data.shrink_reference_run(out)
    path = os.path.join(HERE, 'reference_run.npz')
    np.savez_compressed(path, **out)
    print("wrote %s: %d arrays, %.1f KB" % (path, len(out), os.path.getsize(path) / 1024.0))


if __name__ == '__main__':
    main()
