"""The oracle against golden vectors produced by the reference's OWN Python source
(/root/reference/src/e2eflow/core/*.py, unmodified) executed under the TensorFlow-API stand-in of
tests/golden/tf_shim.py -- see tests/golden/make_reference_run.py for what that does and does not
pin.  Runs without /root/reference: only the committed fixture is read."""
import os

import numpy as np
import pytest
import torch

from oracle import flownet as oflownet
from oracle import image_warp as oimage_warp
from oracle import losses as olosses
from oracle import unsupervised as ounsup
import golden_data
import synth

G = golden_data.load_reference_run()
WEIGHTS = dict(ternary=1.0, smooth_2nd=3.0, fb=0.2, occ=12.4, photo=0.5, grad=0.25, smooth_1st=0.75, sym=0.3)


def t(name, grad=False):
    return torch.from_numpy(G[name]).clone().requires_grad_(grad)


def close(got, want, rtol=2e-5, atol_rel=2e-6, msg=""):
    got = got.detach().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    want = np.asarray(want)
    atol = atol_rel * max(float(np.abs(want).max()), 1e-12)
    np.testing.assert_allclose(got, want, rtol=rtol, atol=atol, err_msg=msg)


def test_image_warp_values_and_gradients():
    im, flow = t('L_im1', True), t('L_ffw', True)
    w = oimage_warp.image_warp(im, flow)
    close(w, G['warp_out'])
    gsel = torch.linspace(-1, 1, w.numel()).reshape(w.shape)
    gi, gf = torch.autograd.grad((w * gsel).sum(), (im, flow))
    close(gi, G['warp_dim'])
    close(gf, G['warp_dflow'], rtol=1e-4, atol_rel=1e-5)


def test_masks_and_single_terms():
    im1, im2, ffw, fbw = t('L_im1'), t('L_im2'), t('L_ffw'), t('L_fbw')
    mask = olosses.create_border_mask(im1, 0.1)
    assert np.array_equal(mask.numpy(), G['border_mask'])
    assert np.array_equal(olosses.create_outgoing_mask(ffw * 4).numpy(), G['outgoing_mask'])
    occ = olosses.occlusion(ffw, fbw)
    assert np.array_equal(occ[0].numpy(), G['occ_fw']) and np.array_equal(occ[1].numpy(), G['occ_bw'])
    assert 0 < G['occ_fw'].mean() < 1 and 0 < G['outgoing_mask'].mean() < 1          # non-trivial masks
    for d in (1, 2, 3):
        close(olosses.ternary_loss(im1, im2, mask, max_distance=d), G['ternary_d%d' % d], msg="ternary %d" % d)
    close(olosses.photometric_loss(im1 - im2, mask), G['photometric'])
    close(olosses.gradient_loss(im1, im2, mask), G['gradient_loss'])
    close(olosses.smoothness_loss(ffw), G['smoothness_1st'])
    close(olosses.second_order_loss(ffw), G['smoothness_2nd'])
    close(olosses.charbonnier_loss(ffw, mask, truncate=0.7, alpha=0.3, beta=2.0), G['charbonnier_trunc'])


@pytest.mark.parametrize("tag,mode,use_border,dist", [('fb', 'fb', True, 3), ('none', '', False, 1), ('disocc', 'disocc', True, 2)])
def test_compute_losses_all_terms_and_flow_gradients(tag, mode, use_border, dist):
    im1, im2 = t('L_im1'), t('L_im2')
    fw, bw = t('L_ffw', True), t('L_fbw', True)
    border = olosses.create_border_mask(im1, 0.1) if use_border else None
    res = olosses.compute_losses(im1, im2, fw, bw, border_mask=border, mask_occlusion=mode, data_max_distance=dist)
    total = 0.0
    for k in sorted(WEIGHTS):
        close(res[k], G['cl_%s_%s' % (tag, k)], msg=k)
        total = total + WEIGHTS[k] * res[k]
    gfw, gbw = torch.autograd.grad(total, (fw, bw))
    close(gfw, G['cl_%s_dfw' % tag], rtol=2e-4, atol_rel=2e-5, msg="dflow_fw")
    close(gbw, G['cl_%s_dbw' % tag], rtol=2e-4, atol_rel=2e-5, msg="dflow_bw")


def _variables(spec, seed, key):
    v = oflownet.init_variables(spec, False, seed=seed)
    s = sum(float(x.double().sum()) for x in v.values())
    a = sum(float(x.double().abs().sum()) for x in v.values())
    if not np.allclose([s, a], G[key], rtol=1e-12):
        pytest.skip("this torch build draws different random weights than the one the fixture was made with")
    return v


@pytest.mark.parametrize("tag,spec,seed", [('c', 'c', 21), ('s', 's', 22), ('cs', 'cs', 23)])
def test_flownet_every_output_of_every_network(tag, spec, seed):
    v = _variables(spec, seed, 'fn_%s_vars' % tag)
    fw, bw = oflownet.flownet(v, t('fn_%s_im1' % tag), t('fn_%s_im2' % tag), spec, backward_flow=True)
    assert len(fw) == len(spec)
    for n in range(len(spec)):
        assert len(fw[n]) == 5
        for lvl in range(5):
            close(fw[n][lvl], G['fn_%s_net%d_fw%d' % (tag, n, lvl)], rtol=1e-4, atol_rel=1e-5, msg="net %d fw %d" % (n, lvl))
            close(bw[n][lvl], G['fn_%s_net%d_bw%d' % (tag, n, lvl)], rtol=1e-4, atol_rel=1e-5, msg="net %d bw %d" % (n, lvl))


def test_flownet_full_resolution_variant():
    v = oflownet.init_variables('s', True, seed=24)
    s_ = sum(float(x.double().sum()) for x in v.values())
    a_ = sum(float(x.double().abs().sum()) for x in v.values())
    if not np.allclose([s_, a_], G['fn_sfull_vars'], rtol=1e-12):
        pytest.skip("different random weights")
    fw, bw = oflownet.flownet(v, t('fn_sfull_im1'), t('fn_sfull_im2'), 's', full_resolution=True, backward_flow=True)
    assert len(fw[0]) == 7 and tuple(fw[0][0].shape) == (1, 64, 64, 2)
    for lvl in range(7):
        close(fw[0][lvl], G['fn_sfull_fw%d' % lvl], rtol=1e-4, atol_rel=1e-5, msg="fw %d" % lvl)
        close(bw[0][lvl], G['fn_sfull_bw%d' % lvl], rtol=1e-4, atol_rel=1e-5, msg="bw %d" % lvl)


@pytest.mark.parametrize("tag,spec,seed,extra", [('c', 'c', 31, {}), ('s', 's', 32, {'pyramid_loss': False}),
                                                 ('cs', 'cs', 33, {'train_all': True})])
def test_unsupervised_loss_value_flows_and_gradients(tag, spec, seed, extra):
    v = _variables(spec, seed, 'ul_%s_vars' % tag)
    leaves = {k: x.clone().requires_grad_(True) for k, x in v.items()}
    params = dict(synth.KITTI_PARAMS, flownet=spec, **extra)
    loss, ffw, fbw = ounsup.unsupervised_loss(leaves, (t('ul_%s_im1' % tag), t('ul_%s_im2' % tag)), params,
                                              synth.KITTI_NORMALIZATION, augment=False, return_flow=True)
    close(loss, G['ul_%s_loss' % tag], rtol=2e-5)
    close(*golden_data.run_flow(G, ffw, 'ul_%s_flow_fw' % tag), rtol=1e-4, atol_rel=1e-5)
    close(*golden_data.run_flow(G, fbw, 'ul_%s_flow_bw' % tag), rtol=1e-4, atol_rel=1e-5)
    names = [str(n) for n in G['ul_%s_grad_names' % tag]]
    assert names == sorted(leaves)
    grads = torch.autograd.grad(loss, [leaves[k] for k in names], allow_unused=True)
    norms = np.array([0.0 if g is None else float(g.double().norm()) for g in grads])
    want = G['ul_%s_grad_norms' % tag]
    assert np.array_equal(norms == 0.0, want == 0.0)       # the same variables are (not) trained
    # hard masks can flip on 1e-7 differences (SURVEY.md H4): norms to 1e-3, small gradients in full
    np.testing.assert_allclose(norms, want, rtol=2e-3)
    for k, g in zip(names, grads):
        key = 'ul_%s_grad/%s' % (tag, k)
        if key in G:
            err = float((g - torch.from_numpy(G[key])).norm() / max(float(torch.from_numpy(G[key]).norm()), 1e-20))
            assert err < 2e-3, "%s: relative L2 gradient error %.2e" % (k, err)


def test_augmentation_cores_against_the_reference_run():
    """spatial_transformer.transformer, random_affine and random_photometric of the reference, run
    with recorded random draws; the oracle's deterministic cores get the same draws as inputs."""
    from oracle import augment as oaug
    a1, a2, mask = t('aug_im1'), t('aug_im2'), t('aug_mask')
    close(oaug.transformer(a1, t('aug_theta'), (20, 30)), G['aug_transformer'], rtol=1e-4, atol_rel=1e-5)
    flip = torch.where(t('aug_affine_flip') > 0.5, -torch.ones(3), torch.ones(3))      # augment.py:38-41
    assert (flip < 0).any() and (flip > 0).any()                                        # both branches drawn
    theta = oaug.affine_matrices(t('aug_affine_tx'), t('aug_affine_ty'), t('aug_affine_rot'), t('aug_affine_scale'), flip)
    for i, x in enumerate((a1, a2, mask)):
        got = oaug.transformer(x, theta, (x.shape[1], x.shape[2]))
        # positions that land within float rounding of a pixel edge may pick the other neighbour
        diff = (got - torch.from_numpy(G['aug_affine_out%d' % i])).abs()
        assert float((diff > 1e-4).float().mean()) < 2e-3, float((diff > 1e-4).float().mean())
    got = oaug.photometric([a1, a2], t('aug_photo_contrast'), t('aug_photo_gamma'), t('aug_photo_colour'),
                           t('aug_photo_noise'), t('aug_photo_brightness'))
    close(got[0], G['aug_photo_out0'], rtol=1e-5, atol_rel=1e-6)
    close(got[1], G['aug_photo_out1'], rtol=1e-5, atol_rel=1e-6)


def test_product_evaluation_utilities_against_the_reference_run():
    """core/flow_util.py and the resize helpers of core/input.py are plain torch in the product and
    run on the CPU: compared directly with the reference files' own output (SURVEY.md 8f N3)."""
    from unflow_b200.e2eflow.core import flow_util as FU
    from unflow_b200.e2eflow.core import input as IN
    fl, gt, mocc, mnoc = t('fu_flow'), t('fu_gt'), t('fu_mocc'), t('fu_mnoc')

    def same(got, key, tol=2e-5):
        want = G[key]
        got = got.detach().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
        assert got.shape == want.shape, (key, got.shape, want.shape)
        assert np.array_equal(np.isnan(got), np.isnan(want)), key          # atan2(0,0) is NaN in the reference
        np.testing.assert_allclose(np.nan_to_num(got), np.nan_to_num(want), rtol=tol, atol=tol, err_msg=key)

    same(FU.flow_to_color(fl), 'fu_color')
    same(FU.flow_to_color(fl, mocc, max_flow=10.0), 'fu_color_mask_max')
    same(FU.flow_error_image(fl, gt, mocc, mnoc), 'fu_error_log')
    same(FU.flow_error_image(fl, gt, mocc, mnoc, log_colors=False), 'fu_error_lin')
    same(FU.flow_error_image(fl, gt, mocc), 'fu_error_log_nonoc')
    same(FU.flow_error_avg(gt, fl, mocc), 'fu_aee')
    same(FU.outlier_pct(gt, fl, mocc), 'fu_outlier_pct')
    same(FU.outlier_ratio(gt, fl, mnoc, threshold=2.0, relative=None), 'fu_outlier_ratio_abs')
    img = t('in_img')
    same(IN.resize_input(img.reshape(-1), 10, 16, 14, 20), 'in_resize_input', tol=1e-4)
    same(IN.resize_output_crop(img, 10, 24, 3), 'in_resize_output_crop')
    same(IN.resize_output(img, 7, 30, 3), 'in_resize_output', tol=1e-4)
    same(IN.resize_output_flow(fl[:1], 18, 8, 2), 'in_resize_output_flow', tol=1e-4)
    assert [IN.frame_name_to_num(n) for n in ('0000000000.png', '0000000120.png', '7.png')] == G['in_frame_nums'].tolist()


def test_input_pairing_and_config_parsing_against_the_reference_run(tmp_path):
    """File pairing / ordering of core/input.py + kitti/input.py and config parsing of util.py: the
    reference code ran with stub queues that only record the file lists (SURVEY.md 8f N1 / N4)."""
    import json
    from unflow_b200 import run as R
    from unflow_b200.e2eflow.kitti.input import KITTIInput
    listing = json.loads(str(G['input_listing_json']))
    root = str(tmp_path)
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

    rel = lambda f: os.path.relpath(f, root)
    cases = {'plain': (dict(), dict(swap_images=False)),
             'skipped_swap_shift3': (dict(skipped_frames=True), dict(swap_images=True, shift=3)),
             'skipped_shift4_seed5': (dict(skipped_frames=True), dict(swap_images=False, shift=4, seed=5)),
             'skip01': (dict(), dict(swap_images=False, skip=[0, 1]))}
    for tag, (kw, call) in cases.items():
        pairs = KITTIInput(Data(), batch_size=2, dims=(4, 6), normalize=False, **kw).raw_pairs(**call)
        want_first, want_second = listing['raw_' + tag]
        assert [rel(a) for a, _ in pairs] == want_first, tag
        assert [rel(b) for _, b in pairs] == want_second, tag
    ki = KITTIInput(Data(), batch_size=1, dims=(4, 6), normalize=False)
    for tag, hold in (('all', None), ('hold3', 3)):
        f1, f2, occ, noc = listing['train2012_' + tag]
        pairs = ki.image_pairs('data_stereo_flow/training/colored_0', hold)
        got_occ, got_noc = ki._flow_files('data_stereo_flow/training', hold)
        assert [rel(a) for a, _ in pairs] == f1 and [rel(b) for _, b in pairs] == f2, tag
        assert [rel(x) for x in got_occ] == occ and [rel(x) for x in got_noc] == noc, tag

    want = json.loads(str(G['config_json']))
    ini = tmp_path / 'config.ini'
    ini.write_text(str(G['config_ini']))
    cfg = R.config_dict(str(ini))
    assert cfg == want['config']
    ft = dict(cfg['train'])
    ft.update(cfg['train_kitti_ft'])
    R.convert_input_strings(ft, cfg['dirs'])
    assert ft == want['kitti_ft']


def test_learning_rate_schedule_against_the_reference_lines():
    """train.py:224-244 (cut out of the reference source and executed at fixture time) vs
    core/train.py: learning_rate_at."""
    import json
    from unflow_b200.e2eflow.core.train import learning_rate_at
    schedules = json.loads(str(G['lr_schedules_json']))
    for name, prm in schedules.items():
        got = [learning_rate_at(int(it), prm) for it in G['lr_probes']]
        np.testing.assert_allclose(got, G['lr_' + name], rtol=0, atol=0, err_msg=name)


def test_finetune_restore_plan_against_the_reference_lines():
    """train.py:23-37 (executed at fixture time) vs run.py: external_restores and
    tf_checkpoint.net_names."""
    import json
    from unflow_b200 import run as R
    from unflow_b200.e2eflow.core import tf_checkpoint as ck
    plans = json.loads(str(G['restore_plans_json']))
    assert len(plans) == 36
    for key, want in plans.items():
        spec, train_all, n_ft, has = key.split('|')
        params = {'flownet': spec, 'train_all': train_all == 'True', 'finetune': ['ex%d' % i for i in range(int(n_ft))]}
        assert R.external_restores(params, has == '1') == want['external'], key
        assert ck.net_names(spec) == want['net_names'], key


@pytest.mark.parametrize("tag,full,seed,levels", [('s', False, 22, 5), ('sfull', True, 24, 7)])
def test_product_flownet_s_on_the_cpu_against_the_reference_run(tag, full, seed, levels):
    """FlowNetS needs none of the custom CUDA ops, so the PRODUCT's network definition
    (core/flownet.py on the plain conv path) runs on the CPU and is held directly to the output of
    the reference's own flownet.py."""
    from unflow_b200.e2eflow.core.flownet import FlowNetVariables, flownet
    tfv = _variables('s', seed, 'fn_%s_vars' % tag) if not full else oflownet.init_variables('s', True, seed=seed)
    v = FlowNetVariables('s', full, seed=0).load_tf_dict(tfv)
    with torch.no_grad():
        fw, bw = flownet(t('fn_%s_im1' % tag), t('fn_%s_im2' % tag), 's', full_resolution=full, backward_flow=True,
                         variables=v)
    assert len(fw[0]) == levels
    for lvl in range(levels):
        key = ('fn_s_net0_%s%d' if not full else 'fn_sfull_%s%d')
        close(fw[0][lvl], G[key % ('fw', lvl)], rtol=1e-4, atol_rel=1e-5, msg="fw %d" % lvl)
        close(bw[0][lvl], G[key % ('bw', lvl)], rtol=1e-4, atol_rel=1e-5, msg="bw %d" % lvl)


@pytest.mark.parametrize("tag,spec,seed", [('c', 'c', 21), ('cs', 'cs', 23)])
def test_product_flownet_c_and_stack_on_the_cpu_against_the_reference_run(monkeypatch, tag, spec, seed):
    """The product's FlowNetC / stacked definition with its two CUDA entry points (correlation,
    image_warp) swapped for the oracle's CPU ops, against the reference's own flownet.py output."""
    from oracle import ops as oops
    from unflow_b200.e2eflow.core import flownet as F
    monkeypatch.setattr(F, 'correlation', oops.correlation)
    monkeypatch.setattr(F, 'image_warp', oimage_warp.image_warp)
    v = F.FlowNetVariables(spec, False, seed=0).load_tf_dict(_variables(spec, seed, 'fn_%s_vars' % tag))
    with torch.no_grad():
        fw, bw = F.flownet(t('fn_%s_im1' % tag), t('fn_%s_im2' % tag), spec, backward_flow=True, variables=v)
    assert len(fw) == len(spec)
    for n in range(len(spec)):
        for lvl in range(5):
            close(fw[n][lvl], G['fn_%s_net%d_fw%d' % (tag, n, lvl)], rtol=1e-4, atol_rel=1e-5, msg="net %d fw %d" % (n, lvl))
            close(bw[n][lvl], G['fn_%s_net%d_bw%d' % (tag, n, lvl)], rtol=1e-4, atol_rel=1e-5, msg="net %d bw %d" % (n, lvl))


@pytest.mark.parametrize("tag,spec,seed,extra", [('c', 'c', 31, {}), ('s', 's', 32, {'pyramid_loss': False}),
                                                 ('cs', 'cs', 33, {'train_all': True})])
def test_product_unsupervised_loss_host_path_on_the_cpu_against_the_reference_run(monkeypatch, tag, spec, seed, extra):
    """The product's whole Python host path -- unsupervised_loss, flownet, the unfused compute_losses
    and every loss term -- with only the CUDA entry points (correlation, image_warp, forward_warp,
    downsample) swapped for the oracle's CPU ops, against the reference's own unsupervised.py run."""
    from oracle import ops as oops
    from oracle import util as outil
    from unflow_b200.e2eflow.core import flownet as F
    from unflow_b200.e2eflow.core import losses as L
    from unflow_b200.e2eflow.core import unsupervised as U
    monkeypatch.setattr(F, 'correlation', oops.correlation)
    monkeypatch.setattr(F, 'image_warp', oimage_warp.image_warp)
    monkeypatch.setattr(L, 'image_warp', oimage_warp.image_warp)
    monkeypatch.setattr(L, 'forward_warp', oops.forward_warp)
    monkeypatch.setattr(U, 'downsample', outil.downsample)
    v = F.FlowNetVariables(spec, False, seed=0).load_tf_dict(_variables(spec, seed, 'ul_%s_vars' % tag))
    params = dict(synth.KITTI_PARAMS, flownet=spec, **extra)
    loss, ffw, fbw = U.unsupervised_loss((t('ul_%s_im1' % tag), t('ul_%s_im2' % tag)), params,
                                         synth.KITTI_NORMALIZATION, augment=False, return_flow=True, variables=v)
    close(loss, G['ul_%s_loss' % tag], rtol=2e-5)
    close(*golden_data.run_flow(G, ffw, 'ul_%s_flow_fw' % tag), rtol=1e-4, atol_rel=1e-5)
    close(*golden_data.run_flow(G, fbw, 'ul_%s_flow_bw' % tag), rtol=1e-4, atol_rel=1e-5)
    loss.backward()
    names = [str(n) for n in G['ul_%s_grad_names' % tag]]
    want = dict(zip(names, G['ul_%s_grad_norms' % tag]))
    for scope in v.kinds:
        w, b = v.weights(scope)
        for p, name in ((w, scope + '/weights'), (b, scope + '/biases')):
            norm = 0.0 if p.grad is None else float(p.grad.double().norm())
            assert (norm == 0.0) == (want[name] == 0.0), name
            np.testing.assert_allclose(norm, want[name], rtol=2e-3, err_msg=name)
