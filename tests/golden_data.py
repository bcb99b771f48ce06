"""Helpers for the golden fixtures under tests/golden/.

Inputs that are seeded draws of torch's CPU generator are not stored: a fixture keeps their SHA-256
and the tests draw them again, checked against it.  Outputs too large to keep whole are stored as a
fixed sample (``sample_index``: numpy's legacy RandomState, whose streams never change)."""
import hashlib
import os

import numpy as np
import torch

import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SAMPLE = 4096


def digest(a):
    a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.float32).tobytes()).hexdigest()


def sample_index(n, k=SAMPLE):
    """Flat indices of the stored sample of an n-element output: all of them up to k, else k fixed ones."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.RandomState(0).choice(n, k, replace=False))


def sample(a, k=SAMPLE):
    a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
    return a.reshape(-1)[sample_index(a.size, k)]


def check_digest(name, a, want):
    assert digest(a) == str(want), ("%s: this torch build draws other inputs than the one the fixture "
                                    "was made with" % name)
    return a


# ------------------------------------------------------------------------------------------------
# reference_run.npz (tests/golden/make_reference_run.py)
# ------------------------------------------------------------------------------------------------
# input images of the flownet / unsupervised_loss cases: key prefix -> (height, width, seed, centred)
RUN_IMAGES = {'fn_c': (64, 128, 121, True), 'fn_s': (64, 64, 122, True), 'fn_cs': (64, 64, 123, True),
              'fn_sfull': (64, 64, 124, True),
              'ul_c': (128, 128, 131, False), 'ul_s': (128, 128, 132, False), 'ul_cs': (128, 128, 133, False)}
# full-resolution output flows of unsupervised_loss, stored as a sample of RUN_FLOW_SAMPLE elements
RUN_FLOWS = ['ul_%s_flow_%s' % (tag, d) for tag in ('c', 's', 'cs') for d in ('fw', 'bw')]
RUN_FLOW_SAMPLE = 8192


def run_images(prefix):
    h, w, seed, centred = RUN_IMAGES[prefix]
    i1, i2, _ = synth.image_pair(1, h, w, seed=seed)
    if centred:
        i1, i2 = i1 / 255.0 - 0.4, i2 / 255.0 - 0.4
    return i1.numpy(), i2.numpy()


def shrink_reference_run(out):
    """The arrays the reference run produced -> what reference_run.npz stores."""
    out = dict(out)
    for prefix in RUN_IMAGES:
        for key, a in zip((prefix + '_im1', prefix + '_im2'), run_images(prefix)):
            assert np.array_equal(out[key], a), key
            out[key + '_sha256'] = np.array(digest(out.pop(key)))
    for key in RUN_FLOWS:
        flow = out.pop(key)
        out[key + '_shape'] = np.array(flow.shape)
        out[key + '_sample'] = sample(flow, RUN_FLOW_SAMPLE)
    return out


class ReferenceRun(dict):
    """reference_run.npz as a dict; the input images that are not stored are drawn on first use."""

    def __missing__(self, key):
        prefix, _, which = key.rpartition('_')
        if prefix not in RUN_IMAGES or which not in ('im1', 'im2'):
            raise KeyError(key)
        for k, a in zip((prefix + '_im1', prefix + '_im2'), run_images(prefix)):
            self[k] = check_digest(k, a, self[k + '_sha256'])
        return self[key]


def load_reference_run():
    with np.load(os.path.join(GOLDEN, "reference_run.npz")) as z:
        return ReferenceRun((k, z[k]) for k in z.files)


def run_flow(G, got, key):
    """(sample of the output flow ``got``, the stored sample of the reference's) for RUN_FLOWS keys."""
    assert tuple(got.shape) == tuple(G[key + '_shape']), (key, tuple(got.shape))
    idx = torch.from_numpy(sample_index(got.numel(), RUN_FLOW_SAMPLE)).to(got.device)
    return got.detach().reshape(-1)[idx], G[key + '_sample']
