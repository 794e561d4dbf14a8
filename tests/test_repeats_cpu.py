"""Test-time repeats on the CPU: the restated accumulation (tests/repeats_ref.py) against what the reference's own
evaluate() loops did (tests/golden/ref_repeats.npz), and the host-side argument checks of the two accumulate entry
points of the C ABI (no GPU needed: they refuse before the first CUDA call)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import metric_ref
from tests import repeats_ref as rr
from tests.util import golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _masks(name, ftype, nofeat):
    """Per repeat, the concatenated per-point feature mask ``mask[inds_reverse]`` the reference rebuilds every repeat."""
    if not nofeat:
        return None
    n_scenes, R = rr.CASES[name][4], rr.CASES[name][5]
    return [torch.cat([(lambda it: it[4][it[5]])(rr.scene_inputs(name, sc, r)) for sc in range(n_scenes)]) for r in range(R)]


@pytest.mark.parametrize('name', sorted(rr.CASES))
def test_accumulation_reproduces_the_reference_labels_and_miou(name):
    ftype, ds, _, _, n_scenes, R, nofeat, _ = rr.CASES[name]
    g = golden('ref_repeats.npz')
    assert int(g[f'{name}_seed']) == rr.case_seed(name)
    gt = torch.cat([rr.scene_inputs(name, sc, 0)[2] for sc in range(n_scenes)])
    if 'nuscenes' in ds:
        gt = rr.nuscenes_subset(gt, gt)
    assert np.array_equal(gt.numpy(), g[f'{name}_gt'])
    preds = [torch.from_numpy(p) for p in g[f'{name}_pred']]
    assert preds[0].dtype == (torch.float32 if ftype == 'logits' else torch.float16)
    _, mapper = rr.text_and_mapper(name)
    labels = rr.accumulate(preds, mapper=mapper, masks=_masks(name, ftype, nofeat))
    n_classes = rr.N_CLASSES[ds]
    for r in range(R):
        assert np.array_equal(labels[r].numpy(), g[f'{name}_labels'][r]), f'prefix {r}'
        miou, _ = metric_ref.mean_iou(labels[r].numpy(), gt.numpy(), n_classes)
        assert miou == pytest.approx(float(g[f'{name}_miou'][r]), abs=1e-12)
    if ftype == 'logits':
        for r in range(R):
            own = preds[r].max(1)[1]
            assert np.array_equal(own.numpy(), g[f'{name}_own_labels'][r])
            assert metric_ref.mean_iou(own.numpy(), gt.numpy(), n_classes)[0] == pytest.approx(float(g[f'{name}_own_miou'][r]), abs=1e-12)


def test_first_repeat_turns_negative_zero_into_positive_zero():
    pred = torch.tensor([[-0.0, 1.0]], dtype=torch.float16)
    store = pred + 0.0
    assert not torch.signbit(store[0, 0]) and torch.signbit(pred[0, 0])


_CHILD = r'''
import ctypes, json, os, sys
sys.path.insert(0, sys.argv[1])
from openscene_b200 import _cabi as C
L = C.lib()
X = ctypes.c_void_p(256)                    # never dereferenced: every call below must be refused on the host
def acc(**kw):
    a = dict(feat=X, f16=0, feat2=None, sa=None, sb=None, n_vox=10, c=768, inv=X, n_pts=20, text=X, k=20, nrm=0, store=X,
             first=1, label=X)
    a.update(kw)
    return L.osb_match_accumulate(*a.values(), None)
def lg(**kw):
    a = dict(logits=X, n_vox=10, c=20, inv=X, n_pts=20, store=X, first=1, cur=X, acc=X)
    a.update(kw)
    return L.osb_logits_accumulate(*a.values(), None)
cases = {
    'c256': lambda: acc(c=256), 'k481': lambda: acc(k=481), 'k0': lambda: acc(k=0), 'null_store': lambda: acc(store=None),
    'no_inds_shape': lambda: acc(inv=None), 'half_select': lambda: acc(feat2=X, sa=X), 'neg_pts': lambda: acc(n_pts=-1),
    'lg_null_store': lambda: lg(store=None), 'lg_c0': lambda: lg(c=0), 'lg_no_inds_shape': lambda: lg(inv=None),
}
if os.environ.get('OSB_MATCH_SIMT') == '1':
    cases = {'simt': lambda: acc()}
out = {}
for name, f in cases.items():
    rc = f()
    out[name] = [rc, (L.osb_last_error() or b'').decode()]
print('RESULT ' + json.dumps(out))
'''


def _child(env_extra=None):
    env = dict(os.environ, **(env_extra or {}))
    p = subprocess.run([sys.executable, '-c', _CHILD, ROOT], capture_output=True, text=True, timeout=300, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    return json.loads([l for l in p.stdout.splitlines() if l.startswith('RESULT ')][-1][len('RESULT '):])


def test_accumulate_entries_refuse_bad_arguments_on_the_host():
    res = _child()
    expect = {'c256': 'feature width 256', 'k481': 'outside 1..480', 'k0': 'outside 1..480', 'null_store': 'store',
              'no_inds_shape': 'must equal n_vox', 'half_select': 'select arrays', 'neg_pts': 'bad shape',
              'lg_null_store': 'store', 'lg_c0': 'bad shape', 'lg_no_inds_shape': 'must equal n_vox'}
    for name, needle in expect.items():
        rc, err = res[name]
        assert rc != 0, f'{name}: accepted'
        assert needle in err, f'{name}: {err!r}'


def test_accumulate_refuses_the_cuda_core_cross_check_path():
    rc, err = _child({'OSB_MATCH_SIMT': '1'})['simt']
    assert rc != 0 and 'OSB_MATCH_SIMT' in err
