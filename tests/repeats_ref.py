"""Test-time repeats: the seeded inputs of tests/golden/ref_repeats.npz and a CPU restatement of the accumulation.

The golden file holds what the reference's own ``run/evaluate.py:evaluate()`` and ``run/eval_mink.py:evaluate()`` did with
these inputs (scripts/make_golden.py ``ref_repeats``).  The inputs themselves are not stored: ``scene_inputs`` and
``voxel_features`` regenerate them from the seeds, so the GPU tests can feed the same numbers to the device kernels.
"""
import numpy as np
import torch

# name -> (feature_type, dataset, K text rows (or C logits), feature width, scenes, repeats, mark_no_feature, mapper)
CASES = {
    'ensemble': ('ensemble', 'scannet_3d', 20, 512, 2, 3, False, False),
    'distill': ('distill', 'scannet_3d', 20, 512, 1, 3, False, False),
    'fusion_nofeat': ('fusion', 'scannet_3d', 20, 512, 1, 3, True, False),
    'nuscenes': ('ensemble', 'nuscenes_3d', 16, 512, 1, 3, False, True),
    'mink_logits': ('logits', 'scannet_3d', 20, 20, 1, 3, False, False),
}
N_CLASSES = {'scannet_3d': 20, 'nuscenes_3d': 16}
N_PTS, N_VOX = 500, 220


def case_seed(name):
    return 1000 + sorted(CASES).index(name) * 100


def text_and_mapper(name):
    """Unit-norm fp16 text embeddings [K, C] and the case's mapper (``map_nuscenes_details``-style: several text rows
    name the same evaluation class) or None."""
    ftype, _, k, c, _, _, _, with_mapper = CASES[name]
    if ftype == 'logits':
        return None, None
    t = np.random.RandomState(case_seed(name) + 1).randn(k, c)
    t /= np.linalg.norm(t, axis=1, keepdims=True)
    mapper = None
    if with_mapper:
        mapper = np.arange(k, dtype=np.int64)
        mapper[[3, 7, 12]] = [2, 6, 11]
    return torch.from_numpy(t.astype(np.float16)), (torch.from_numpy(mapper) if mapper is not None else None)


def scene_inputs(name, scene, rep):
    """What the loader yields for (scene, repeat): coords int32 [Nv,4], feat fp32 [Nv,3], label int64 [Np],
    feat_3d fp16 [Nv,C], mask bool [Nv], inds_reverse int64 [Np].  The gt labels depend on the scene only."""
    ftype, ds, _, c, _, _, _, _ = CASES[name]
    s = case_seed(name) + 10 * scene
    g = np.random.RandomState(s)
    label = g.randint(0, N_CLASSES[ds], N_PTS).astype(np.int64)
    label[g.rand(N_PTS) < (0.25 if 'nuscenes' in ds else 0.05)] = 255
    r = np.random.RandomState(s + rep + 1)
    nv = N_VOX - 7 * rep + 3 * scene
    coords = np.concatenate([np.zeros((nv, 1), np.int32), r.randint(0, 40, (nv, 3)).astype(np.int32)], 1)
    inds_reverse = np.concatenate([np.arange(nv), r.randint(0, nv, N_PTS - nv)])
    r.shuffle(inds_reverse)
    feat_3d = (r.randn(nv, c) * (0.5 + r.rand(nv, 1))).astype(np.float16) if ftype != 'logits' else np.zeros((nv, 0), np.float16)
    feat_3d[r.rand(nv) < 0.1] = 0                                     # voxels without a fused feature are zero rows (val split)
    mask = np.abs(feat_3d.astype(np.float32)).sum(1) > 0 if ftype != 'logits' else np.ones(nv, bool)
    return (torch.from_numpy(coords), torch.ones(nv, 3), torch.from_numpy(label), torch.from_numpy(feat_3d),
            torch.from_numpy(mask), torch.from_numpy(inds_reverse.astype(np.int64)))


def voxel_features(name, scene, rep, n_vox):
    """The network's output for (scene, repeat): fp32 [Nv, C] (class logits for 'logits')."""
    _, _, _, c, _, _, _, _ = CASES[name]
    r = np.random.RandomState(case_seed(name) + 10 * scene + rep + 50)
    return torch.from_numpy((r.randn(n_vox, c) * (0.3 + r.rand(n_vox, 1))).astype(np.float32))


def accumulate(preds, mapper=None, masks=None):
    """run/evaluate.py:399-425 (and run/eval_mink.py:208-210 for fp32 logits): ``store = 0.0``, then per repeat
    ``store = pred + store`` in the dtype of ``pred`` and the labels ``store.float().max(1)[1]``, mapped through
    ``mapper`` and set to 256 where that repeat's own mask is False.  preds: R tensors [N, K] over the concatenated
    scenes (the nuScenes subset already taken).  Returns R label tensors, one per repeat prefix."""
    store, out = 0.0, []
    for r, pred in enumerate(preds):
        store = pred + store
        lab = store.float().max(1)[1]
        if mapper is not None:
            lab = mapper[lab]
        if masks is not None:
            lab = lab.clone()
            lab[~masks[r]] = 256
        out.append(lab)
    return out


def nuscenes_subset(x, gt):
    """evaluate.py:335-339 / eval_mink.py:185-188: only points with gt != 255 are evaluated."""
    return x[torch.as_tensor(gt) != 255]
