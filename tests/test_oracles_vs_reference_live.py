"""The CPU oracles against what the REFERENCE's own functions returned on random cases beyond the other fixtures
(tests/golden/ref_fusion_random.npz and ref_metric_random.npz, written by scripts/make_golden.py from the reference tree).

* oracle/fusion_ref.compute_mapping  vs  scripts/feature_fusion/fusion_util.py: PointCloudToImageMapper.compute_mapping
* oracle/metric_ref                  vs  util/metric.py (confusion_matrix, evaluate) and util/util.py (intersectionAndUnion[GPU])
Bit-exact (integer work); mIoU to 1e-12."""
import numpy as np
import pytest

from tests.util import golden


def fusion_cases():
    """(seed, points, poses, depths, intrinsics, cut bound, visibility threshold) of the eight view sets."""
    from openscene_b200.synth import fusion_case
    for seed in range(100, 108):
        with_depth = seed % 3 != 0
        pts, poses, depths, intr = fusion_case(seed, 2500 + 300 * (seed % 5), with_depth)
        yield seed, pts, poses, depths, intr, [0, 5, 10, 20][seed % 4], [0.25, 0.1, 0.5][seed % 3]


def metric_cases():
    """(seed, class count, dataset name, pred, gt, with 'no feature' predictions) of the six label sets."""
    for seed, (C, ds) in enumerate([(20, 'scannet_3d'), (21, 'matterport_3d'), (40, 'matterport_3d_40'), (80, 'matterport_3d_80'),
                                    (160, 'matterport_3d_160'), (16, 'nuscenes_3d')]):
        rng = np.random.RandomState(500 + seed)
        n = 20000
        gt = rng.randint(0, C, n)
        gt[rng.rand(n) < 0.15] = 255
        gt[gt == (seed % C)] = (seed + 1) % C                  # one class never occurs in gt
        pred = np.where(rng.rand(n) < 0.5, np.minimum(gt, C - 1), rng.randint(0, C, n))
        nofeat = seed % 2 == 1
        if nofeat:
            pred[rng.rand(n) < 0.07] = 256
        yield seed, C, ds, pred, gt, nofeat


def test_fusion_mapping_oracle_equals_the_reference_on_random_views():
    from oracle import fusion_ref
    g = golden('ref_fusion_random.npz')
    n_vis = 0
    for seed, pts, poses, depths, intr, cut, thres in fusion_cases():
        want_all = g[f'mapping_{seed}']
        assert len(want_all) == len(poses), seed
        for pose, depth, want in zip(poses, depths, want_all):
            got = fusion_ref.compute_mapping(pose, pts, depth, intr, (320, 240), cut, thres)
            assert np.array_equal(got, want), seed
            n_vis += int(want[:, 2].sum())
    assert n_vis > 5000                                       # the cases exercise the visible branch


def test_metric_oracles_equal_the_reference_on_random_labels():
    from oracle import metric_ref
    g = golden('ref_metric_random.npz')
    for seed, C, ds, pred, gt, nofeat in metric_cases():
        assert np.array_equal(metric_ref.confusion_matrix(pred, gt, C).astype(np.int64), g[f'confusion_{seed}']), ds
        assert metric_ref.mean_iou(pred, gt, C)[0] == pytest.approx(float(g[f'miou_{seed}']), rel=1e-12), ds
        if not nofeat:
            # the reference's NumPy and torch versions agreed with each other when the fixture was made
            i, u, t = metric_ref.intersection_and_union(pred, gt, C)
            for a, name in ((i, 'inter'), (u, 'union'), (t, 'target')):
                assert np.array_equal(a, g[f'{name}_{seed}']), (ds, name)
