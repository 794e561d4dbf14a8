"""Host half of the drop-in voxeliser against what the REFERENCE's own class returned (tests/golden/ref_voxelizer_*.npz,
written by scripts/make_golden.py from the reference's ``dataset/voxelizer.py``).

``openscene_b200.voxelize.Voxelizer.get_transformation_matrix`` must consume the global NumPy RNG exactly as
``dataset/voxelizer.py:46-76`` does -- the loaders seed / share that stream (dataset/point_loader.py:58-61), so a different draw
order would change every augmentation after it.  Compared bit for bit, matrices and the next draws of the stream, over the
constructor forms the reference's loaders use; the NumPy oracle (oracle/voxelize_ref.py) is held to the same reference on random
clouds beyond the four committed fixtures."""
import numpy as np
import pytest

from tests.util import golden

ROT = ((-np.pi / 64, np.pi / 64), (-np.pi / 64, np.pi / 64), (-np.pi, np.pi))        # point_loader.py:58-61
FORMS = [
    dict(voxel_size=0.02, use_augmentation=True, scale_augmentation_bound=(0.9, 1.1), rotation_augmentation_bound=ROT),
    dict(voxel_size=0.05, use_augmentation=True, scale_augmentation_bound=(0.9, 1.1), rotation_augmentation_bound=ROT),
    dict(voxel_size=0.02, use_augmentation=False, scale_augmentation_bound=(0.9, 1.1), rotation_augmentation_bound=ROT),
    dict(voxel_size=0.02, use_augmentation=True, scale_augmentation_bound=None, rotation_augmentation_bound=ROT),
    dict(voxel_size=0.02, use_augmentation=True, scale_augmentation_bound=(0.9, 1.1), rotation_augmentation_bound=None),
    dict(voxel_size=0.02, use_augmentation=True, scale_augmentation_bound=(0.9, 1.1),
         rotation_augmentation_bound=(None, (-0.1, 0.1), (-np.pi, np.pi))),
]
MATRIX_SEEDS = range(25)


def form_kwargs(form):
    return dict(FORMS[form], clip_bound=None, translation_augmentation_ratio_bound=((-0.2, 0.2), (-0.2, 0.2), (0, 0)),
                ignore_label=255)


def random_clouds():
    """(trial, points, augmentation on, voxel size): dense clouds with many duplicates, negative coordinates, fp32 and fp64."""
    rng = np.random.RandomState(2024)
    for trial in range(12):
        n = int(rng.randint(500, 6000))
        extent, shift = float(rng.uniform(0.3, 5.0)), float(rng.uniform(-3.0, 1.0))
        dtype = np.float32 if trial % 3 == 0 else np.float64
        pts = (rng.rand(n, 3) * extent + shift).astype(dtype)
        yield trial, pts, trial % 2 == 0, float(rng.choice([0.02, 0.05, 0.1]))


@pytest.mark.parametrize('form', range(len(FORMS)))
def test_matrix_and_rng_stream_equal_the_reference(form):
    from openscene_b200.voxelize import Voxelizer as Mine
    g = golden('ref_voxelizer_matrices.npz')
    mine = Mine(**form_kwargs(form))
    for seed in MATRIX_SEEDS:
        np.random.seed(seed)
        b_v, b_r = mine.get_transformation_matrix()
        tail_mine = np.random.rand(4)                    # what the next consumer of the stream would see
        assert np.array_equal(g['m_v'][form, seed], b_v) and np.array_equal(g['m_r'][form, seed], b_r), (form, seed)
        assert np.array_equal(g['tail'][form, seed], tail_mine), "the two classes consumed the RNG stream differently"


def test_oracle_equals_the_reference_on_random_clouds():
    """oracle/voxelize_ref.py vs the reference's voxelize() beyond the committed fixtures, augmentation on and off; the
    rigid matrix is the one the reference drew for the cloud."""
    from oracle import voxelize_ref
    g = golden('ref_voxelizer_random.npz')
    for trial, pts, _, _ in random_clouds():
        cv, o_inds, o_inv, _ = voxelize_ref.voxelize(pts, g[f'matrix_{trial}'])
        assert np.array_equal(cv, g[f'coords_{trial}']), trial
        assert np.array_equal(o_inds, g[f'inds_{trial}']) and np.array_equal(o_inv, g[f'inds_reverse_{trial}']), trial
