"""The REFERENCE's own, unmodified ``models/mink_unet.py`` / ``models/disnet.py``, imported on top of THIS repository's
``MinkowskiEngine`` package (the drop-in boundary, SURVEY.md 8b), as recorded in tests/golden/ref_models.npz by
scripts/make_golden.py: state-dict keys, shapes and a fixed sample of the weights each architecture gets from
``torch.manual_seed(0)``.  The table-driven mirror ``openscene_b200/minkunet.py`` must build exactly that, so existing
checkpoints load with ``strict=True`` (run/evaluate.py:168) and the same seed gives the same network; the GPU test runs
that network the way run/evaluate.py:284-289 calls it."""
import types

import numpy as np
import pytest
import torch

from tests.util import golden, rel_row_err

SAMPLE = 16           # weights recorded per state-dict entry, evenly spaced over its flattened values


def weight_sample(sd):
    """[entries, SAMPLE] float64 (NaN-padded): evenly spaced values of every state-dict entry; [entries, 2]: sum, sum of squares."""
    sample = np.full((len(sd), SAMPLE), np.nan)
    sums = np.zeros((len(sd), 2))
    for i, v in enumerate(sd.values()):
        flat = v.detach().double().reshape(-1).numpy()
        pick = np.unique(np.linspace(0, flat.size - 1, min(flat.size, SAMPLE)).astype(np.int64))
        sample[i, :len(pick)] = flat[pick]
        sums[i] = flat.sum(), (flat * flat).sum()
    return sample, sums


def assert_matches_reference(model, tag):
    """`model`'s state dict == the reference model recorded under `tag`: keys and shapes exactly, weights to fp32 rounding (the
    CPU normal sampler may differ in the last bit between instruction sets)."""
    g = golden('ref_models.npz')
    sd = model.state_dict()
    assert list(sd.keys()) == g[f'{tag}_keys'].tolist()
    assert [str(tuple(v.shape)) for v in sd.values()] == g[f'{tag}_shapes'].tolist()
    sample, sums = weight_sample(sd)
    np.testing.assert_allclose(sample, g[f'{tag}_sample'], rtol=1e-6, atol=1e-9, equal_nan=True)
    np.testing.assert_allclose(sums, g[f'{tag}_sums'], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize('arch', ['MinkUNet18A', 'MinkUNet34C'])
def test_reference_model_file_builds_on_the_product_package(arch):
    from openscene_b200 import minkunet
    g = golden(f'unet_{arch}.npz')
    torch.manual_seed(0)
    mirror = minkunet.mink_unet(in_channels=3, out_channels=768, D=3, arch=arch)
    assert_matches_reference(mirror, arch)
    sd = mirror.state_dict()
    assert list(sd.keys()) == g['state_keys'].tolist()
    assert [str(tuple(v.shape)) for v in sd.values()] == g['state_shapes'].tolist()
    assert sum(p.numel() for p in mirror.parameters()) == int(g['n_params'])
    # a checkpoint written by one build loads strictly into another
    torch.manual_seed(1)
    minkunet.mink_unet(in_channels=3, out_channels=768, D=3, arch=arch).load_state_dict(sd, strict=True)


def test_reference_disnet_on_the_product_package():
    from openscene_b200 import minkunet
    cfg = types.SimpleNamespace(arch_3d='MinkUNet18A', feature_2d_extractor='openseg')
    torch.manual_seed(0)
    assert_matches_reference(minkunet.DisNet(cfg=cfg), 'DisNet_openseg')
    g = golden('unet_MinkUNet18A.npz')
    assert [k[len('net3d.'):] for k in minkunet.DisNet(cfg=cfg).state_dict()] == g['state_keys'].tolist()
    cfg.feature_2d_extractor = 'lseg'
    net = minkunet.DisNet(cfg=cfg)
    assert net.net3d.final.kernel.shape == (96, 512)
    assert list(net.state_dict().keys()) == golden('ref_models.npz')['DisNet_lseg_keys'].tolist()
    assert [str(tuple(v.shape)) for v in net.state_dict().values()] == golden('ref_models.npz')['DisNet_lseg_shapes'].tolist()


@pytest.mark.gpu
@pytest.mark.parametrize('arch', ['MinkUNet18A', 'MinkUNet34C'])
def test_reference_model_file_forwards_on_the_gpu(arch):
    """`model(sinput)` exactly as run/evaluate.py:284-289 calls it, on the network the reference builds, product engine
    underneath."""
    import MinkowskiEngine as ME
    from openscene_b200 import minkunet, synth
    g = golden(f'unet_{arch}.npz')
    torch.manual_seed(0)
    model = minkunet.mink_unet(in_channels=3, out_channels=768, D=3, arch=arch)
    assert_matches_reference(model, arch)
    synth.randomize_bn_stats(model, 1)
    model = model.eval().cuda()
    with torch.no_grad():
        out = model(ME.SparseTensor(torch.from_numpy(g['feats']).cuda(), torch.from_numpy(g['coords']).cuda()))
    assert rel_row_err(out.cpu().numpy()[g['rows']], g['out_rows']) < 1e-3


ALL_ARCHS = ['MinkUNet14A', 'MinkUNet14B', 'MinkUNet14C', 'MinkUNet14D', 'MinkUNet18A', 'MinkUNet18B', 'MinkUNet18D',
             'MinkUNet34A', 'MinkUNet34B', 'MinkUNet34C']
OTHER_ARCHS = [a for a in ALL_ARCHS if a not in ('MinkUNet18A', 'MinkUNet34C')]
REJECTED = ('MinkUNet50', 'MinkUNet101', 'nonsense')


@pytest.mark.parametrize('arch', OTHER_ARCHS)
def test_every_factory_architecture_matches_the_mirror(arch):
    """The eight other names `mink_unet()` accepts (models/mink_unet.py:241-263): the reference's class on the product package and
    the table-driven mirror give the same state-dict keys, shapes and seeded weights, and load each other's checkpoints."""
    from openscene_b200 import minkunet
    torch.manual_seed(0)
    mir = minkunet.mink_unet(in_channels=3, out_channels=20, D=3, arch=arch)
    assert_matches_reference(mir, f'{arch}_20')
    torch.manual_seed(1)
    minkunet.mink_unet(in_channels=3, out_channels=20, D=3, arch=arch).load_state_dict(mir.state_dict(), strict=True)


def test_factory_rejects_what_the_reference_rejects():
    """`mink_unet(arch=...)` raises for names outside its list -- MinkUNet50 / MinkUNet101 included: the reference defines those
    classes (models/mink_unet.py:191-199) but gives them no PLANES, so they cannot be constructed there either."""
    from openscene_b200 import minkunet
    assert golden('ref_models.npz')['rejected'].tolist() == list(REJECTED)
    for arch in REJECTED:
        with pytest.raises(Exception):
            minkunet.mink_unet(arch=arch)
