"""Test-time repeats on the device: the accumulate epilogue of the tensor-core matcher and the logits accumulation bit
for bit against torch's fold, the reference's own loop outputs (tests/golden/ref_repeats.npz), and ``RepeatEvaluator``
against R separate single-pass evaluations on the same voxelisation matrices."""
import numpy as np
import pytest
import torch

from openscene_b200 import matching, synth
from openscene_b200.fused_features import remap_fused_features
from openscene_b200.metric import ConfusionMeter
from openscene_b200.pipeline import RepeatEvaluator
from openscene_b200.voxelize import voxelize_points
from tests import repeats_ref as rr
from tests.util import golden

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _inputs(c, k, seed, n_vox=1500, n_pts=4000):
    g = torch.Generator().manual_seed(seed)
    f = torch.randn(n_vox, c, generator=g) * (0.2 + torch.rand(n_vox, 1, generator=g))
    f[:40] = 0
    f[:40, 0] = 2.0 ** -24                                   # one fp16 subnormal: scores round to +0 or -0 by the text's sign
    f2 = (torch.randn(n_vox, c, generator=g) * 0.5).half()
    inv = torch.randint(0, n_vox, (n_pts,), generator=g)
    text = torch.from_numpy(synth.text_embeddings(k, c, seed=seed))
    return f.to(DEV), f2.to(DEV), inv.to(DEV), text.to(DEV)


def _bits(x):
    return x.view(torch.int16)


@pytest.mark.parametrize('c', [512, 768])
@pytest.mark.parametrize('k', [16, 20, 160])
@pytest.mark.parametrize('mode', ['distill', 'fusion', 'ensemble'])
def test_match_accumulate_is_the_fp16_fold_of_the_match_scores(mode, k, c):
    R = 3
    store = torch.empty((4000, k), dtype=torch.float16, device=DEV)
    ref = 0.0
    saw_neg_zero = False
    for r in range(R):
        f, f2, inv, text = _inputs(c, k, 10 * r + k + c)
        if mode == 'distill':
            s, _ = matching.match_distill(f, inv, text)
            label = matching.match_accumulate(f, inv, text, store, r == 0)
        elif mode == 'fusion':
            s, _ = matching.match_fusion(f.half(), inv, text)
            label = matching.match_accumulate(f.half(), inv, text, store, r == 0)
        else:
            s, _, _, _ = matching.match_ensemble(f, f2, inv, text)
            _, _, smax2d = matching._scores(f2, inv, text, normalize=True, want_scores=False, want_smax=True)
            _, _, smax3d = matching._scores(f, inv, text, normalize=True, want_scores=False, want_smax=True)
            label = matching.match_accumulate(f, inv, text, store, r == 0, feat2=f2, smax3d=smax3d, smax2d=smax2d)
        saw_neg_zero |= bool((torch.signbit(s) & (s == 0)).any())
        ref = s + ref
        assert torch.equal(_bits(store), _bits(ref)), f'repeat {r}: store differs from the torch fold'
        assert torch.equal(label, ref.float().max(1)[1]), f'repeat {r}: label is not the first argmax of the store'
    if mode != 'ensemble':
        assert saw_neg_zero                                  # the -0 -> +0 rule of the first repeat was exercised


@pytest.mark.parametrize('c', [20, 13, 40])
def test_logits_accumulate_is_the_fp32_fold_and_both_argmaxes(c):
    g = torch.Generator().manual_seed(c)
    n_vox, n_pts = 3000, 7000
    store = torch.empty((n_pts, c), dtype=torch.float32, device=DEV)
    ref = 0.0
    for r in range(4):
        x = torch.round(torch.randn(n_vox, c, generator=g) * 4) / 4       # coarse grid: ties and -0 on purpose
        x[:5] = -0.0
        x[5:8] = float('-inf')
        x, inv = x.to(DEV), torch.randint(0, n_vox, (n_pts,), generator=g).to(DEV)
        cur, acc = matching.logits_accumulate(x, inv, store, r == 0)
        pred = x[inv]
        ref = pred + ref
        assert torch.equal(store.view(torch.int32), ref.view(torch.int32))
        assert torch.equal(cur, pred.max(1)[1]) and torch.equal(acc, ref.max(1)[1])


def test_accumulate_wrappers_refuse_mismatched_shapes():
    f, _, inv, text = _inputs(768, 20, 0)
    with pytest.raises(ValueError, match='store must be'):
        matching.match_accumulate(f, inv, text, torch.empty((inv.shape[0], 21), dtype=torch.float16, device=DEV), True)
    with pytest.raises(ValueError, match='store must be'):
        matching.match_accumulate(f, inv, text, torch.empty((inv.shape[0], 20), dtype=torch.float32, device=DEV), True)
    with pytest.raises(ValueError, match='store must be'):
        matching.logits_accumulate(f[:, :20], inv, torch.empty((inv.shape[0] - 1, 20), device=DEV), True)
    with pytest.raises(RuntimeError, match='outside 1..480'):
        t = torch.from_numpy(synth.text_embeddings(481, 768)).to(DEV)
        matching.match_accumulate(f, inv, t, torch.empty((inv.shape[0], 481), dtype=torch.float16, device=DEV), True)


@pytest.mark.parametrize('name', sorted(rr.CASES))
def test_golden_reference_loops(name):
    """The seeded inputs the reference's evaluate() saw, through the device kernels: per-prefix labels and mIoU."""
    ftype, ds, k, c, n_scenes, R, nofeat, _ = rr.CASES[name]
    g = golden('ref_repeats.npz')
    text, mapper = rr.text_and_mapper(name)
    text = text.to(DEV) if text is not None else None
    mapper = mapper.to(DEV) if mapper is not None else None
    labels = [[] for _ in range(R)]
    own = [[] for _ in range(R)]
    gts = []
    for sc in range(n_scenes):
        store = None
        for r in range(R):
            coords, _, gt, feat_3d, mask, inv = rr.scene_inputs(name, sc, r)
            inv = inv.to(DEV)
            out = rr.voxel_features(name, sc, r, coords.shape[0]).to(DEV)
            if r == 0:
                gts.append(gt)
            if ftype == 'logits':
                store = torch.empty((inv.shape[0], c), dtype=torch.float32, device=DEV) if store is None else store
                cur, lab = matching.logits_accumulate(out, inv, store, r == 0)
                own[r].append(cur.cpu())
            else:
                store = torch.empty((inv.shape[0], k), dtype=torch.float16, device=DEV) if store is None else store
                f3 = feat_3d.to(DEV)
                if ftype == 'distill':
                    lab = matching.match_accumulate(out, inv, text, store, r == 0)
                elif ftype == 'fusion':
                    lab = matching.match_accumulate(f3, inv, text, store, r == 0)
                else:
                    _, _, s2 = matching._scores(f3, inv, text, normalize=True, want_scores=False, want_smax=True)
                    _, _, s3 = matching._scores(out, inv, text, normalize=True, want_scores=False, want_smax=True)
                    lab = matching.match_accumulate(out, inv, text, store, r == 0, feat2=f3, smax3d=s3, smax2d=s2)
            if mapper is not None:
                lab = mapper[lab]
            if nofeat:
                lab = lab.clone()
                lab[~mask.to(DEV)[inv]] = 256
            labels[r].append(lab.cpu())
    gt = torch.cat(gts)
    keep = gt != 255 if 'nuscenes' in ds else torch.ones_like(gt, dtype=torch.bool)
    for r in range(R):
        lab = torch.cat(labels[r])[keep]
        ref = torch.from_numpy(g[f'{name}_labels'][r])
        if ftype == 'logits':                                # fp32 adds and argmax: exact
            assert torch.equal(lab, ref)
            assert torch.equal(torch.cat(own[r]), torch.from_numpy(g[f'{name}_own_labels'][r]))
        else:                                                # tensor-core fp16 product vs the CPU's: last-bit ties
            assert (lab == ref).float().mean() >= 0.995, f'prefix {r}'
        m = ConfusionMeter(rr.N_CLASSES[ds], DEV)
        m.update(torch.cat(labels[r]).to(DEV), gt.to(DEV))                # gt 255 dropped by the ignore id
        assert abs(m.evaluate()[0] - float(g[f'{name}_miou'][r])) <= 5e-3, f'prefix {r}'


# ------------------------------------------------------------------ RepeatEvaluator end to end
R = 5


def _room(seed=3, nuscenes=False):
    pts = synth.room_points((1.0, 0.8, 0.6), 2, seed=seed)
    rng = np.random.RandomState(seed)
    n = len(pts)
    n_classes = 16 if nuscenes else 20
    gt = rng.randint(0, n_classes, n)
    gt[rng.rand(n) < (0.3 if nuscenes else 0.05)] = 255
    mask_full = rng.rand(n) < 0.8
    feat = (rng.randn(int(mask_full.sum()), 768) * 0.3).astype(np.float16)
    from openscene_b200 import pipeline
    from openscene_b200.voxelize import Voxelizer
    vox = Voxelizer(voxel_size=0.02, use_augmentation=True, scale_augmentation_bound=pipeline.LOADER_SCALE_BOUND,
                    rotation_augmentation_bound=pipeline.LOADER_ROTATION_BOUND)
    np.random.seed(seed + 1)
    mats = [(lambda vr: vr[1] @ vr[0])(vox.get_transformation_matrix()) for _ in range(R)]
    return (torch.from_numpy(pts).to(DEV), torch.from_numpy(gt).to(DEV), (torch.from_numpy(feat).to(DEV), torch.from_numpy(mask_full).to(DEV)),
            mats)


_MODELS = {}


def _model(out_channels):
    if out_channels not in _MODELS:
        _MODELS[out_channels] = synth.build_model('MinkUNet18A', out_channels, seed=7).eval().to(DEV)
    return _MODELS[out_channels]


def _solo(engine, ftype, points, gt, fused, mats, text, n_classes, mapper=None, nofeat=False):
    """R separate single-pass evaluations with the accumulation in torch: (network outputs, per-prefix labels, mIoUs)."""
    store, outs, labels, mious = 0.0, [], [], []
    for M in mats:
        cv, inds, inv, _ = voxelize_points(points, M)
        coords = torch.zeros((cv.shape[0], 4), dtype=torch.int32, device=DEV)
        coords[:, 1:] = cv
        fv, mv = remap_fused_features(fused[0], fused[1], inds, split='val', device=DEV)
        out = engine(coords, torch.ones((cv.shape[0], 3), device=DEV)) if ftype != 'fusion' else None
        if ftype == 'distill':
            s, _ = matching.match_distill(out, inv, text)
        elif ftype == 'fusion':
            s, _ = matching.match_fusion(fv, inv, text)
        elif ftype == 'ensemble':
            s, _, _, _ = matching.match_ensemble(out, fv, inv, text)
        else:
            s = out[inv]
        outs.append(out)
        store = s + store
        lab = store.float().max(1)[1]
        if mapper is not None:
            lab = mapper[lab]
        if nofeat:
            lab[~mv[inv]] = 256
        labels.append(lab)
        m = ConfusionMeter(n_classes, DEV)
        m.update(lab, gt)
        mious.append(m.evaluate()[0])
    return outs, labels, mious


@pytest.mark.parametrize('ftype', ['ensemble', 'distill', 'logits'])
def test_repeat_evaluator_matches_separate_passes(ftype):
    from openscene_b200.engine import FusedMinkUNet
    points, gt, fused, mats = _room()
    engine = FusedMinkUNet(_model(20 if ftype == 'logits' else 768))
    text = None if ftype == 'logits' else torch.from_numpy(synth.text_embeddings(20)).to(DEV)
    ev = RepeatEvaluator(engine, text, feature_type=ftype, test_repeats=R)
    final = ev.add_scene(points, gt, fused=fused, matrices=mats)
    outs, labels, mious = _solo(engine, ftype, points, gt, fused, mats, text, 20)
    # the batched forward: every repeat's rows give the scores of a solo forward up to split-K summation order
    vox = [voxelize_points(points, M)[:3] for M in mats]
    for r, out in enumerate(ev._forward(vox, None)):
        inv = vox[r][2]
        score = (lambda x: x[inv]) if ftype == 'logits' else \
            (lambda x: matching._scores(x, inv, text, normalize=ftype == 'ensemble')[0])
        s, ref = score(out).float(), score(outs[r]).float()
        assert float((s - ref).abs().max()) < 1e-3 * float(ref.abs().max()) + 1e-3, f'repeat {r}'
    assert (final == labels[-1]).float().mean() >= 0.999
    got = [m[0] for m in ev.results()]
    assert len(got) == R
    assert np.allclose(got, mious, atol=1e-3), (got, mious)
    if ftype == 'logits':
        own = [m[0] for m in ev.repeat_results()]
        assert len(own) == R and all(0.0 <= v <= 1.0 for v in own)
    else:
        with pytest.raises(RuntimeError):
            ev.repeat_results()


def test_repeat_evaluator_fusion_with_mapper_and_no_feature_mask():
    points, gt, fused, mats = _room(seed=5)
    text = torch.from_numpy(synth.text_embeddings(24)).to(DEV)
    mapper = torch.arange(24, device=DEV) % 20                        # several text rows name the same class
    ev = RepeatEvaluator(None, text, feature_type='fusion', test_repeats=R, mapper=mapper, mark_no_feature_to_unknown=True)
    final = ev.add_scene(points, gt, fused=fused, matrices=mats)
    _, labels, mious = _solo(None, 'fusion', points, gt, fused, mats, text, 20, mapper=mapper, nofeat=True)
    assert (final == 256).any() and torch.equal(final, labels[-1])   # no network: the fused path is deterministic
    assert np.allclose([m[0] for m in ev.results()], mious, atol=1e-12)


def test_repeat_evaluator_nuscenes_drops_unlabelled_points():
    from openscene_b200.engine import FusedMinkUNet
    points, gt, fused, mats = _room(seed=9, nuscenes=True)
    engine = FusedMinkUNet(_model(768))
    text = torch.from_numpy(synth.text_embeddings(16)).to(DEV)
    ev = RepeatEvaluator(engine, text, feature_type='ensemble', test_repeats=R, dataset='nuscenes_3d')
    ev.add_scene(points, gt, fused=fused, matrices=mats)
    _, labels, _ = _solo(engine, 'ensemble', points, gt, fused, mats, text, 16)
    keep = gt != 255
    from oracle import metric_ref
    for r, (miou, _, _) in enumerate(ev.results()):                   # the reference evaluates the gt != 255 subset only
        ref, _ = metric_ref.mean_iou(labels[r][keep].cpu().numpy(), gt[keep].cpu().numpy(), 16)
        assert abs(miou - ref) <= 1e-3, r


def test_repeat_evaluator_refuses_bad_arguments():
    points, gt, fused, mats = _room()
    text = torch.from_numpy(synth.text_embeddings(20)).to(DEV)
    ev = RepeatEvaluator(None, text, feature_type='fusion', test_repeats=R)
    with pytest.raises(ValueError, match='matrices'):
        ev.add_scene(points, gt, fused=fused, matrices=mats[:3])
    with pytest.raises(ValueError, match='labels'):
        ev.add_scene(points, gt[:-1], fused=fused, matrices=mats)
    with pytest.raises(ValueError, match='needs fused'):
        ev.add_scene(points, gt, matrices=mats)
    with pytest.raises(ValueError, match='feature_type'):
        RepeatEvaluator(None, text, feature_type='mean')
