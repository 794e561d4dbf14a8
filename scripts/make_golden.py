"""Generate tests/golden/*.npz from a checkout of the reference project (OpenScene), named by OSB_REFERENCE_ROOT.

1. voxelizer_*.npz : outputs of the reference's own ``dataset/voxelizer.py`` (imported unmodified, with the
   ``collections.Sequence/Iterable`` aliases Python 3.12 needs) for seeded inputs + the exact 4x4 matrix it drew.
2. unet_*.npz      : activations of the reference's unmodified ``models/mink_unet.py`` run on the CPU oracle
   (oracle/me_cpu.py registered as ``MinkowskiEngine``) in fp64, seeded weights, eval-mode BN with randomised
   statistics, on a small synthetic room.  These pin the *topology*; the ME arithmetic itself is the oracle's
   (parity unpinned against real MinkowskiEngine -- see oracle/__init__.py).

3. fusion_mapping_*.npz : outputs of the reference's own ``PointCloudToImageMapper.compute_mapping``
   (scripts/feature_fusion/fusion_util.py, imported with a stub ``tensorflow`` the method never touches) for seeded
   points, camera poses and z-buffer depth images.
4. metric_*.npz    : outputs of the reference's ``util/metric.py`` and ``util/util.py`` intersection/union helpers
   (stub ``open3d`` / ``clip`` / ``matplotlib``; ``Tensor.cuda`` patched to the identity -- no GPU here).

5. loader_*.npz    : what the reference's own ``FusedFeatureLoader.__getitem__`` (dataset/feature_loader.py) returns for
   synthetic scene / fused-feature files written to a scratch directory (``SharedArray`` stubbed; ``torch.load`` given
   the ``weights_only=False`` default of the PyTorch the reference targets), plus the 4x4 matrix its voxeliser drew.

6. ref_voxelizer_matrices.npz, ref_voxelizer_random.npz, ref_fusion_random.npz, ref_metric_random.npz : what the
   reference's own ``Voxelizer``, ``PointCloudToImageMapper`` and metric functions return on the seeded random cases of
   tests/test_voxelizer_matrix_vs_reference.py and tests/test_oracles_vs_reference_live.py.
7. ref_models.npz  : the reference's ``models/mink_unet.py`` / ``models/disnet.py`` built on this repository's
   ``MinkowskiEngine`` package: state-dict keys, shapes and a fixed sample of the seeded weights of every architecture
   its factory accepts, plus the names it rejects (tests/test_reference_models_on_product.py).

8. ref_repeats.npz : the reference's own ``run/evaluate.py:evaluate()`` and ``run/eval_mink.py:evaluate()`` with
   ``test_repeats = 3``, run on the CPU over a fake loader / model that yield the seeded inputs of tests/repeats_ref.py
   (``SparseTensor`` and ``Tensor.cuda`` patched to no-ops, ``precompute_text_related_properties`` to the seeded text and
   mapper, ``metric.evaluate`` wrapped to record the labels it is given, the caller's concatenated per-repeat ``pred``
   and the mIoU it returns).

Usage: OSB_REFERENCE_ROOT=<reference checkout> python scripts/make_golden.py [voxelizer] [unet] [fusion] [metric] [loader]
                                                                           [ref_random] [ref_models] [ref_repeats]
(``ref_models`` imports this repository's MinkowskiEngine, ``unet`` the oracle's: run them in separate processes.)
"""
import collections
import collections.abc
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get('OSB_REFERENCE_ROOT', '')
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, 'tests', 'golden')


def golden_voxelizer():
    collections.Sequence = collections.abc.Sequence      # voxelization_utils.py:6
    collections.Iterable = collections.abc.Iterable      # voxelizer.py:55
    sys.path.insert(0, REF)
    from dataset.voxelizer import Voxelizer
    cases = {
        'aug_f64': dict(n=4000, extent=3.0, voxel=0.05, aug=True, dtype=np.float64, seed=1),
        'noaug_f32': dict(n=3000, extent=2.0, voxel=0.05, aug=False, dtype=np.float32, seed=2),
        'dups_f64': dict(n=5000, extent=0.6, voxel=0.05, aug=True, dtype=np.float64, seed=3),
        'neg_f64': dict(n=2000, extent=4.0, voxel=0.02, aug=True, dtype=np.float64, seed=4, shift=-2.0),
    }
    for name, c in cases.items():
        rng = np.random.RandomState(c['seed'])
        pts = (rng.rand(c['n'], 3) * c['extent'] + c.get('shift', 0.0)).astype(c['dtype'])
        vox = Voxelizer(voxel_size=c['voxel'], clip_bound=None, use_augmentation=c['aug'],
                        scale_augmentation_bound=(0.9, 1.1),
                        rotation_augmentation_bound=((-np.pi / 64, np.pi / 64), (-np.pi / 64, np.pi / 64), (-np.pi, np.pi)),
                        translation_augmentation_ratio_bound=((-0.2, 0.2), (-0.2, 0.2), (0, 0)))
        np.random.seed(c['seed'] + 100)
        M_v, M_r = vox.get_transformation_matrix()
        rigid = (M_r @ M_v) if c['aug'] else M_v
        np.random.seed(c['seed'] + 100)          # same draws inside voxelize()
        feats = np.zeros((c['n'], 3), dtype=np.float32)
        labels = np.zeros(c['n'], dtype=np.int64)
        coords_aug, _, _, inds_rec, inds = vox.voxelize(pts, feats, labels, return_ind=True)
        np.savez_compressed(os.path.join(OUT, f'voxelizer_{name}.npz'), points=pts, matrix=rigid,
                            coords_vox=coords_aug, inds=np.asarray(inds), inds_reverse=np.asarray(inds_rec))
        print(name, 'points', c['n'], '-> voxels', len(inds))


def golden_unet():
    from oracle import me_cpu
    me_cpu.install_as_minkowski_engine()
    sys.path.insert(0, REF)
    from models.mink_unet import mink_unet as ref_mink_unet
    from openscene_b200 import synth
    coords = synth.scene('tiny')
    print('tiny scene voxels', len(coords))
    for arch in ('MinkUNet18A', 'MinkUNet34C'):
        torch.manual_seed(0)
        model = ref_mink_unet(in_channels=3, out_channels=768, D=3, arch=arch)
        synth.randomize_bn_stats(model, 1)
        model = model.double().eval()
        rng = np.random.RandomState(7)
        feats = torch.from_numpy(rng.rand(len(coords), 3).astype(np.float32)).double()   # fp32-representable
        with torch.no_grad():
            x = me_cpu.SparseTensor(feats, torch.from_numpy(coords))
            out = model(x)
        out = out.numpy()
        rows = np.sort(np.random.RandomState(11).choice(len(coords), 128, replace=False))
        keys = list(model.state_dict().keys())
        shapes = [tuple(v.shape) for v in model.state_dict().values()]
        np.savez_compressed(os.path.join(OUT, f'unet_{arch}.npz'), coords=coords, feats=feats.numpy().astype(np.float32),
                            rows=rows, out_rows=out[rows].astype(np.float32),
                            row_norm=np.linalg.norm(out, axis=1).astype(np.float32),
                            col_sum=out.sum(0).astype(np.float64),
                            state_keys=np.array(keys), state_shapes=np.array([str(s) for s in shapes]),
                            n_params=np.int64(sum(p.numel() for p in model.parameters())))
        print(arch, 'params', sum(p.numel() for p in model.parameters()), 'out', out.shape, 'abs mean', np.abs(out).mean())


def _stub_modules(*names):
    import types
    for nm in names:
        parts = nm.split('.')
        for i in range(1, len(parts) + 1):
            sub = '.'.join(parts[:i])
            if sub not in sys.modules:
                sys.modules[sub] = types.ModuleType(sub)
            if i > 1:
                setattr(sys.modules['.'.join(parts[:i - 1])], parts[i - 1], sys.modules[sub])


def golden_fusion():
    _stub_modules('tensorflow', 'tensorflow.io', 'tensorflow.compat', 'tensorflow.compat.v1')
    sys.path.insert(0, os.path.join(REF, 'scripts', 'feature_fusion'))
    from fusion_util import PointCloudToImageMapper, adjust_intrinsic, make_intrinsic
    from openscene_b200.synth import fusion_case
    # the intrinsics helpers with the ScanNet / Matterport-style numbers the fusion scripts use (scannet_openseg.py:124-160)
    k0 = make_intrinsic(fx=577.870605, fy=577.870605, mx=319.5, my=239.5)
    k1 = adjust_intrinsic(k0.copy(), intrinsic_image_dim=[640, 480], image_dim=(320, 240))
    k2 = adjust_intrinsic(make_intrinsic(1075.1, 1075.8, 629.7, 522.3), intrinsic_image_dim=[1280, 1024], image_dim=(640, 512))
    np.savez_compressed(os.path.join(OUT, 'fusion_intrinsics.npz'), k0=k0, k1=k1, k2=k2)
    cases = {'depth_cut10': dict(seed=21, n=6000, with_depth=True, cut=10),
             'depth_cut0': dict(seed=22, n=5000, with_depth=True, cut=0),
             'nodepth_cut5': dict(seed=23, n=5000, with_depth=False, cut=5)}
    for name, c in cases.items():
        pts, poses, depths, intr = fusion_case(c['seed'], c['n'], c['with_depth'])
        mapper = PointCloudToImageMapper(image_dim=(320, 240), intrinsics=intr, visibility_threshold=0.25, cut_bound=c['cut'])
        maps = np.stack([mapper.compute_mapping(p, pts, d) for p, d in zip(poses, depths)])
        np.savez_compressed(os.path.join(OUT, f'fusion_mapping_{name}.npz'), seed=c['seed'], n=c['n'], with_depth=c['with_depth'],
                            cut=c['cut'], mapping=maps.astype(np.int32))
        print('fusion', name, 'visible per frame', maps[:, :, 2].sum(1))


def golden_metric():
    _stub_modules('open3d', 'clip', 'matplotlib', 'matplotlib.patches', 'matplotlib.pyplot')
    sys.path.insert(0, REF)
    from util import metric as ref_metric
    from util import util as ref_util
    from dataset import label_constants as lc
    # class counts evaluate() derives from the dataset name (util/metric.py:47-60)
    np.savez_compressed(os.path.join(OUT, 'metric_class_counts.npz'), names=np.array(['scannet_3d', 'matterport_3d_40', 'matterport_3d_80',
                        'matterport_3d_160', 'matterport_3d', 'nuscenes_3d']),
                        counts=np.array([len(lc.SCANNET_LABELS_20), len(lc.MATTERPORT_LABELS_40), len(lc.MATTERPORT_LABELS_80),
                                         len(lc.MATTERPORT_LABELS_160), len(lc.MATTERPORT_LABELS_21), len(lc.NUSCENES_LABELS_16)]))
    orig_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        for name, (C, ds, seed, nofeat) in {'scannet20': (20, 'scannet_3d', 31, False), 'mp160_nofeat': (160, 'matterport_3d_160', 32, True),
                                            'nuscenes16': (16, 'nuscenes_3d', 33, False)}.items():
            rng = np.random.RandomState(seed)
            n = 50000
            gt = rng.randint(0, C, n)
            gt[rng.rand(n) < 0.1] = 255
            gt[gt == 3] = 5                                      # a class that never occurs in gt
            pred = np.where(rng.rand(n) < 0.6, np.minimum(gt, C - 1), rng.randint(0, C, n))
            if nofeat:
                pred[rng.rand(n) < 0.05] = 256
            conf = ref_metric.confusion_matrix(pred.copy(), gt.copy(), C)
            miou = ref_metric.evaluate(pred.copy(), gt.copy(), stdout=False, dataset=ds)
            out = dict(pred=pred.astype(np.int32), gt=gt.astype(np.int32), C=C, confusion=conf.astype(np.int64), miou=np.float64(miou))
            if not nofeat:
                i_np, u_np, t_np = ref_util.intersectionAndUnion(pred.copy(), gt.copy(), C, 255)
                i_t, u_t, t_t = ref_util.intersectionAndUnionGPU(torch.from_numpy(pred.copy()), torch.from_numpy(gt.copy()), C, 255)
                assert np.array_equal(i_np, i_t.numpy()) and np.array_equal(u_np, u_t.numpy()) and np.array_equal(t_np, t_t.numpy())
                out.update(inter=i_np.astype(np.int64), union=u_np.astype(np.int64), target=t_np.astype(np.int64))
            np.savez_compressed(os.path.join(OUT, f'metric_{name}.npz'), **out)
            print('metric', name, 'mIoU', miou)
    finally:
        torch.Tensor.cuda = orig_cuda


def golden_loader():
    import functools
    import shutil
    import tempfile
    collections.Sequence = collections.abc.Sequence
    collections.Iterable = collections.abc.Iterable
    _stub_modules('SharedArray')
    sys.path.insert(0, REF)
    from dataset.feature_loader import FusedFeatureLoader
    orig_load = torch.load
    torch.load = functools.partial(orig_load, weights_only=False)
    tmp = tempfile.mkdtemp(prefix='osb_golden_')
    try:
        cases = {'train': dict(split='train', seed=51, legacy=False), 'val': dict(split='val', seed=52, legacy=False),
                 'train_legacy': dict(split='train', seed=53, legacy=True)}
        for name, c in cases.items():
            rng = np.random.RandomState(c['seed'])
            n, C = 3000, 16
            locs = (rng.rand(n, 3) * np.array([1.2, 1.0, 0.8])).astype(np.float32)
            colors = (rng.rand(n, 3) * 2 - 1).astype(np.float32)
            labels = rng.randint(0, 20, n).astype(np.float64)
            labels[rng.rand(n) < 0.1] = -100
            root = os.path.join(tmp, name, 'scannet_3d')
            os.makedirs(os.path.join(root, c['split']))
            featdir = os.path.join(tmp, name, 'feat')
            os.makedirs(featdir)
            torch.save((locs, colors, labels), os.path.join(root, c['split'], 'scene0000_00_vh_clean_2.pth'))
            mask_full = torch.from_numpy(rng.rand(n) < 0.4)
            M = int(mask_full.sum())
            feat = torch.from_numpy(rng.randn(M, C).astype(np.float16))
            blob = {'feat': feat, 'mask_full': mask_full}
            legacy_mask = None
            if c['legacy']:
                legacy_mask = torch.from_numpy(rng.rand(M) < 0.7)
                blob = {'feat': feat, 'mask': legacy_mask.nonzero()[:, 0], 'mask_full': mask_full}
            torch.save(blob, os.path.join(featdir, 'scene0000_00_0.pt'))
            loader = FusedFeatureLoader(datapath_prefix=root, datapath_prefix_feat=featdir, voxel_size=0.05, split=c['split'],
                                        aug=False, memcache_init=False, eval_all=(c['split'] != 'train'), input_color=False)
            np.random.seed(c['seed'] + 100)
            M_v, M_r = loader.voxelizer.get_transformation_matrix()
            np.random.seed(c['seed'] + 100)                       # same draws inside __getitem__ -> voxelize()
            item = loader[0]
            coords, feats, lab, feat_3d, mask = item[:5]
            out = dict(locs=locs, labels_in=labels, mask_full=mask_full.numpy(), feat=feat.numpy(), matrix=M_r @ M_v,
                       coords=coords.numpy(), feats=feats.numpy(), labels=lab.numpy(), feat_3d=feat_3d.numpy(), mask=mask.numpy(),
                       split=c['split'])
            if legacy_mask is not None:
                out['legacy_mask'] = legacy_mask.numpy()
            if len(item) > 5:
                out['inds_reverse'] = item[5].numpy()
            np.savez_compressed(os.path.join(OUT, f'loader_{name}.npz'), **out)
            print('loader', name, 'voxels', coords.shape[0], 'feat rows', feat_3d.shape[0], 'mask true', int(mask.sum()))
    finally:
        torch.load = orig_load
        shutil.rmtree(tmp, ignore_errors=True)


def golden_ref_random():
    """The reference's Voxelizer, PointCloudToImageMapper and metric functions on the random cases of the tests."""
    from tests import test_oracles_vs_reference_live as to
    from tests import test_voxelizer_matrix_vs_reference as tv
    collections.Sequence = collections.abc.Sequence
    collections.Iterable = collections.abc.Iterable
    _stub_modules('tensorflow', 'tensorflow.io', 'tensorflow.compat', 'tensorflow.compat.v1',
                  'open3d', 'clip', 'matplotlib', 'matplotlib.patches', 'matplotlib.pyplot')
    sys.path.insert(0, REF)
    sys.path.insert(0, os.path.join(REF, 'scripts', 'feature_fusion'))
    from dataset.voxelizer import Voxelizer
    from fusion_util import PointCloudToImageMapper
    from util import metric as ref_metric
    from util import util as ref_util

    shape = (len(tv.FORMS), len(tv.MATRIX_SEEDS))
    m_v, m_r, tail = np.zeros(shape + (4, 4)), np.zeros(shape + (4, 4)), np.zeros(shape + (4,))
    for form in range(len(tv.FORMS)):
        vox = Voxelizer(**tv.form_kwargs(form))
        for seed in tv.MATRIX_SEEDS:
            np.random.seed(seed)
            m_v[form, seed], m_r[form, seed] = vox.get_transformation_matrix()
            tail[form, seed] = np.random.rand(4)
    np.savez_compressed(os.path.join(OUT, 'ref_voxelizer_matrices.npz'), m_v=m_v, m_r=m_r, tail=tail)

    out = {}
    for trial, pts, aug, vsize in tv.random_clouds():
        n = len(pts)
        vox = Voxelizer(voxel_size=vsize, clip_bound=None, use_augmentation=aug, scale_augmentation_bound=(0.9, 1.1),
                        rotation_augmentation_bound=tv.ROT, translation_augmentation_ratio_bound=((-0.2, 0.2), (-0.2, 0.2), (0, 0)))
        np.random.seed(trial)
        M_v, M_r = vox.get_transformation_matrix()
        np.random.seed(trial)                                     # same draws inside voxelize()
        coords_aug, _, _, inds_rec, inds = vox.voxelize(pts, np.zeros((n, 3), np.float32), np.zeros(n, np.int64), return_ind=True)
        out.update({f'matrix_{trial}': (M_r @ M_v) if aug else M_v, f'coords_{trial}': coords_aug,
                    f'inds_{trial}': np.asarray(inds), f'inds_reverse_{trial}': np.asarray(inds_rec)})
    np.savez_compressed(os.path.join(OUT, 'ref_voxelizer_random.npz'), **out)

    out = {}
    for seed, pts, poses, depths, intr, cut, thres in to.fusion_cases():
        mapper = PointCloudToImageMapper(image_dim=(320, 240), intrinsics=intr, visibility_threshold=thres, cut_bound=cut)
        maps = np.stack([mapper.compute_mapping(p, pts, d) for p, d in zip(poses, depths)])
        assert maps.min() >= 0 and maps.max() < 1 << 15
        out[f'mapping_{seed}'] = maps.astype(np.int16)
    np.savez_compressed(os.path.join(OUT, 'ref_fusion_random.npz'), **out)

    out = {}
    orig_cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self           # intersectionAndUnionGPU calls .cuda()
    try:
        for seed, C, ds, pred, gt, nofeat in to.metric_cases():
            out[f'confusion_{seed}'] = ref_metric.confusion_matrix(pred.copy(), gt.copy(), C).astype(np.int64)
            out[f'miou_{seed}'] = np.float64(ref_metric.evaluate(pred.copy(), gt.copy(), stdout=False, dataset=ds))
            if not nofeat:
                i_np, u_np, t_np = ref_util.intersectionAndUnion(pred.copy(), gt.copy(), C, 255)
                i_t, u_t, t_t = ref_util.intersectionAndUnionGPU(torch.from_numpy(pred.copy()), torch.from_numpy(gt.copy()), C, 255)
                for name, a, b in (('inter', i_np, i_t), ('union', u_np, u_t), ('target', t_np, t_t)):
                    assert np.array_equal(a.astype(np.int64), b.numpy().astype(np.int64))
                    out[f'{name}_{seed}'] = a.astype(np.int64)
    finally:
        torch.Tensor.cuda = orig_cuda
    np.savez_compressed(os.path.join(OUT, 'ref_metric_random.npz'), **out)
    print('ref_random written')


def golden_ref_models():
    """The reference's model files on this repository's MinkowskiEngine package: keys, shapes, sampled seeded weights."""
    import importlib
    import types
    from tests import test_reference_models_on_product as tm
    for name in [m for m in sys.modules if m.split('.')[0] in ('MinkowskiEngine', 'models')]:
        del sys.modules[name]
    import MinkowskiEngine as ME
    assert ME.MinkowskiConvolution.__module__.startswith('openscene_b200')
    sys.path.insert(0, REF)
    mu = importlib.import_module('models.mink_unet')
    dn = importlib.import_module('models.disnet')
    assert os.path.realpath(mu.__file__).startswith(os.path.realpath(REF))
    out = {}

    def record(tag, model):
        sd = model.state_dict()
        out[f'{tag}_keys'] = np.array(list(sd.keys()))
        out[f'{tag}_shapes'] = np.array([str(tuple(v.shape)) for v in sd.values()])
        out[f'{tag}_sample'], out[f'{tag}_sums'] = tm.weight_sample(sd)

    for arch in ('MinkUNet18A', 'MinkUNet34C'):
        torch.manual_seed(0)
        record(arch, mu.mink_unet(in_channels=3, out_channels=768, D=3, arch=arch))
    for arch in tm.OTHER_ARCHS:
        torch.manual_seed(0)
        record(f'{arch}_20', mu.mink_unet(in_channels=3, out_channels=20, D=3, arch=arch))
    for ext in ('openseg', 'lseg'):
        torch.manual_seed(0)
        record(f'DisNet_{ext}', dn.DisNet(cfg=types.SimpleNamespace(arch_3d='MinkUNet18A', feature_2d_extractor=ext)))
    for arch in tm.REJECTED:
        try:
            mu.mink_unet(arch=arch)
        except Exception:
            continue
        raise AssertionError(f'the reference accepts {arch}')
    try:
        mu.MinkUNet50(3, 20, 3)
        raise AssertionError('the reference constructs MinkUNet50')
    except TypeError:                                         # PLANES is None: self.PLANES[0] fails in network_initialization
        pass
    out['rejected'] = np.array(tm.REJECTED)
    np.savez_compressed(os.path.join(OUT, 'ref_models.npz'), **out)
    print('ref_models written')


def golden_ref_repeats():
    """The reference's test_repeats loops on seeded inputs (tests/repeats_ref.py)."""
    import importlib
    import logging
    import shutil
    import tempfile
    import types
    from tests import repeats_ref as rr
    collections.Sequence = collections.abc.Sequence
    collections.Iterable = collections.abc.Iterable
    _stub_modules('open3d', 'clip', 'matplotlib', 'matplotlib.patches', 'matplotlib.pyplot', 'tensorboardX', 'SharedArray')
    sys.modules['tensorboardX'].SummaryWriter = object
    sys.path.insert(0, REF)
    ev = importlib.import_module('run.evaluate')
    em = importlib.import_module('run.eval_mink')
    from util import metric as ref_metric
    assert os.path.realpath(ev.__file__).startswith(os.path.realpath(REF))
    orig_cuda, orig_eval = torch.Tensor.cuda, ref_metric.evaluate
    torch.Tensor.cuda = lambda self, *a, **k: self
    calls = []

    def recording_evaluate(pred_ids, gt_ids, stdout=False, dataset='scannet_3d'):
        miou = orig_eval(pred_ids.copy(), gt_ids.copy(), stdout=False, dataset=dataset)
        calls.append((np.asarray(pred_ids).copy(), sys._getframe(1).f_locals['pred'].clone(), miou, np.asarray(gt_ids).copy()))
        return miou

    ref_metric.evaluate = recording_evaluate
    out = {}
    tmp = tempfile.mkdtemp(prefix='osb_golden_')
    try:
        for name, (ftype, ds, k, c, n_scenes, R, nofeat, _) in sorted(rr.CASES.items()):
            state = {}

            class Loader:                                   # what the DataLoader yields: one scene per batch
                dataset = types.SimpleNamespace(offset=0)      # evaluate.py sets it to the repeat; eval_mink.py does not
                passes = 0

                def __iter__(self):
                    rep = self.passes
                    self.passes += 1
                    assert ftype == 'logits' or rep == self.dataset.offset
                    for sc in range(n_scenes):
                        state['key'] = (sc, rep)
                        item = rr.scene_inputs(name, sc, rep)
                        yield item if ftype != 'logits' else (item[0], item[1], item[2], item[5])

                def __len__(self):
                    return n_scenes

            class Model(torch.nn.Module):                   # seeded voxel features for the scene / repeat being loaded
                def forward(self, _sinput):
                    sc, rep = state['key']
                    return rr.voxel_features(name, sc, rep, len(rr.scene_inputs(name, sc, rep)[0]))

            model = Model()

            args = types.SimpleNamespace(test_repeats=R, feature_type=ftype, save_folder=tmp, model_path=tmp,
                                         save_feature_as_numpy=False, mark_no_feature_to_unknown=nofeat, vis_input=False,
                                         vis_pred=False, vis_gt=False, eval_iou=True, multiprocessing_distributed=False,
                                         data_root=os.path.join(tmp, ds))
            text, mapper = rr.text_and_mapper(name)
            calls.clear()
            if ftype == 'logits':
                em.args, em.SparseTensor = args, (lambda f, c: None)
                em.evaluate(model, Loader())
                own, acc = calls[0::2], calls[1::2]
                out[f'{name}_own_labels'] = np.stack([c_[0] for c_ in own])
                out[f'{name}_own_miou'] = np.array([c_[2] for c_ in own])
            else:
                ev.args, ev.SparseTensor, ev.logger = args, (lambda f, c: None), logging.getLogger('osb_golden')
                ev.precompute_text_related_properties = lambda _ls: (text, ['c%d' % i for i in range(k)], mapper, None)
                ev.evaluate(model, Loader(), ds)
                acc = calls
            assert len(acc) == R
            out[f'{name}_seed'] = np.int64(rr.case_seed(name))
            out[f'{name}_gt'] = acc[0][3]
            out[f'{name}_labels'] = np.stack([c_[0] for c_ in acc])
            out[f'{name}_miou'] = np.array([c_[2] for c_ in acc])
            out[f'{name}_pred'] = np.stack([c_[1].numpy() for c_ in acc])
            print('ref_repeats', name, 'mIoU per prefix', out[f'{name}_miou'])
    finally:
        torch.Tensor.cuda, ref_metric.evaluate = orig_cuda, orig_eval
        shutil.rmtree(tmp, ignore_errors=True)
    np.savez_compressed(os.path.join(OUT, 'ref_repeats.npz'), **out)
    print('ref_repeats written')


if __name__ == '__main__':
    if not os.path.isdir(REF):
        sys.exit('set OSB_REFERENCE_ROOT to a checkout of the reference project')
    os.makedirs(OUT, exist_ok=True)
    todo = sys.argv[1:] or ['voxelizer', 'unet', 'fusion', 'metric', 'loader', 'ref_random']
    for nm in todo:
        {'voxelizer': golden_voxelizer, 'unet': golden_unet, 'fusion': golden_fusion, 'metric': golden_metric, 'loader': golden_loader,
         'ref_random': golden_ref_random, 'ref_models': golden_ref_models, 'ref_repeats': golden_ref_repeats}[nm]()
