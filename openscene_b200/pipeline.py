"""One entry point for the whole hot path: points -> voxels -> MinkUNet -> open-vocabulary labels, all on the device.

Mirrors the inner loop of ``run/evaluate.py:283-323`` (feature types 'distill' and 'ensemble') for callers that hold raw
points instead of a pre-voxelised batch:

    seg = OpenVocabSegmenter(model, text_features, voxel_size=0.02)
    labels = seg.segment_points(points_xyz)                      # int64 [N_pts]; nothing but the labels leaves the GPU

* ``dataset/voxelizer.py:97-140`` (``Voxelizer.voxelize``: affine, floor, FNV key, first-occurrence unique) runs in
  csrc/voxelize.cu and hands ``inds_reverse`` straight to the matcher -- the voxel->point expansion
  ``predictions[inds_reverse]`` (evaluate.py:290) is fused into the matching kernel's operand load;
* when the caller does not ask for the 768-d features, the final 1x1x1 convolution is re-associated with the text matrix
  (``engine.fold_head``: W W^T = L L^T, U = W T^T) so the [N, 768] feature matrix is never written or read back.
"""
import numpy as np
import torch

from . import _cabi as C
from . import engine as _engine
from . import matching
from .voxelize import voxelize_points


class OpenVocabSegmenter:
    def __init__(self, model, text_features, voxel_size=0.02, normalize=True):
        """model: eval-mode MinkUNet / DisNet on a CUDA device (or a ready ``FusedMinkUNet``); text_features: unit-norm
        [K, C] CLIP text embeddings (util/util.py:24-46).  normalize=True gives cosine scores (the 'ensemble' branch's
        ``x / (|x| + 1e-5)``, evaluate.py:305-310); False the plain dot product of the 'distill' branch (:291)."""
        self.engine = model if isinstance(model, _engine.FusedMinkUNet) else _engine.FusedMinkUNet(model)
        self.device = self.engine.device
        self.text = text_features.to(self.device, torch.float16).contiguous()
        self.voxel_size = voxel_size
        self.normalize = normalize
        self._folded = None
        self._matrix = np.eye(4)
        np.fill_diagonal(self._matrix[:3, :3], 1.0 / voxel_size)

    def _fold(self):
        if self._folded is None or self._folded[3] != self.engine._signature():      # first use, or the model's weights changed
            self._folded = self.engine.fold_head(self.text.float())
        return self._folded

    @torch.no_grad()
    def segment_voxels(self, coords, feats, inds_reverse=None, want_features=False, want_scores=False):
        """coords int32 [Nv,4] (batch,x,y,z), feats fp32 [Nv,3].  Returns (labels int64 [Np], scores fp16 [Np,K] | None,
        features fp32 [Nv,C] | None) with Np = len(inds_reverse) (or Nv)."""
        if not want_features and self.normalize:
            scores, label, _ = self.engine.forward_scores(coords, feats, self._fold(), want_scores=want_scores)
            if inds_reverse is not None:                      # per-voxel results -> per-point (a [Np] / [Np,K] gather)
                inds_reverse = inds_reverse.to(label.device)
                label = label[inds_reverse]
                scores = scores[inds_reverse] if scores is not None else None
            return label, scores, None
        out = self.engine(coords, feats)
        scores, label, _ = matching._scores(out, inds_reverse, self.text, normalize=self.normalize, want_scores=want_scores)
        return label, scores, (out if want_features else None)

    @torch.no_grad()
    def segment_points(self, points, feats=None, matrix=None, want_scores=False):
        """points: CUDA float [N,3] (metres).  feats: per-POINT input features fp32 [N,3] or None (ones, the reference's
        default when ``input_color`` is off, dataset/feature_loader.py:180-184).  Returns int64 labels [N] (and fp16 scores
        [N,K] when asked): every point takes the label of its voxel, exactly ``pred[inds_reverse]`` of the reference."""
        C.require_cuda(points, 'points')
        with torch.cuda.device(self.device):
            cv, inds, inv, _ = voxelize_points(points, self._matrix if matrix is None else matrix)
            n_vox = cv.shape[0]
            coords = torch.zeros((n_vox, 4), dtype=torch.int32, device=self.device)       # batch index 0
            coords[:, 1:] = cv
            f = torch.ones((n_vox, 3), dtype=torch.float32, device=self.device) if feats is None else feats[inds].float()
            label, scores, _ = self.segment_voxels(coords, f, inv, want_features=False, want_scores=want_scores)
        return (label, scores) if want_scores else label


# dataset/point_loader.py:58-61: the bounds of the voxeliser every OpenScene loader builds with use_augmentation=True (:93-99)
LOADER_SCALE_BOUND = (0.9, 1.1)
LOADER_ROTATION_BOUND = ((-np.pi / 64, np.pi / 64), (-np.pi / 64, np.pi / 64), (-np.pi, np.pi))
LOADER_TRANSLATION_BOUND = ((-0.2, 0.2), (-0.2, 0.2), (0, 0))


class RepeatEvaluator:
    """OpenScene's evaluation protocol with ``test_repeats`` (run/evaluate.py:259-425, run/eval_mink.py:159-216) on the
    device, one scene at a time:

        ev = RepeatEvaluator(model, text_features, feature_type='ensemble', test_repeats=5)
        for points, gt, feat, mask_full in scenes:
            ev.add_scene(points, gt, fused=(feat, mask_full))
        ev.results()            # [(mIoU, mAcc, class ious)] after repeats 1..R (the reference's accumu_iou)

    Per scene: R voxelisations (random rotation and scale as the point loader draws them, or the caller's ``matrices``),
    the fused 2-D features remapped per voxelisation, ONE network forward over the R voxel sets as batch indices
    0..R-1, and per repeat the matching of ``feature_type`` folded into a device-resident fp16 score sum
    (``matching.match_accumulate``: ``store = pred + store`` with the reference's fp16 rounding).  After repeat r the
    labels ``argmax(store)`` (mapped by ``mapper``; 256 where repeat r's voxel has no fused feature when
    ``mark_no_feature_to_unknown`` is set for 'fusion', exactly as the reference rebuilds that mask every repeat) update
    confusion matrix r.  Nothing of size N_pts x K leaves the device.

    feature_type 'logits' is run/eval_mink.py: the model returns class logits, the accumulation is fp32
    (``matching.logits_accumulate``) and ``repeat_results()`` also gives each repeat's own score (its ``current_iou``).

    Matrices: when ``matrices`` is not given, R are drawn per scene with ``Voxelizer.get_transformation_matrix()`` from
    NumPy's global RNG.  The reference's DataLoader workers draw from their own RNG streams, so the results equal the
    reference's given the same matrices, not the same seed.  nuScenes: points with gt 255 are left out by the confusion
    matrix's ignore id, which gives the reference's result of dropping them (evaluate.py:335-339)."""

    FEATURE_TYPES = ('distill', 'fusion', 'ensemble', 'logits')

    def __init__(self, model, text_features, feature_type='ensemble', test_repeats=5, voxel_size=0.02, dataset='scannet_3d',
                 mapper=None, mark_no_feature_to_unknown=False, device=None):
        from .metric import _DATASET_CLASSES, ConfusionMeter
        from .voxelize import Voxelizer
        if feature_type not in self.FEATURE_TYPES:
            raise ValueError(f"RepeatEvaluator: feature_type {feature_type!r} not in {self.FEATURE_TYPES}")
        if int(test_repeats) < 1:
            raise ValueError(f"RepeatEvaluator: test_repeats must be >= 1, got {test_repeats}")
        n_classes = next((n for key, n in _DATASET_CLASSES if key in dataset), None)
        if n_classes is None:
            raise ValueError(f"RepeatEvaluator: unknown dataset {dataset!r}")
        self.feature_type = feature_type
        self.R = int(test_repeats)
        if feature_type == 'fusion':
            self.engine = None
            self.device = torch.device(device or 'cuda')
        else:
            self.engine = model if isinstance(model, _engine.FusedMinkUNet) else _engine.FusedMinkUNet(model)
            self.device = self.engine.device
        self.text = None if feature_type == 'logits' else text_features.to(self.device, torch.float16).contiguous()
        self.mapper = None if mapper is None else torch.as_tensor(mapper).to(self.device).long()
        self.mark_no_feature = bool(mark_no_feature_to_unknown) and feature_type == 'fusion'   # evaluate.py:245-248
        self.voxelizer = Voxelizer(voxel_size=voxel_size, use_augmentation=True, scale_augmentation_bound=LOADER_SCALE_BOUND,
                                   rotation_augmentation_bound=LOADER_ROTATION_BOUND,
                                   translation_augmentation_ratio_bound=LOADER_TRANSLATION_BOUND)
        self.meters = [ConfusionMeter(n_classes, self.device) for _ in range(self.R)]
        self.own_meters = [ConfusionMeter(n_classes, self.device) for _ in range(self.R)] if feature_type == 'logits' else None

    def draw_matrices(self):
        """R voxelisation matrices ``M_r @ M_v`` from NumPy's global RNG, in the order the voxeliser draws them."""
        out = []
        for _ in range(self.R):
            M_v, M_r = self.voxelizer.get_transformation_matrix()
            out.append(M_r @ M_v)
        return out

    @torch.no_grad()
    def add_scene(self, points, gt_labels, fused=None, colors=None, matrices=None):
        """points: CUDA float [N,3]; gt_labels int [N] (255 = ignored); fused = (feat [M,C] fp16, mask_full bool [N]) as
        the fusion scripts store them, required by 'fusion' / 'ensemble'; colors: per-point input features [N,3] in
        [-1, 1] or None (ones, the loaders' default without ``input_color``); matrices: R host 4x4 matrices or None.
        Returns the int64 labels [N] after the last repeat (mapped and masked as they enter the metric), on the device."""
        from .fused_features import remap_fused_features
        C.require_cuda(points, 'points')
        if self.feature_type in ('fusion', 'ensemble') and fused is None:
            raise ValueError(f"RepeatEvaluator: feature_type {self.feature_type!r} needs fused=(feat, mask_full)")
        mats = self.draw_matrices() if matrices is None else list(matrices)
        if len(mats) != self.R:
            raise ValueError(f"RepeatEvaluator: {len(mats)} matrices for test_repeats={self.R}")
        dev = self.device
        n_pts = points.shape[0]
        gt = torch.as_tensor(gt_labels).to(dev).long().view(-1)
        if gt.numel() != n_pts:
            raise ValueError(f"RepeatEvaluator: {gt.numel()} labels for {n_pts} points")
        with torch.cuda.device(dev):
            vox = [voxelize_points(points, M)[:3] for M in mats]                   # (coords int32 [nv,3], inds, inds_reverse)
            fvox = [remap_fused_features(fused[0], fused[1], inds, split='val', device=dev) for _, inds, _ in vox] \
                if self.feature_type in ('fusion', 'ensemble') else None
            outs = self._forward(vox, colors) if self.engine is not None else None
            store = None
            for r in range(self.R):
                inv = vox[r][2]
                first = r == 0
                if self.feature_type == 'logits':
                    if store is None:
                        store = torch.empty((n_pts, outs[r].shape[1]), dtype=torch.float32, device=dev)
                    own, label = matching.logits_accumulate(outs[r], inv, store, first)
                    self.own_meters[r].update(self._map(own), gt)
                else:
                    if store is None:
                        store = torch.empty((n_pts, self.text.shape[0]), dtype=torch.float16, device=dev)
                    label = self._match(outs[r] if outs is not None else None, fvox[r][0] if fvox is not None else None,
                                        inv, store, first)
                label = self._map(label)
                if self.mark_no_feature:
                    label[~fvox[r][1][inv]] = 256                               # repeat r's own voxel mask (evaluate.py:405-421)
                self.meters[r].update(label, gt)
        return label

    def _map(self, label):
        return self.mapper[label] if self.mapper is not None else label

    def _forward(self, vox, colors):
        """One forward over the R voxel sets as batch indices 0..R-1; repeat r's features are rows [off_r, off_r + nv_r)."""
        nv = [cv.shape[0] for cv, _, _ in vox]
        coords = torch.empty((sum(nv), 4), dtype=torch.int32, device=self.device)
        feats = torch.ones((sum(nv), 3), dtype=torch.float32, device=self.device)
        off = 0
        for r, (cv, inds, _) in enumerate(vox):
            coords[off:off + nv[r], 0] = r
            coords[off:off + nv[r], 1:] = cv
            if colors is not None:
                feats[off:off + nv[r]] = colors.to(self.device)[inds].float()
            off += nv[r]
        out = self.engine(coords, feats)
        return list(torch.split(out, nv))

    def _match(self, out, feat2d, inv, store, first):
        text = self.text
        if self.feature_type == 'distill':                                   # evaluate.py:288-292
            return matching.match_accumulate(out, inv, text, store, first)
        if self.feature_type == 'fusion':                                    # :293-296
            return matching.match_accumulate(feat2d, inv, text, store, first)
        feat2d = feat2d.half()                                               # ensemble, :302-323
        _, _, smax2d = matching._scores(feat2d, inv, text, normalize=True, want_scores=False, want_smax=True)
        _, _, smax3d = matching._scores(out, inv, text, normalize=True, want_scores=False, want_smax=True)
        return matching.match_accumulate(out, inv, text, store, first, feat2=feat2d, smax3d=smax3d, smax2d=smax2d)

    def results(self):
        """R entries: (mean IoU, mean accuracy, {class: (iou, tp, denom)}) of the accumulated scores after repeats 1..r,
        the reference's ``accumu_iou`` (util/metric.py conventions).  SYNC."""
        return [m.evaluate() for m in self.meters]

    def repeat_results(self):
        """'logits' only: each repeat's own result (run/eval_mink.py:205 ``current_iou``).  SYNC."""
        if self.own_meters is None:
            raise RuntimeError("RepeatEvaluator.repeat_results: only feature_type 'logits' reports each repeat's own score")
        return [m.evaluate() for m in self.own_meters]
