"""Open-vocabulary matching on libosb200 (csrc/match.cu): the three ``feature_type`` branches of
``run/evaluate.py:288-323`` with the same arguments and results (fp16 scores [N_pts, K], int64 labels),
computed in one pass per product without materialising ``predictions[inds_reverse]``."""
import torch

from . import _cabi as C


def _scores(feat, inds_reverse, text, normalize, want_scores=True, want_smax=False):
    C.require_cuda(feat, 'features')
    feat = feat.contiguous()
    text = text.to(device=feat.device, dtype=torch.float16).contiguous()
    is_f16 = feat.dtype == torch.float16
    if not is_f16 and feat.dtype != torch.float32:
        feat = feat.float()
    n_vox, c = feat.shape
    k = text.shape[0]
    assert text.shape[1] == c, f"text embeddings have width {text.shape[1]}, features {c}"
    if inds_reverse is not None:
        inds_reverse = inds_reverse.to(device=feat.device, dtype=torch.int64).contiguous()
        n_pts = inds_reverse.shape[0]
    else:
        n_pts = n_vox
    with torch.cuda.device(feat.device):
        scores = torch.empty((n_pts, k), dtype=torch.float16, device=feat.device) if want_scores else None
        label = torch.empty(n_pts, dtype=torch.int64, device=feat.device)
        smax = torch.empty(n_pts, dtype=torch.float32, device=feat.device) if want_smax else None
        C.call('osb_match_scores', C.ptr(feat), int(is_f16), n_vox, c, C.ptr(inds_reverse), n_pts, C.ptr(text), k,
               int(normalize), C.ptr(scores), C.ptr(label), C.ptr(smax), C.stream_ptr())
    return scores, label, smax


def match_distill(predictions, inds_reverse, text_features):
    """evaluate.py:288-292: ``pred = predictions[inds_reverse].half() @ text.t(); label = argmax``."""
    s, l, _ = _scores(predictions, inds_reverse, text_features, normalize=False)
    return s, l


def match_fusion(feat_3d, inds_reverse, text_features):
    """evaluate.py:293-296 (fused 2-D features, fp16)."""
    s, l, _ = _scores(feat_3d, inds_reverse, text_features, normalize=False)
    return s, l


def match_ensemble(predictions, feat_3d, inds_reverse, text_features, return_features=False):
    """evaluate.py:302-323: cosine scores of both feature sets, per-point winner, final product.

    Returns (pred fp16 [N_pts,K], label int64 [N_pts], feat_ensemble fp16 [N_pts,C] or None, mask bool)."""
    feat_3d = feat_3d.to(predictions.device)
    if feat_3d.dtype != torch.float16:
        feat_3d = feat_3d.half()
    _, _, smax2d = _scores(feat_3d, inds_reverse, text_features, normalize=True, want_scores=False, want_smax=True)
    _, _, smax3d = _scores(predictions, inds_reverse, text_features, normalize=True, want_scores=False, want_smax=True)
    predictions = predictions.contiguous().float()
    feat_3d = feat_3d.contiguous()
    text = text_features.to(device=predictions.device, dtype=torch.float16).contiguous()
    n_vox, c = predictions.shape
    inv = inds_reverse.to(device=predictions.device, dtype=torch.int64).contiguous() if inds_reverse is not None else None
    n_pts = inv.shape[0] if inv is not None else n_vox
    k = text.shape[0]
    with torch.cuda.device(predictions.device):
        scores = torch.empty((n_pts, k), dtype=torch.float16, device=predictions.device)
        label = torch.empty(n_pts, dtype=torch.int64, device=predictions.device)
        fe = torch.empty((n_pts, c), dtype=torch.float16, device=predictions.device) if return_features else None
        C.call('osb_match_ensemble', C.ptr(predictions), C.ptr(feat_3d), n_vox, c, C.ptr(inv), n_pts, C.ptr(smax3d),
               C.ptr(smax2d), C.ptr(text), k, C.ptr(scores), C.ptr(label), C.ptr(fe), C.stream_ptr())
    return scores, label, fe, smax3d < smax2d


def _inds(inds_reverse, device, n_vox):
    if inds_reverse is None:
        return None, n_vox
    inv = inds_reverse.to(device=device, dtype=torch.int64).contiguous()
    return inv, inv.shape[0]


def match_accumulate(feat, inds_reverse, text_features, store, first, normalize=False, feat2=None, smax3d=None, smax2d=None):
    """One repeat of the ``test_repeats`` loop (run/evaluate.py:385-425) on the device: the fp16 scores of
    ``_scores(feat, ...)`` -- or, with ``feat2`` (fp16 fused features) and the two row maxima, of the ensemble product --
    are added into ``store`` (fp16 [N_pts, K], in place; ``first`` starts it from ``0.0 + pred``).  Returns the int64
    labels ``store.float().max(1)[1]`` of the accumulated scores.  The [N_pts, K] scores are never materialised."""
    C.require_cuda(feat, 'features')
    feat = feat.contiguous()
    is_f16 = feat.dtype == torch.float16
    if not is_f16 and feat.dtype != torch.float32:
        feat = feat.float()
    n_vox, c = feat.shape
    text = text_features.to(device=feat.device, dtype=torch.float16).contiguous()
    k = text.shape[0]
    if text.shape[1] != c:
        raise ValueError(f"match_accumulate: text embeddings have width {text.shape[1]}, features {c}")
    inv, n_pts = _inds(inds_reverse, feat.device, n_vox)
    if store.dtype != torch.float16 or tuple(store.shape) != (n_pts, k) or not store.is_contiguous() or store.device != feat.device:
        raise ValueError(f"match_accumulate: store must be a contiguous fp16 [{n_pts}, {k}] tensor on {feat.device}, "
                         f"got {store.dtype} {tuple(store.shape)} on {store.device}")
    if feat2 is not None:
        if is_f16:
            raise ValueError("match_accumulate: the ensemble product takes fp32 network features")
        feat2 = feat2.to(feat.device, torch.float16).contiguous()
        if feat2.shape != feat.shape:
            raise ValueError(f"match_accumulate: fused features {tuple(feat2.shape)} vs network features {tuple(feat.shape)}")
        smax3d, smax2d = smax3d.contiguous(), smax2d.contiguous()
        if smax3d.shape != (n_pts,) or smax2d.shape != (n_pts,):
            raise ValueError("match_accumulate: smax3d / smax2d must have one fp32 value per point")
    with torch.cuda.device(feat.device):
        label = torch.empty(n_pts, dtype=torch.int64, device=feat.device)
        C.call('osb_match_accumulate', C.ptr(feat), int(is_f16), C.ptr(feat2), C.ptr(smax3d), C.ptr(smax2d), n_vox, c, C.ptr(inv),
               n_pts, C.ptr(text), k, int(normalize), C.ptr(store), int(bool(first)), C.ptr(label), C.stream_ptr())
    return label


def logits_accumulate(logits, inds_reverse, store, first):
    """One repeat of run/eval_mink.py:168-216 on the device: fp32 class logits [N_vox, C] gathered through
    ``inds_reverse`` and added into ``store`` (fp32 [N_pts, C], in place; ``first`` starts it from ``pred + 0.0``).
    Returns (label of this repeat alone, label of the accumulated store), both int64 first-maximum argmaxes."""
    C.require_cuda(logits, 'logits')
    logits = logits.float().contiguous()
    n_vox, c = logits.shape
    inv, n_pts = _inds(inds_reverse, logits.device, n_vox)
    if store.dtype != torch.float32 or tuple(store.shape) != (n_pts, c) or not store.is_contiguous() or store.device != logits.device:
        raise ValueError(f"logits_accumulate: store must be a contiguous fp32 [{n_pts}, {c}] tensor on {logits.device}, "
                         f"got {store.dtype} {tuple(store.shape)} on {store.device}")
    with torch.cuda.device(logits.device):
        cur = torch.empty(n_pts, dtype=torch.int64, device=logits.device)
        acc = torch.empty(n_pts, dtype=torch.int64, device=logits.device)
        C.call('osb_logits_accumulate', C.ptr(logits), n_vox, c, C.ptr(inv), n_pts, C.ptr(store), int(bool(first)), C.ptr(cur),
               C.ptr(acc), C.stream_ptr())
    return cur, acc
