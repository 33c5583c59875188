"""Evaluation API with the reference's names (``tiseg/utils/__init__.py:1-12``): per-image ``pre_eval_*``
functions backed by the CUDA library, and the dataset-level reducers (host arithmetic on a handful of
numbers per image, written against ``tiseg/utils/inst_metrics.py:383-626`` and ``sem_metrics.py:164-303``).

Return types follow the reference: ``np.float64`` / int tuples for the instance metrics, float32 torch
tensors for the semantic counts.  Every ``pre_eval_*`` also accepts a batch ``[N, H, W]`` and then returns a
list of per-image tuples (what ``Dataset.pre_eval`` accumulates).
"""
from collections import OrderedDict

import numpy as np

from . import ops
from . import _lib
from ._lib import is_torch


def _host(a):
    """Result array -> numpy.  For a CUDA tensor the library context is synchronised first: errors only a kernel can
    detect (an instance id outside the supported range) are raised HERE instead of being read back as wrong numbers."""
    if is_torch(a):
        if a.is_cuda:
            _lib.get_ctx(a.device.index).synchronize()
        return a.cpu().numpy()
    return np.asarray(a)


def _is_batch(a):
    return a.ndim == 3


# --------------------------------------------------------------------------- per image (GPU)
def pre_eval_bin_aji(inst_pred, inst_gt):
    """inst_metrics.py:10-92 -> (overall_inter, overall_union)."""
    aji, _ = ops.pair_metrics_bin(inst_pred, inst_gt)
    aji = _host(aji)
    if aji.ndim == 2:
        return [(np.float64(r[0]), np.float64(r[1])) for r in aji]
    return np.float64(aji[0]), np.float64(aji[1])


def pre_eval_bin_pq(inst_pred, inst_gt, match_iou=0.5):
    """inst_metrics.py:138-229 -> (tp, fp, fn, iou_sum).  ``match_iou >= 0.5`` as in the reference's unique-matching
    branch (:197-203); below 0.5 the reference switches to Hungarian matching (:204-218), which none of its callers
    reaches and which is not built."""
    assert match_iou >= 0.0, "Cant' be negative"
    if match_iou < 0.5:
        raise NotImplementedError("match_iou < 0.5 (Hungarian matching, inst_metrics.py:204-218) is not implemented")
    _, pq = ops.pair_metrics_bin(inst_pred, inst_gt, match_iou)
    pq = _host(pq)
    if pq.ndim == 2:
        return [(int(r[0]), int(r[1]), int(r[2]), np.float64(r[3])) for r in pq]
    return int(pq[0]), int(pq[1]), int(pq[2]), np.float64(pq[3])


def _split_multiclass(rec, reduce_zero_label):
    rec = _host(rec).astype(np.float32)          # the reference accumulates into float32 arrays
    cols = tuple(rec[..., k] for k in range(rec.shape[-1]))
    return tuple(c[..., 1:] for c in cols) if reduce_zero_label else cols


def _maps_from_id_lists(inst, id_list_per_class, num_classes):
    """The reference's ``{class: [instance ids]}`` form (what ``assign_sem_class_to_insts`` returns,
    instance_semantic.py:68-93) -> (instance map with unlisted ids removed, class map): every listed instance is painted
    with its class, so the device-side majority vote reproduces the dictionary exactly; ids that appear in no list do not
    take part in the reference's sums at all (inst_metrics.py:103-131) and are zeroed.  A uint16 map stays uint16."""
    inst = np.asarray(_host(inst))
    top = int(inst.max()) if inst.size else 0
    lut = np.full(top + 2, -1, np.int64)
    for cls, ids in id_list_per_class.items():
        if not 0 <= int(cls) < num_classes:
            raise IndexError("class id %r outside [0, %d)" % (cls, num_classes))     # the reference indexes [num_classes] arrays
        for i in ids:
            i = int(i)
            if 0 < i <= top:
                if lut[i] not in (-1, int(cls)):
                    raise ValueError("instance id %d is listed under two classes" % i)
                lut[i] = int(cls)
    cls_of = lut[np.clip(inst, 0, top + 1)]
    keep = (cls_of >= 0) & (inst > 0)
    ids = np.uint16 if inst.dtype == np.uint16 else np.int32
    return np.where(keep, inst, 0).astype(ids), np.where(keep, cls_of, 0).astype(np.uint8)


def _multiclass(inst_pred, inst_gt, a, b, num_classes):
    """dispatch on the reference's argument form (id dictionaries) vs the semantic maps themselves"""
    if isinstance(a, dict) and isinstance(b, dict):
        ip, sp = _maps_from_id_lists(inst_pred, a, num_classes)
        ig, sg = _maps_from_id_lists(inst_gt, b, num_classes)
        r = ops.pair_metrics_multiclass(ip, sp, ig, sg, num_classes, want_bin=False)
        aji, pq = _host(r["aji"]).copy(), _host(r["pq"]).copy()
        # slot 0 of PQ counts the LIST entries of class 0 (inst_metrics.py:249-252), id 0 included only if it is listed
        if 0 in a or 0 in b:
            pq[0, :] = 0
            pq[0, 1], pq[0, 2] = len(a[0]), len(b[0])       # (KeyError like the reference if only one side lists class 0)
        return aji, pq
    r = ops.pair_metrics_multiclass(inst_pred, a, inst_gt, b, num_classes, want_bin=False)
    return r["aji"], r["pq"]


def pre_eval_aji(inst_pred, inst_gt, pred_id_list_per_class, gt_id_list_per_class, num_classes, reduce_zero_label=True):
    """inst_metrics.py:95-135 -> (inter[C-1], union[C-1]) float32.  Called like the reference (conic.py:178-188) with the
    two ``{class: [instance ids]}`` dictionaries of ``assign_sem_class_to_insts``; the two semantic maps may be passed in
    their place, the class assignment (instance_semantic.py:68-93) then runs on the device as well."""
    aji, _ = _multiclass(inst_pred, inst_gt, pred_id_list_per_class, gt_id_list_per_class, num_classes)
    return _split_multiclass(aji, reduce_zero_label)


def pre_eval_pq(inst_pred, inst_gt, pred_id_list_per_class, gt_id_list_per_class, num_classes, reduce_zero_label=True):
    """inst_metrics.py:232-280 -> (tp, fp, fn, iou)[C-1] float32; arguments as ``pre_eval_aji``."""
    _, pq = _multiclass(inst_pred, inst_gt, pred_id_list_per_class, gt_id_list_per_class, num_classes)
    return _split_multiclass(pq, reduce_zero_label)


def pre_eval_all_semantic_metric(pred_label, target_label, num_classes, ignore_index=255, reduce_zero_label=True):
    """sem_metrics.py:16-53 -> (TP, TN, FP, FN, Pred, GT) float32 torch tensors [C-1] (a list of such tuples
    for a batch)."""
    import torch
    counts, valid = ops.sem_counts(pred_label, target_label, num_classes, ignore_index)
    counts, valid = _host(counts), _host(valid)

    batch = counts.ndim == 3
    t = torch.from_numpy(np.ascontiguousarray(counts if batch else counts[None]).astype(np.float32))      # [N, 5, C]
    tp, fp, fn, pr, gt = (t[:, k] for k in range(5))
    tn = pr.sum(1, keepdim=True) - (tp + fp + fn)       # sem_metrics.py:43: total = histc(pred).sum() over every class
    pack = (tp, tn, fp, fn, pr, gt)
    if reduce_zero_label:
        pack = tuple(x[:, 1:] for x in pack)
    out = [tuple(x[j] for x in pack) for j in range(t.shape[0])]
    return out if batch else out[0]


# --------------------------------------------------------------------------- convenience scores
# (binary_panoptic_quality, binary_inst_dice, dice_similarity_coefficient and precision_recall are compared with the
# reference's own functions; binary_aggregated_jaccard_index, aggregated_jaccard_index and panoptic_quality RAISE in
# the reference — inst_metrics.py:292, 307, 353 hand semantic maps to functions that expect per-class id lists — so
# these three follow the formulas of the corresponding reducers instead.)
def binary_aggregated_jaccard_index(inst_pred, inst_gt):
    i, u = pre_eval_bin_aji(inst_pred, inst_gt)
    return 0. if i == 0. or u == 0. else i / u


def aggregated_jaccard_index(inst_pred, inst_gt, sem_pred, sem_gt, num_classes):
    i, u = pre_eval_aji(inst_pred, inst_gt, sem_pred, sem_gt, num_classes)
    return 0. if np.sum(i) == 0. or np.sum(u) == 0. else np.sum(i) / np.sum(u)


def _dq_sq_pq(tp, fp, fn, iou, eps_dq=0.0):
    dq = tp / (tp + 0.5 * fp + 0.5 * fn + eps_dq)
    sq = iou / (tp + 1.0e-6)
    return dq, sq, dq * sq


def binary_panoptic_quality(inst_pred, inst_gt, match_iou=0.5):
    return _dq_sq_pq(*pre_eval_bin_pq(inst_pred, inst_gt, match_iou))


def panoptic_quality(inst_pred, inst_gt, sem_pred, sem_gt, num_classes, match_iou=0.5):
    tp, fp, fn, iou = pre_eval_pq(inst_pred, inst_gt, sem_pred, sem_gt, num_classes)
    return _dq_sq_pq(np.sum(tp), np.sum(fp), np.sum(fn), np.sum(iou))


def binary_inst_dice(inst_pred, inst_gt, match_iou=0.5):
    tp, fp, fn, _ = pre_eval_bin_pq(inst_pred, inst_gt, match_iou)
    return 2 * tp / (2 * tp + fp + fn)


# --------------------------------------------------------------------------- dataset-level reducers (host)
def _columns(pre_eval_results, arity):
    cols = tuple(zip(*pre_eval_results))
    assert len(cols) == arity
    return cols


def _finish(ret, nan_to_num):
    if nan_to_num is not None:
        ret = OrderedDict({k: np.nan_to_num(v, nan=nan_to_num) for k, v in ret.items()})
    return ret


def pre_eval_to_bin_aji(pre_eval_results, nan_to_num=None):
    inter, union = _columns(pre_eval_results, 2)
    return _finish({'Aji': sum(np.sum(x) for x in inter) / sum(np.sum(x) for x in union)}, nan_to_num)


def pre_eval_to_imw_aji(pre_eval_results, nan_to_num=None):
    inter, union = _columns(pre_eval_results, 2)
    return _finish({'Aji': np.array([np.sum(i) / np.sum(u) for i, u in zip(inter, union)])}, nan_to_num)


def pre_eval_to_aji(pre_eval_results, nan_to_num=None):
    inter, union = _columns(pre_eval_results, 2)
    return _finish({'Aji': sum(inter) / sum(union)}, nan_to_num)


def _pq_dict(tp, fp, fn, iou, nan_to_num, analysis_mode):
    dq, sq, pq = _dq_sq_pq(tp, fp, fn, iou)
    ret = _finish({'DQ': dq, 'SQ': sq, 'PQ': pq}, nan_to_num)
    if analysis_mode:
        ret.update({'pq_TP': tp, 'pq_FP': fp, 'pq_FN': fn, 'pq_IoU': np.round(iou, 2)})
    return ret


def pre_eval_to_bin_pq(pre_eval_results, nan_to_num=None, analysis_mode=False):
    cols = _columns(pre_eval_results, 4)
    tp, fp, fn, iou = (sum(np.sum(x) for x in col) for col in cols)
    return _pq_dict(tp, fp, fn, iou, nan_to_num, analysis_mode)


def pre_eval_to_pq(pre_eval_results, nan_to_num=None, analysis_mode=False):
    cols = _columns(pre_eval_results, 4)
    tp, fp, fn, iou = (sum(col) for col in cols)
    return _pq_dict(tp, fp, fn, iou, nan_to_num, analysis_mode)


def pre_eval_to_imw_pq(pre_eval_results, nan_to_num=None):
    cols = _columns(pre_eval_results, 4)
    rows = [_dq_sq_pq(np.sum(tp), np.sum(fp), np.sum(fn), np.sum(iou), eps_dq=1.0e-6) for tp, fp, fn, iou in zip(*cols)]
    ret = {k: np.array([r[j] for r in rows]) for j, k in enumerate(('DQ', 'SQ', 'PQ'))}
    return _finish(ret, nan_to_num)


def pre_eval_to_imw_inst_dice(pre_eval_results, nan_to_num=None):
    tp, fp, fn, _ = _columns(pre_eval_results, 4)
    return _finish({'InstDice': np.array([2 * a / (2 * a + b + c) for a, b, c in zip(tp, fp, fn)])}, nan_to_num)


def pre_eval_to_inst_dice(pre_eval_results, nan_to_num=None):
    tp, fp, fn, _ = _columns(pre_eval_results, 4)
    tp, fp, fn = sum(tp), sum(fp), sum(fn)
    return _finish({'InstDice': 2 * tp / (2 * tp + fp + fn)}, nan_to_num)


_SEM_ALLOWED = ['Accuracy', 'IoU', 'Dice', 'Recall', 'Precision']


def _sem_formulas(TP, TN, FP, FN, P, G, metrics):
    ret = {}
    for m in metrics:
        if m == 'Accuracy':
            ret[m] = (TP + TN) / G.sum()
        elif m == 'IoU':
            ret[m] = TP / (P + G - TP)
        elif m == 'Dice':
            ret[m] = 2 * TP / (P + G)
        elif m == 'Recall':
            ret[m] = TP / (TP + FN)
        elif m == 'Precision':
            ret[m] = TP / (TP + FP)
    return ret


def total_area_to_sem_metrics(total_area_TP, total_area_TN, total_area_FP, total_area_FN, total_area_pred_label,
                              total_area_label, metrics=['IoU'], nan_to_num=None):
    if isinstance(metrics, str):
        metrics = [metrics]
    if not set(metrics).issubset(set(_SEM_ALLOWED)):
        raise KeyError('metrics {} is not supported'.format(metrics))
    ret = _sem_formulas(total_area_TP, total_area_TN, total_area_FP, total_area_FN, total_area_pred_label,
                        total_area_label, metrics)
    return _finish({k: v.numpy() for k, v in ret.items()}, nan_to_num)


def pre_eval_to_sem_metrics(pre_eval_results, metrics=['IoU'], nan_to_num=None, beta=1):
    """sem_metrics.py:214-247: sequential float32 sums over the images, then the ratio formulas."""
    cols = _columns(pre_eval_results, 6)
    return total_area_to_sem_metrics(*(sum(col) for col in cols), metrics, nan_to_num)


def pre_eval_to_imw_sem_metrics(pre_eval_results, metrics=['IoU'], nan_to_num=None):
    """sem_metrics.py:164-211: per image, classes summed first."""
    import torch
    cols = _columns(pre_eval_results, 6)
    sums = [[torch.sum(x) for x in col] for col in cols]
    ret = {}
    for m in [k for k in _SEM_ALLOWED if k in metrics]:
        ret[m] = np.array([_sem_formulas(*vals, [m])[m].numpy() for vals in zip(*sums)])
    order = [k for k in ('Accuracy', 'IoU', 'Dice', 'Recall', 'Precision') if k in ret]
    return _finish(OrderedDict((k, ret[k]) for k in order), nan_to_num)


def dice_similarity_coefficient(pred_label, target_label, num_classes, nan_to_num=None):
    res = pre_eval_all_semantic_metric(pred_label, target_label, num_classes, reduce_zero_label=False)
    return pre_eval_to_sem_metrics([res], ['Dice'], nan_to_num)['Dice']


def precision_recall(pred_label, target_label, num_classes, nan_to_num=None):
    res = pre_eval_all_semantic_metric(pred_label, target_label, num_classes, reduce_zero_label=False)
    r = pre_eval_to_sem_metrics([res], ['Precision', 'Recall'], nan_to_num)
    return r['Precision'], r['Recall']


# --------------------------------------------------------------------------- tiseg/datasets/utils exports
def re_instance(instance_map):
    """datasets/utils/instance_semantic.py:5-15: sorted unique non-zero ids -> 1..K (int32)."""
    return ops.re_instance(instance_map)


def assign_sem_class_to_insts(inst_seg, sem_seg, num_classes):
    """datasets/utils/instance_semantic.py:68-93 -> {class: [instance ids]} (id 0 always listed under class 0, ids in
    ascending order inside a class, classes in order of first appearance over the ascending ids)."""
    table = _host(ops.assign_sem_class(inst_seg, sem_seg, num_classes))
    out = {}
    for v in np.flatnonzero(table != 255):
        out.setdefault(int(table[v]), []).append(int(v))
    return out
