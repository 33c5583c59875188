"""Test-time tails of the reference's segmentors (``tiseg/models/segmentors/*.py``): everything between the
CNN heads' raw outputs and ``[{'sem_pred': ..., 'inst_pred': ...}]``, with the reference's method names and
argument meaning.  The CNN (``calculate``) is not here — it stays in PyTorch / cuDNN; these classes take its
logits.  All compute runs in the CUDA library; inputs may be numpy arrays or CUDA tensors, single tiles
``[H, W]`` or batches ``[N, H, W]``.

    post = UNet(num_classes=2)                     # unet.py
    out = post.forward_eval(sem_logits)            # [T, C, H, W] logits of the T TTA variants
    out[0]['sem_pred'], out[0]['inst_pred']

Dtypes: ``sem_pred`` uint8, ``inst_pred`` int32 (the reference returns int32 / int64 with the same values).
"""
import numpy as np

from . import ops
from ._lib import is_torch


def _as_class_map(pred):
    """argmax output (int64 in the reference) -> uint8 working copy."""
    if is_torch(pred):
        import torch
        return pred.to(torch.uint8).contiguous()
    return np.ascontiguousarray(pred, dtype=np.uint8)


def generate_direction_differential_map(dir_map, direction_classes=9, background=None, use_reg=False):
    """tiseg/models/utils/direct_diff_map.py:95-167 for the label form (``use_reg=False``, nine direction classes):
    dir_map ``[N, H, W]`` tensor (N == 1: the reference normalises over the whole tensor and supports batch size 1 only,
    :104) or ``[H, W]`` numpy array -> fp32 tensor ``[1, H, W]`` with values in {0, 0.5, 1} on the input's device."""
    import torch
    if use_reg:
        raise NotImplementedError("generate_direction_differential_map(use_reg=True): the angle-regression variant "
                                  "(multi_task_cdnet.py:304-317) is not part of the rebuilt path")
    if direction_classes != 9:
        raise NotImplementedError("only nine direction classes (eight angles + background), the shipped configuration")
    x = dir_map if is_torch(dir_map) else np.asarray(dir_map)
    if x.ndim == 2:
        x = x[None]
    if x.ndim != 3 or x.shape[0] != 1:
        raise ValueError("dir_map must be [1, H, W] or [H, W]: the reference supports batch size 1 only")
    if is_torch(x):
        dd = ops.ddm(x.to(torch.uint8))
        return dd if is_torch(dd) else torch.from_numpy(dd).to(x.device)
    return torch.from_numpy(np.asarray(ops.ddm(x.astype(np.uint8))))


def _wrap(sem_pred, inst_pred):
    if sem_pred.ndim == 2:
        return [{'sem_pred': sem_pred, 'inst_pred': inst_pred}]
    return [{'sem_pred': s, 'inst_pred': i} for s, i in zip(sem_pred, inst_pred)]


class _UNetFamily:
    """unet.py:71-93 and siblings: per class fill holes -> remove_small_objects(5) -> label -> dilation."""
    radius = 1
    has_edge = False

    def __init__(self, num_classes, test_cfg=None):
        self.num_classes = num_classes
        self.test_cfg = dict(test_cfg or {})

    def postprocess(self, pred):
        edge = self.num_classes if self.has_edge else None
        radius = self.test_cfg.get('radius', self.radius)
        work = _as_class_map(pred)
        max_class = self.num_classes if self.has_edge else self.num_classes - 1
        sem_pred, inst_pred = ops.postproc_unet(work, max_class, radius, edge)
        if edge is not None and work is not pred:
            pred[pred == edge] = 0                      # the reference zeroes the edge class in the caller's map
        return sem_pred, inst_pred

    def forward_eval(self, sem_logit):
        """sem_logit: raw logits ``[T, C, H, W]`` (or ``[N, T, C, H, W]``) of the TTA variants."""
        sem_pred = ops.softmax_argmax(sem_logit)
        return _wrap(*self.postprocess(sem_pred))


class UNet(_UNetFamily):            # unet.py:71-93 (radius 1)
    pass


class MicroNet(_UNetFamily):        # micronet.py:185-207
    pass


class CUNet(_UNetFamily):           # cunet.py:70-93: 3-class map, edge class = num_classes
    radius, has_edge = 3, True


class FullNet(CUNet):               # fullnet.py:190-213
    pass


class CMicroNet(CUNet):             # cmicronet.py:186-209
    pass


class DCAN(_UNetFamily):            # dcan.py:193-217: the contour head splits touching cells
    radius = 3

    def postprocess(self, cell_pred, cont_pred):
        work = _as_class_map(cell_pred)
        sem_pred, inst_pred = ops.postproc_unet(work, self.num_classes - 1, self.test_cfg.get('radius', self.radius),
                                                None, kill=cont_pred)
        if work is not cell_pred:
            cell_pred[cont_pred > 0] = 0
        return sem_pred, inst_pred

    def forward_eval(self, cell_logit, cont_logit):
        return _wrap(*self.postprocess(ops.softmax_argmax(cell_logit), ops.softmax_argmax(cont_logit)))


class CDNet(CUNet):
    """cdnet.py: direction-guided refinement (inference tail :183-217, ``_ddm_enhencement`` :354-367) followed by
    the CUNet-style postprocess with radius 3 (:96-119)."""

    def __init__(self, num_classes, num_angles=8, test_cfg=None):
        super().__init__(num_classes, test_cfg)
        self.num_angles = num_angles

    def inference_tail(self, sem_logit, dir_logit, point_logit, ori_hw=None, window=0, overlap=0):
        """head outputs of the T TTA variants -> (refined sem probabilities, dir_map of variant 0, class map).  Without
        ``ori_hw``: the heads already reverse-transformed, ``[T, C, H, W]`` or ``[N, T, C, H, W]``.  With ``ori_hw`` = (H, W):
        per head the list of raw variant outputs on the TRANSFORMED image ([N, C, Ht, Wt], or its windows
        [N, M, C, w, w] for split inference), the transforms from test_cfg, as ``Dist.inference_tail``."""
        if_ddm = self.test_cfg.get('if_ddm', False)
        if ori_hw is None:
            r = ops.cdnet_refine(sem_logit, dir_logit, point_logit, if_ddm=if_ddm)
        else:
            rots, flips = _tta_lists(self.test_cfg)
            r = ops.cdnet_refine_tta(sem_logit, dir_logit, point_logit, rots, flips, ori_hw, window, overlap, if_ddm=if_ddm)
        return r['sem_prob'], r['dir_map'], r['cls']

    _enh_mode = 0

    @classmethod
    def _ddm_enhencement(cls, sem_logit, dd_map, point_logit):
        """cdnet.py:354-367 with the reference's arguments: sem_logit ``[1, C, H, W]`` TTA-mean probabilities (modified in
        place and returned), dd_map ``[1, H, W]``, point_logit ``[1, 1, H, W]``.  (inference_tail fuses it with the rest.)"""
        if sem_logit.shape[0] != 1:
            raise ValueError("_ddm_enhencement: batch size 1 only (torch.max over the whole point map, cdnet.py:357)")
        if is_torch(sem_logit) and not sem_logit.is_contiguous():
            work = sem_logit.contiguous()
            ops.ddm_enhance(work, dd_map, point_logit[:, 0], mode=cls._enh_mode)
            sem_logit.copy_(work)
            return sem_logit
        return ops.ddm_enhance(sem_logit, dd_map, point_logit[:, 0], mode=cls._enh_mode)

    def forward_eval(self, sem_logit, dir_logit, point_logit):
        _, dir_map, sem_pred = self.inference_tail(sem_logit, dir_logit, point_logit)
        sem_pred, inst_pred = self.postprocess(sem_pred)
        out = _wrap(sem_pred, inst_pred)
        return out


def _tta_lists(test_cfg):
    """the reference's loop order: rotate_degrees outer, flip_directions inner"""
    rots, flips = test_cfg.get('rotate_degrees', [0]), test_cfg.get('flip_directions', ['none'])
    return [r for r in rots for _ in flips], [f for _ in rots for f in flips]


class Dist:
    """dist.py:262-284: semantic argmax passes through, instances from the distance-map watershed."""

    def __init__(self, num_classes=2, test_cfg=None):
        self.num_classes = num_classes
        self.test_cfg = dict(test_cfg or {})

    def postprocess(self, sem_pred, dist_logit):
        return sem_pred, ops.postproc_dist(dist_logit)

    def inference_tail(self, sem_variants, dist_variants, ori_hw, window=0, overlap=0):
        """dist.py:369-410 after the CNN: the raw outputs of the TTA variants on the TRANSFORMED image (per variant
        [N, C, Ht, Wt], or its windows [N, M, C, w, w] for split inference) -> (sem class map [N, H, W], TTA-mean
        distance map [N, H, W]): reverse transform + softmax + mean for the semantic head, reverse transform + plain
        mean for the distance head, both fused into one pass each."""
        rots, flips = _tta_lists(self.test_cfg)
        sem_pred = ops.softmax_argmax_tta(sem_variants, rots, flips, ori_hw, window, overlap)
        dist = ops.tta_mean(dist_variants, rots, flips, ori_hw, window, overlap)
        return sem_pred, dist[:, 0]

    def forward_eval(self, sem_logit, dist_logit):
        """sem_logit ``[T, C, H, W]`` raw; dist_logit ``[H, W]`` = TTA mean of the distance head (dist.py:398-406)."""
        sem_pred = ops.softmax_argmax(sem_logit)
        return _wrap(*self.postprocess(sem_pred, dist_logit))


class HoverNet:
    """hovernet.py:267-365."""

    def __init__(self, num_classes=3, test_cfg=None):
        self.num_classes = num_classes
        self.test_cfg = dict(test_cfg or {})

    def hover_post_proc(self, fore_map, hv_map, fx=1, scale_factor=1):
        return ops.postproc_hover(fore_map, hv_map, scale_factor=scale_factor, fx=fx)

    def inference_tail(self, sem_variants, hv_variants, fore_variants, ori_hw, window=0, overlap=0):
        """hovernet.py:367-414 after the CNN -> (sem class map [N,H,W], hv map [N,H,W,2] of variant 0 — the reference
        keeps ``hv_logit_list[0]`` (:406) — and the foreground probability [N,H,W] = channel 1 of the TTA-mean softmax)."""
        rots, flips = _tta_lists(self.test_cfg)
        sem_pred = ops.softmax_argmax_tta(sem_variants, rots, flips, ori_hw, window, overlap)
        hv = ops.tta_mean(hv_variants[:1], rots[:1], flips[:1], ori_hw, window, overlap)
        _, fore = ops.softmax_argmax_tta(fore_variants, rots, flips, ori_hw, window, overlap, want_prob=True)
        hv = hv.permute(0, 2, 3, 1).contiguous() if is_torch(hv) else np.ascontiguousarray(np.moveaxis(hv, 1, -1))
        return sem_pred, hv, fore[:, 1]

    def forward_eval(self, sem_logit, hv_map, fore_prob):
        """sem_logit ``[T, C, H, W]`` raw; hv_map ``[H, W, 2]``; fore_prob ``[H, W]`` (softmax channel 1)."""
        sem_pred = ops.softmax_argmax(sem_logit)
        inst_pred = self.hover_post_proc(fore_prob, hv_map, scale_factor=self.test_cfg.get('scale_factor', 1))
        return _wrap(sem_pred, inst_pred)


class MultiTaskUNet:
    """multi_task_unet.py:68-106 (inner map has no edge class)."""
    edge_id = None
    returns_canvas = True

    def __init__(self, num_classes, test_cfg=None):
        self.num_classes = num_classes
        self.test_cfg = dict(test_cfg or {})

    def postprocess(self, inner_pred, sem_pred):
        canvas, inst_pred = ops.postproc_multitask(inner_pred, sem_pred, self.num_classes - 1, self.edge_id, 20)
        return (canvas if self.returns_canvas else sem_pred), inst_pred

    def forward_eval(self, inner_logit, sem_logit):
        return _wrap(*self.postprocess(ops.softmax_argmax(inner_logit), ops.softmax_argmax(sem_logit)))


class MultiTaskCUNet(MultiTaskUNet):    # multi_task_cunet.py:69-108: three-class inner map, edge = 2
    edge_id = 2


class MultiTaskCDNet(MultiTaskCUNet):
    """multi_task_cdnet.py: direction-guided refinement of the three-class head (inference tail :262-330 with its own
    ``_ddm_enhencement`` :548-564) followed by the multi-task postprocess (:220-243, which returns the RAW sem_pred, not
    the canvas)."""
    returns_canvas = False
    _enh_mode = 1

    def __init__(self, num_classes, num_angles=8, test_cfg=None, if_ddm=False, use_regression=False):
        super().__init__(num_classes, test_cfg)
        if num_angles != 8:
            raise NotImplementedError("the direction differential map is built for eight angles (nine classes)")
        # use_regression (multi_task_cdnet.py:304-315): dir_logit is then the ONE-channel angle head, in radians
        self.num_angles, self.if_ddm, self.use_regression = num_angles, if_ddm, use_regression

    def inference_tail(self, tc_logit, sem_logit, dir_logit, point_logit, ori_hw=None, window=0, overlap=0):
        """head outputs of the T TTA variants -> (refined tc probabilities, sem class map, dir_map of variant 0, tc class
        map).  Without ``ori_hw``: already reverse-transformed, [T, C, H, W] or [N, T, C, H, W].  With ``ori_hw``: per head
        the list of raw variant outputs, as ``CDNet.inference_tail``."""
        # (the channel axis is -3 of a reverse-transformed stack, of a whole variant and of a window stack alike)
        dch = np.shape(dir_logit if ori_hw is None else dir_logit[0])[-3]
        if dch != (1 if self.use_regression else self.num_angles + 1):
            raise ValueError("dir_logit has %d channels; use_regression=%s expects %d" % (
                dch, self.use_regression, 1 if self.use_regression else self.num_angles + 1))
        if ori_hw is None:
            r = ops.mtcdnet_refine(tc_logit, sem_logit, dir_logit, point_logit, if_ddm=self.if_ddm)
        else:
            rots, flips = _tta_lists(self.test_cfg)
            r = ops.mtcdnet_refine_tta(tc_logit, sem_logit, dir_logit, point_logit, rots, flips, ori_hw, window, overlap,
                                       if_ddm=self.if_ddm)
        return r['tc_prob'], r['sem_cls'], r['dir_map'], r['tc_cls']

    _ddm_enhencement = classmethod(CDNet._ddm_enhencement.__func__)

    def forward_eval(self, tc_logit, sem_logit, dir_logit=None, point_logit=None):
        if dir_logit is None:                       # two heads only: the plain multi-task tail
            return super().forward_eval(tc_logit, sem_logit)
        _, sem_pred, _, tc_pred = self.inference_tail(tc_logit, sem_logit, dir_logit, point_logit)
        return _wrap(*self.postprocess(tc_pred, sem_pred))


def three_class_gt(sem_gt_w_bound, num_classes):
    """multi_task_cdnet_debug.py:164-168 / multi_task_cunet_debug.py: the three-class target the debug segmentors emit
    next to their prediction: 0 background, 1 inside (any class), 2 boundary (label == num_classes)."""
    x = sem_gt_w_bound
    if is_torch(x):
        import torch
        return torch.where(x == 0, 0, torch.where(x == num_classes, 2 if num_classes > 1 else 1, 1)).to(torch.uint8)
    x = np.asarray(x)
    return np.where(x == 0, 0, np.where(x == num_classes, 2 if num_classes > 1 else 1, 1)).astype(np.uint8)


class _DebugTail:
    """the ``*_debug`` segmentors return ``tc_pred`` / ``tc_gt`` next to the predictions (consumed by
    ``MoNuSegDatasetDebug``)"""

    def forward_eval_debug(self, sem_gt_w_bound, *logits):
        if len(logits) == 4:
            _, sem_pred, _, tc_pred = self.inference_tail(*logits)
        else:
            tc_pred, sem_pred = ops.softmax_argmax(logits[0]), ops.softmax_argmax(logits[1])
        tc_gt = three_class_gt(sem_gt_w_bound, self.num_classes)
        sem_out, inst_pred = self.postprocess(tc_pred, sem_pred)
        out = _wrap(sem_out, inst_pred)
        if len(out) == 1:
            out[0].update(tc_pred=tc_pred if tc_pred.ndim == 2 else tc_pred[0], tc_gt=tc_gt if tc_gt.ndim == 2 else tc_gt.reshape(tc_gt.shape[-2:]))
        else:
            tg = tc_gt.reshape((-1,) + tuple(tc_gt.shape[-2:]))
            for j, o in enumerate(out):
                o.update(tc_pred=tc_pred[j], tc_gt=tg[j])
        return out


class MultiTaskCDNetDebug(_DebugTail, MultiTaskCDNet):      # multi_task_cdnet_debug.py:228-249
    pass


class MultiTaskCUNetDebug(_DebugTail, MultiTaskCUNet):      # multi_task_cunet_debug.py
    pass
