"""Array-level operators over the C-ABI CUDA library.

Every function takes numpy arrays (host buffers; the library stages them) or CUDA tensors
(zero-copy, stream-ordered) shaped ``[H, W]`` or batched ``[N, H, W]`` and returns arrays of the same
kind.  Names follow the scipy / scikit-image calls the reference makes (SURVEY.md §8a).
"""
import math

import numpy as np

from . import _lib
from ._lib import as_input, batched, empty_like_kind, get_ctx, net_inputs, ptr
from ._lib import is_torch as _lib_is_torch


def _dev(a):
    return a.device.index if (_lib.is_torch(a) and a.is_cuda) else None


def _unbatch(out, was2d):
    return out[0] if was2d else out


def _inplace_arg(a, dtype, what):
    """Arguments the reference mutates in place are handed to the library as they are (no converted copy could carry
    the mutation back), so they must already be C-contiguous arrays of the exact dtype."""
    if _lib.is_torch(a):
        ok = a.dtype == _lib._torch_dtype(dtype) and a.is_contiguous()
    else:
        ok = isinstance(a, np.ndarray) and a.dtype == np.dtype(dtype) and a.flags.c_contiguous and a.flags.writeable
    if not ok:
        raise TypeError("%s must be a writeable C-contiguous %s array (it is modified in place), got %s %s" % (
            what, np.dtype(dtype).name, type(a).__name__, getattr(a, "dtype", None)))
    return a


def softmax_argmax(logits, want_prob=False):
    """A1.  logits ``[T, C, H, W]`` / ``[N, T, C, H, W]`` fp32, fp16 or bf16 (T = TTA variants) ->
    class map uint8 (and the fp32 TTA-mean probabilities ``[.., C, H, W]`` when ``want_prob``).  Half-precision logits
    are read as they are (2 B per element) and give the outputs of their fp32 upcast, bit for bit."""
    (x,), dt = net_inputs(logits)
    single = x.ndim == 4
    if single:
        x = x[None]
    N, T, C, H, W = x.shape
    cls = empty_like_kind(x, (N, H, W), np.uint8)
    prob = empty_like_kind(x, (N, C, H, W), np.float32) if want_prob else None
    get_ctx(_dev(x)).call("tiseg_softmax_argmax_typed", dt, ptr(x), N, T, C, H, W, ptr(prob), ptr(cls))
    if single:
        cls, prob = cls[0], (prob[0] if want_prob else None)
    return (cls, prob) if want_prob else cls


def label(img, background=0, connectivity=None, return_num=False):
    """skimage.measure.label (A5) / scipy.ndimage.label with the cross structure (connectivity=1)."""
    conn = 2 if connectivity is None else int(connectivity)
    if getattr(img, "dtype", None) in (np.uint8, np.bool_) or str(getattr(img, "dtype", "")) in ("torch.uint8", "torch.bool"):
        x, fn = as_input(img, np.uint8), "tiseg_label_u8"
    else:
        x, fn = as_input(img, np.int32), "tiseg_label"
    x, was2d = batched(x)
    N, H, W = x.shape
    out = empty_like_kind(x, (N, H, W), np.int32)
    cnt = empty_like_kind(x, (N,), np.int32)
    get_ctx(_dev(x)).call(fn, ptr(x), N, H, W, int(background), conn, ptr(out), ptr(cnt))
    out = _unbatch(out, was2d)
    if return_num:
        return out, (int(cnt[0]) if was2d else cnt)
    return out


def re_instance(inst):
    """datasets/utils/instance_semantic.py:5-15."""
    x, was2d = batched(as_input(inst, np.int32))
    N, H, W = x.shape
    out = empty_like_kind(x, (N, H, W), np.int32)
    get_ctx(_dev(x)).call("tiseg_re_instance", ptr(x), N, H, W, ptr(out), ptr(None))
    return _unbatch(out, was2d)


def binary_fill_holes(mask):
    x, was2d = batched(as_input(mask, np.uint8))
    N, H, W = x.shape
    out = empty_like_kind(x, (N, H, W), np.uint8)
    get_ctx(_dev(x)).call("tiseg_fill_holes", ptr(x), N, H, W, ptr(out))
    return _unbatch(out, was2d)


def remove_small_objects(ar, min_size=64, connectivity=1):
    """skimage.morphology.remove_small_objects: bool / uint8 input -> component analysis;
    integer label input -> the labels are the components."""
    dt = str(getattr(ar, "dtype", ""))
    if dt in ("bool", "uint8", "torch.bool", "torch.uint8"):
        x, was2d = batched(as_input(ar, np.uint8))
        N, H, W = x.shape
        out = empty_like_kind(x, (N, H, W), np.uint8)
        get_ctx(_dev(x)).call("tiseg_remove_small_objects", ptr(x), N, H, W, int(min_size), int(connectivity), ptr(out))
    else:
        x, was2d = batched(as_input(ar, np.int32))
        N, H, W = x.shape
        out = empty_like_kind(x, (N, H, W), np.int32)
        get_ctx(_dev(x)).call("tiseg_remove_small_labels", ptr(x), N, H, W, int(min_size), ptr(out))
    return _unbatch(out, was2d)


def _morph(fn, lab, footprint, radius):
    x, was2d = batched(as_input(lab, np.int32))
    N, H, W = x.shape
    out = empty_like_kind(x, (N, H, W), np.int32)
    get_ctx(_dev(x)).call(fn, ptr(x), N, H, W, {"disk": 0, "square": 1}[footprint], int(radius), ptr(out))
    return _unbatch(out, was2d)


def dilation(lab, footprint="disk", radius=1):
    """skimage.morphology.dilation(lab, disk(radius)) / square(2*radius+1) on a label image."""
    return _morph("tiseg_dilate_labels", lab, footprint, radius)


def erosion(lab, footprint="disk", radius=1):
    return _morph("tiseg_erode_labels", lab, footprint, radius)


def postproc_unet(cls, max_class, radius=1, edge_id=None, kill=None):
    """A2.  Returns (sem_pred uint8, inst_pred int32).  ``cls`` (uint8) is modified in place when
    ``edge_id`` / ``kill`` are given, like the reference."""
    x, was2d = batched(_inplace_arg(cls, np.uint8, "postproc_unet: cls"))
    N, H, W = x.shape
    k = None
    if kill is not None:
        k, _ = batched(as_input(kill, np.uint8))
    sem = empty_like_kind(x, (N, H, W), np.uint8)
    inst = empty_like_kind(x, (N, H, W), np.int32)
    get_ctx(_dev(x)).call("tiseg_postproc_unet", ptr(x), N, H, W, int(max_class), int(radius),
                          -1 if edge_id is None else int(edge_id), ptr(k), ptr(sem), ptr(inst))
    return _unbatch(sem, was2d), _unbatch(inst, was2d)


def watershed(image, markers, mask=None):
    """skimage.segmentation.watershed(image, markers, mask=mask) (connectivity 1, no lines)."""
    dt = str(getattr(image, "dtype", ""))
    if dt in ("uint8", "torch.uint8"):
        im, fn = as_input(image, np.uint8), "tiseg_watershed_u8"
    else:
        im, fn = as_input(image, np.float64), "tiseg_watershed_f64"
    im, was2d = batched(im)
    mk, _ = batched(as_input(markers, np.int32))
    ms = None
    if mask is not None:
        ms, _ = batched(as_input(mask, np.uint8))
    N, H, W = im.shape
    out = empty_like_kind(im, (N, H, W), np.int32)
    get_ctx(_dev(im)).call(fn, ptr(im), ptr(mk), ptr(ms), N, H, W, ptr(out))
    return _unbatch(out, was2d)


def postproc_dist(dist, debug=False, lamb=0):
    """A8.  dist fp32, fp16 or bf16 -> inst int32 (and, with ``debug``, the marker and raw-flood maps).  ``lamb`` is the
    first argument of ``dynamic_watershed_alias`` (dist.py:114); the reference's test path passes 0.0 (dist.py:281).
    A half-precision map gives the outputs of its fp32 upcast."""
    (x,), dt = net_inputs(dist)
    x, was2d = batched(x)
    N, H, W = x.shape
    if int(lamb) != lamb:
        raise ValueError("lamb must be an integer number of grey levels")
    inst = empty_like_kind(x, (N, H, W), np.int32)
    mk = empty_like_kind(x, (N, H, W), np.int32) if debug else None
    ws = empty_like_kind(x, (N, H, W), np.int32) if debug else None
    get_ctx(_dev(x)).call("tiseg_postproc_dist_lambda_typed", dt, ptr(x), N, H, W, int(lamb), ptr(inst), ptr(mk), ptr(ws))
    if debug:
        return _unbatch(inst, was2d), _unbatch(mk, was2d), _unbatch(ws, was2d)
    return _unbatch(inst, was2d)


def pair_metrics_bin(inst_pred, inst_gt, match_iou=0.5):
    """A16 + A17 in one pass.  -> (aji [N,2] fp64 = (inter, union), pq [N,4] fp64 = (tp, fp, fn, iou)).
    ``match_iou`` >= 0.5: a pair counts as a PQ match when its IoU is greater (inst_metrics.py:197-203)."""
    p, was2d = batched(as_input(inst_pred, np.int32))
    # a uint16 ground truth (ids < 65536) is taken as it is: half the bytes to upload
    gt16 = str(getattr(inst_gt, "dtype", "")) in ("uint16", "torch.uint16")
    g, _ = batched(as_input(inst_gt, np.uint16 if gt16 else np.int32))
    if tuple(p.shape) != tuple(g.shape):
        raise ValueError("prediction / ground-truth shape mismatch: %r vs %r" % (tuple(p.shape), tuple(g.shape)))
    N, H, W = p.shape
    aji = empty_like_kind(p, (N, 2), np.float64)
    pq = empty_like_kind(p, (N, 4), np.float64)
    import ctypes
    get_ctx(_dev(p)).call("tiseg_pair_metrics_bin_u16gt" if gt16 else "tiseg_pair_metrics_bin_iou", ptr(p), ptr(g), N, H, W,
                          ctypes.c_double(float(match_iou)), ptr(aji), ptr(pq))
    return (aji[0], pq[0]) if was2d else (aji, pq)


def sem_counts(pred, gt, num_classes, ignore_index=255):
    """A19.  -> (counts [N,5,C] int64 = TP, FP, FN, Pred, GT; valid [N] int64)."""
    p, was2d = batched(as_input(pred, np.uint8))
    g, _ = batched(as_input(gt, np.uint8))
    N, H, W = p.shape
    counts = empty_like_kind(p, (N, 5, num_classes), np.int64)
    valid = empty_like_kind(p, (N,), np.int64)
    get_ctx(_dev(p)).call("tiseg_sem_counts", ptr(p), ptr(g), N, H, W, int(num_classes), int(ignore_index),
                          ptr(counts), ptr(valid))
    return (counts[0], valid[0]) if was2d else (counts, valid)


def pair_metrics_multiclass(inst_pred, sem_pred, inst_gt, sem_gt, num_classes, want_bin=True):
    """A18 (+ A16/A17 from the same pair table).  -> dict(aji [N,C,2], pq [N,C,4], bin_aji [N,2], bin_pq [N,4])
    fp64; slot 0 of the class axis is the reference's class-0 slot."""
    p, was2d = batched(as_input(inst_pred, np.int32))
    g, _ = batched(as_input(inst_gt, np.int32))
    ps, _ = batched(as_input(sem_pred, np.uint8))
    gs, _ = batched(as_input(sem_gt, np.uint8))
    N, H, W = p.shape
    C = int(num_classes)
    aji = empty_like_kind(p, (N, C, 2), np.float64)
    pq = empty_like_kind(p, (N, C, 4), np.float64)
    baji = empty_like_kind(p, (N, 2), np.float64) if want_bin else None
    bpq = empty_like_kind(p, (N, 4), np.float64) if want_bin else None
    get_ctx(_dev(p)).call("tiseg_pair_metrics_multiclass", ptr(p), ptr(ps), ptr(g), ptr(gs), N, H, W, C,
                          ptr(aji), ptr(pq), ptr(baji), ptr(bpq))
    out = dict(aji=aji, pq=pq, bin_aji=baji, bin_pq=bpq)
    if was2d:
        out = {k: (v[0] if v is not None else None) for k, v in out.items()}
    return out


def ddm(dir_map):
    """A12: generate_direction_differential_map(dir_map, 9) -> fp32 map in {0, 0.5, 1}."""
    x, was2d = batched(as_input(dir_map, np.uint8))
    N, H, W = x.shape
    out = empty_like_kind(x, (N, H, W), np.float32)
    get_ctx(_dev(x)).call("tiseg_ddm", ptr(x), N, H, W, ptr(out))
    return _unbatch(out, was2d)


def cdnet_refine(sem_logits, dir_logits, point_logits, if_ddm=True):
    """A12: CDNet.inference tail.  sem_logits [N,T,C,H,W], dir_logits [N,T,9,H,W], point_logits [N,T,1,H,W]
    (or without the leading N), all fp32 or all fp16 / bf16 (read as they are; the outputs are those of their fp32 upcast)
    -> dict(sem_prob [N,C,H,W] fp32, cls uint8, dir_map uint8, dd fp32)."""
    (s, d, p), dt = net_inputs(sem_logits, dir_logits, point_logits)
    single = s.ndim == 4
    if single:
        s, d, p = s[None], d[None], p[None]
    N, T, C, H, W = s.shape
    D = d.shape[2]
    prob = empty_like_kind(s, (N, C, H, W), np.float32)
    cls = empty_like_kind(s, (N, H, W), np.uint8)
    dm = empty_like_kind(s, (N, H, W), np.uint8)
    dd = empty_like_kind(s, (N, H, W), np.float32)
    get_ctx(_dev(s)).call("tiseg_cdnet_refine_typed", dt, ptr(s), ptr(d), ptr(p), N, T, C, D, H, W, 1 if if_ddm else 0,
                          ptr(prob), ptr(cls), ptr(dm), ptr(dd))
    out = dict(sem_prob=prob, cls=cls, dir_map=dm, dd=dd)
    return {k: v[0] for k, v in out.items()} if single else out


def ddm_enhance(sem_prob, dd_map, point_map, mode=0):
    """``_ddm_enhencement`` IN PLACE on ``sem_prob`` [N,C,H,W] / [C,H,W] fp32 (C-contiguous array or tensor): mode 0 =
    CDNet (cdnet.py:354-367), mode 1 = MultiTaskCDNet (multi_task_cdnet.py:548-564).  dd_map / point_map [N,H,W] / [H,W]."""
    x = _inplace_arg(sem_prob, np.float32, "ddm_enhance: sem_prob")
    single = x.ndim == 3
    xb = x[None] if single else x
    d = as_input(dd_map, np.float32)
    q = as_input(point_map, np.float32)
    if single:
        d, q = d.reshape((1,) + tuple(d.shape[-2:])), q.reshape((1,) + tuple(q.shape[-2:]))
    N, C, H, W = xb.shape
    if tuple(d.shape) != (N, H, W) or tuple(q.shape) != (N, H, W):
        raise ValueError("dd_map / point_map must be [N,H,W] matching sem_prob, got %r / %r" % (tuple(d.shape), tuple(q.shape)))
    get_ctx(_dev(xb)).call("tiseg_ddm_enhance", ptr(xb), ptr(d), ptr(q), N, C, H, W, int(mode))
    return sem_prob


def mtcdnet_refine(tc_logits, sem_logits, dir_logits, point_logits, if_ddm=True, want_sem_prob=False):
    """MultiTaskCDNet.inference tail (multi_task_cdnet.py:262-330).  tc_logits [N,T,Ctc,H,W], sem_logits [N,T,Csem,H,W],
    dir_logits [N,T,9,H,W] (or [N,T,1,H,W]: the angle head of use_regression = True), point_logits [N,T,1,H,W] (or without
    the leading N), all fp32 or all fp16 / bf16 (read as they are; the outputs are those of their fp32 upcast) ->
    dict(tc_prob, tc_cls, sem_cls, dir_map, dd[, sem_prob]), probabilities and dd fp32."""
    (t, s, d, p), dt = net_inputs(tc_logits, sem_logits, dir_logits, point_logits)
    single = t.ndim == 4
    if single:
        t, s, d, p = t[None], s[None], d[None], p[None]
    N, T, Ctc, H, W = t.shape
    Csem, D = s.shape[2], d.shape[2]
    tcp = empty_like_kind(t, (N, Ctc, H, W), np.float32)
    tcc = empty_like_kind(t, (N, H, W), np.uint8)
    semc = empty_like_kind(t, (N, H, W), np.uint8)
    semp = empty_like_kind(t, (N, Csem, H, W), np.float32) if want_sem_prob else None
    dm = empty_like_kind(t, (N, H, W), np.uint8)
    dd = empty_like_kind(t, (N, H, W), np.float32)
    get_ctx(_dev(t)).call("tiseg_mtcdnet_refine_typed", dt, ptr(t), ptr(s), ptr(d), ptr(p), N, T, Ctc, Csem, D, H, W, 1 if if_ddm else 0,
                          ptr(tcp), ptr(tcc), ptr(semp), ptr(semc), ptr(dm), ptr(dd))
    out = dict(tc_prob=tcp, tc_cls=tcc, sem_cls=semc, dir_map=dm, dd=dd)
    if want_sem_prob:
        out["sem_prob"] = semp
    return {k: v[0] for k, v in out.items()} if single else out


def align_foreground(pred, foreground, time=20):
    """A13: grows the labels of ``pred`` (int32, modified in place and returned) into ``foreground``."""
    x, was2d = batched(_inplace_arg(pred, np.int32, "align_foreground: pred"))
    f, _ = batched(as_input(foreground, np.uint8))
    N, H, W = x.shape
    get_ctx(_dev(x)).call("tiseg_align_foreground", ptr(x), ptr(f), N, H, W, int(time))
    return pred


def postproc_multitask(inner, sem, max_class, edge_id=None, time=20):
    """Multi-task postprocess -> (sem canvas uint8, inst int32)."""
    a, was2d = batched(as_input(inner, np.uint8))
    s, _ = batched(as_input(sem, np.uint8))
    N, H, W = a.shape
    canvas = empty_like_kind(a, (N, H, W), np.uint8)
    inst = empty_like_kind(a, (N, H, W), np.int32)
    get_ctx(_dev(a)).call("tiseg_postproc_multitask", ptr(a), ptr(s), N, H, W, int(max_class),
                          -1 if edge_id is None else int(edge_id), int(time), ptr(canvas), ptr(inst))
    return _unbatch(canvas, was2d), _unbatch(inst, was2d)


def postproc_hover(fore_map, hv_map, scale_factor=1, debug=False, fx=1):
    """A11: hover_post_proc.  fore_map [N,H,W], hv_map [N,H,W,2], both fp32 or both fp16 / bf16 (read as they are; the
    outputs are those of their fp32 upcast) -> inst int32 (with ``debug`` also the blb mask, the flooded fp64 image and
    the markers).  ``fx`` sets the Sobel kernel size and the marker size threshold with the reference's expressions
    (hovernet.py:283-365): ``fx = 0.5`` runs the chain on 20x data at its native size.  An fx whose ksize cv2.Sobel
    refuses (even, or above 31: fx 0.05, 0.25, 0.75, >= 1.6, ...) raises TisegError, as the reference raises cv2.error."""
    # clamped to int32, so that an absurd fx reaches the library's range check instead of wrapping in ctypes
    ksize, obj_size = [max(-2 ** 31, min(v, 2 ** 31 - 1)) for v in (int((20 * fx) + 1), math.ceil(10 * (fx ** 2)))]
    (f, hv), dt = net_inputs(fore_map, hv_map)
    f, was2d = batched(f)
    if hv.ndim == 3:
        hv = hv[None]
    N, H, W = f.shape
    if tuple(hv.shape) != (N, H, W, 2):
        raise ValueError("hv_map must be [N,H,W,2] (HWC), got %r" % (tuple(hv.shape),))
    inst = empty_like_kind(f, (N, H, W), np.int32)
    sf = int(scale_factor)                      # the debug maps live at the resolution the chain runs at
    blb = empty_like_kind(f, (N, H * sf, W * sf), np.uint8) if debug else None
    dist = empty_like_kind(f, (N, H * sf, W * sf), np.float64) if debug else None
    mk = empty_like_kind(f, (N, H * sf, W * sf), np.int32) if debug else None
    get_ctx(_dev(f)).call("tiseg_postproc_hover_ex", dt, ptr(f), ptr(hv), N, H, W, int(scale_factor), ksize, obj_size, ptr(inst),
                          ptr(blb), ptr(dist), ptr(mk))
    if debug:
        return tuple(_unbatch(x, was2d) for x in (inst, blb, dist, mk))
    return _unbatch(inst, was2d)


def distance_transform_edt(mask):
    """A14.  scipy.ndimage.distance_transform_edt of a binary mask -> fp64 (bit-identical)."""
    x, was2d = batched(as_input(np.asarray(mask) != 0 if not _lib_is_torch(mask) else mask != 0, np.uint8))
    N, H, W = x.shape
    out = empty_like_kind(x, (N, H, W), np.float64)
    get_ctx(_dev(x)).call("tiseg_distance_transform_edt", ptr(x), N, H, W, ptr(out))
    return _unbatch(out, was2d)


def distance_transform_cdt(mask, metric="chessboard"):
    """A14.  scipy.ndimage.distance_transform_cdt (chessboard) of a binary mask -> int32."""
    if metric != "chessboard":
        raise ValueError("only the chessboard metric (the one the reference uses) is implemented")
    x, was2d = batched(as_input(np.asarray(mask) != 0 if not _lib_is_torch(mask) else mask != 0, np.uint8))
    N, H, W = x.shape
    out = empty_like_kind(x, (N, H, W), np.int32)
    get_ctx(_dev(x)).call("tiseg_distance_transform_cdt", ptr(x), N, H, W, ptr(out))
    return _unbatch(out, was2d)


def reconstruction(seed, mask, method="erosion"):
    """A9.  skimage.morphology.reconstruction(seed, mask, method='erosion') for uint8 images (3x3 footprint)."""
    if method != "erosion":
        raise ValueError("only method='erosion' (the one the reference uses, dist.py:56) is implemented")
    sd, was2d = batched(as_input(seed, np.uint8))
    mk, _ = batched(as_input(mask, np.uint8))
    N, H, W = sd.shape
    out = empty_like_kind(sd, (N, H, W), np.uint8)
    get_ctx(_dev(sd)).call("tiseg_reconstruction_erosion_u8", ptr(sd), ptr(mk), N, H, W, ptr(out))
    return _unbatch(out, was2d)


_FLIPS = {"none": 0, None: 0, "horizontal": 1, "vertical": 2, "diagonal": 3}


def softmax_argmax_tta(variants, rotate_degrees, flip_directions, ori_hw, window=0, overlap=0, want_prob=False):
    """Window stitch + TTA reverse + softmax + mean + argmax in one pass (base.py:255-295, 321-339, 365-381).

    ``variants``: one array per TTA variant, in the reference's loop order (rotate_degrees outer, flip_directions
    inner; pass the flattened lists), each the raw network output on the TRANSFORMED image: [N, C, Ht, Wt] for whole
    inference (``window = 0``) or [N, M, C, window, window] for split inference.  ``ori_hw`` = (H, W) of the image.
    The variants may be fp32, or all fp16 / bf16: they are packed and read in their dtype, and the outputs are those of
    their fp32 upcast.  Returns the class map [N, H, W] uint8 (and the fp32 mean probabilities [N, C, H, W] with
    ``want_prob``)."""
    import ctypes
    from . import _lib
    T = len(variants)
    if not (T == len(rotate_degrees) == len(flip_directions)):
        raise ValueError("one rotate_degree and one flip_direction per variant")
    H, W = int(ori_hw[0]), int(ori_hw[1])
    vs, dt = net_inputs(*variants)
    N = int(vs[0].shape[0])
    C = int(vs[0].shape[1] if window == 0 else vs[0].shape[2])
    rots = (ctypes.c_int * T)(*[int(r) for r in rotate_degrees])
    flips = (ctypes.c_int * T)(*[_FLIPS[f] for f in flip_directions])
    per_tile = int(_lib.load().tiseg_tta_input_elems(T, C, H, W, rots, int(window), int(overlap)))
    if sum(int(np.prod(v.shape[1:])) for v in vs) != per_tile:
        raise ValueError("variant shapes do not match the transforms / window geometry")
    if _lib_is_torch(vs[0]):
        import torch
        packed = torch.cat([v.reshape(N, -1) for v in vs], dim=1).contiguous()
    else:
        packed = np.ascontiguousarray(np.concatenate([v.reshape(N, -1) for v in vs], axis=1))
    cls = empty_like_kind(packed, (N, H, W), np.uint8)
    prob = empty_like_kind(packed, (N, C, H, W), np.float32) if want_prob else None
    get_ctx(_dev(packed)).call("tiseg_softmax_argmax_tta_typed", dt, ptr(packed), N, T, C, H, W, rots, flips, int(window),
                               int(overlap), ptr(prob), ptr(cls))
    return (cls, prob) if want_prob else cls


def tta_mean(variants, rotate_degrees, flip_directions, ori_hw, window=0, overlap=0):
    """Window stitch + TTA reverse + PLAIN mean of a regression head (dist.py:398-410: ``sum(dist_logit_list) /
    len(dist_logit_list)``; hovernet.py:406 keeps ``hv_logit_list[0]``: pass that one variant).  Arguments as
    ``softmax_argmax_tta`` (fp32, or all fp16 / bf16).  -> [N, C, H, W] fp32."""
    import ctypes
    T = len(variants)
    if not (T == len(rotate_degrees) == len(flip_directions)):
        raise ValueError("one rotate_degree and one flip_direction per variant")
    H, W = int(ori_hw[0]), int(ori_hw[1])
    vs, dt = net_inputs(*variants)
    N = int(vs[0].shape[0])
    C = int(vs[0].shape[1] if window == 0 else vs[0].shape[2])
    rots = (ctypes.c_int * T)(*[int(r) for r in rotate_degrees])
    flips = (ctypes.c_int * T)(*[_FLIPS[f] for f in flip_directions])
    per_tile = int(_lib.load().tiseg_tta_input_elems(T, C, H, W, rots, int(window), int(overlap)))
    if sum(int(np.prod(v.shape[1:])) for v in vs) != per_tile:
        raise ValueError("variant shapes do not match the transforms / window geometry")
    if _lib_is_torch(vs[0]):
        import torch
        packed = torch.cat([v.reshape(N, -1) for v in vs], dim=1).contiguous()
    else:
        packed = np.ascontiguousarray(np.concatenate([v.reshape(N, -1) for v in vs], axis=1))
    out = empty_like_kind(packed, (N, C, H, W), np.float32)
    get_ctx(_dev(packed)).call("tiseg_tta_mean_typed", dt, ptr(packed), N, T, C, H, W, rots, flips, int(window), int(overlap), ptr(out))
    return out


def mudslide_watershed(seg, dir_graph, fore):
    """models/utils/postprocess.py:158-181.  seg / fore: masks, dir_graph: direction labels 0..8 (modified in place when
    it is a uint8 array or tensor; otherwise the updated copy is written back into the caller's array).
    -> (pred, boundary) boolean masks."""
    s, was2d = batched(as_input(np.asarray(seg) != 0 if not _lib_is_torch(seg) else seg != 0, np.uint8))
    f, _ = batched(as_input(np.asarray(fore) != 0 if not _lib_is_torch(fore) else fore != 0, np.uint8))
    d_in = dir_graph
    d, _ = batched(as_input(d_in, np.uint8))
    if not d.flags.writeable if not _lib_is_torch(d) else False:
        d = d.copy()
    N, H, W = s.shape
    pred = empty_like_kind(s, (N, H, W), np.uint8)
    bnd = empty_like_kind(s, (N, H, W), np.uint8)
    get_ctx(_dev(s)).call("tiseg_mudslide_watershed", ptr(s), ptr(d), ptr(f), N, H, W, ptr(pred), ptr(bnd))
    dv = _unbatch(d, was2d)
    if dv is not d_in and not (_lib_is_torch(d_in) and d_in.data_ptr() == d.data_ptr()):
        if _lib_is_torch(d_in):
            d_in.copy_(dv.to(d_in.dtype))
        elif isinstance(d_in, np.ndarray) and not np.shares_memory(d_in, d):
            d_in[...] = np.asarray(dv).astype(d_in.dtype)
    to_bool = (lambda a: a.bool()) if _lib_is_torch(pred) else (lambda a: a.astype(bool))
    return to_bool(_unbatch(pred, was2d)), to_bool(_unbatch(bnd, was2d))


def assign_sem_class(inst, sem, num_classes):
    """Class of every instance id as a table [N, VM] uint8 (255 = id absent); see ``metrics.assign_sem_class_to_insts``."""
    x, was2d = batched(as_input(inst, np.int32))
    sm, _ = batched(as_input(sem, np.uint8))
    N, H, W = x.shape
    VM = max(H * W + 1, 1 << 16)
    table = empty_like_kind(x, (N, VM), np.uint8)
    get_ctx(_dev(x)).call("tiseg_assign_sem_class", ptr(x), ptr(sm), N, H, W, int(num_classes), ptr(table))
    return table[0] if was2d else table


def gen_instance_hv_map(inst):
    """datasets/ops/hv_map.py:18-97.  inst [H,W] / [N,H,W] int -> [.., H, W, 2] fp32 (x map, y map)."""
    x, was2d = batched(as_input(inst, np.int32))
    N, H, W = x.shape
    out = empty_like_kind(x, (N, H, W, 2), np.float32)
    get_ctx(_dev(x)).call("tiseg_gen_hv_map", ptr(x), N, H, W, ptr(out))
    return out[0] if was2d else out


def instance_distance_map(inst, inst_norm=True):
    """The distance target of DistanceLabelMake (datasets/ops/distance_map.py:59-110) for an instance map that
    already went through its ``_fix_inst``: per-instance chessboard distance, optionally divided by its maximum."""
    x, was2d = batched(as_input(inst, np.int32))
    N, H, W = x.shape
    out = empty_like_kind(x, (N, H, W), np.float32)
    get_ctx(_dev(x)).call("tiseg_instance_distance_map", ptr(x), N, H, W, 1 if inst_norm else 0, ptr(out))
    return _unbatch(out, was2d)


def fix_inst(inst):
    """``_fix_inst`` of the label makers (datasets/ops/distance_map.py:41-57 and its copies)."""
    x, was2d = batched(as_input(inst, np.int32))
    N, H, W = x.shape
    out = empty_like_kind(x, (N, H, W), np.int32)
    get_ctx(_dev(x)).call("tiseg_fix_inst", ptr(x), N, H, W, ptr(out))
    return _unbatch(out, was2d)


def bound_label(sem, inst, edge_id=2, selem_radius=3):
    """BoundLabelMake.__call__ after ``_fix_inst`` (datasets/ops/bound_map.py:62-88) -> (sem_gt, sem_gt_w_bound)."""
    if isinstance(selem_radius, int):
        selem_radius = (selem_radius, selem_radius)
    x, was2d = batched(as_input(inst, np.int32))
    s, _ = batched(as_input(sem, np.uint8))
    N, H, W = x.shape
    sem_out = empty_like_kind(x, (N, H, W), np.uint8)
    bound = empty_like_kind(x, (N, H, W), np.uint8)
    get_ctx(_dev(x)).call("tiseg_bound_label", ptr(s), ptr(x), N, H, W, int(edge_id), int(selem_radius[0]),
                          int(selem_radius[1]), ptr(sem_out), ptr(bound))
    return _unbatch(sem_out, was2d), _unbatch(bound, was2d)


def unet_weight_map(inst, w0=10.0, sigma=5.0):
    """UNetLabelMake after ``_fix_inst`` (datasets/ops/unet_map.py:53-98): -> (instances eroded by diamond(1), fp64 loss
    weight map with the uniform class weight 1 added)."""
    x, was2d = batched(as_input(inst, np.int32))
    N, H, W = x.shape
    inner = empty_like_kind(x, (N, H, W), np.int32)
    wmap = empty_like_kind(x, (N, H, W), np.float64)
    get_ctx(_dev(x)).call("tiseg_unet_weight_map", ptr(x), N, H, W, float(w0), float(sigma), ptr(inner), ptr(wmap))
    return _unbatch(inner, was2d), _unbatch(wmap, was2d)


def gaussian_kernel1d(sigma, radius):
    """scipy.ndimage._filters._gaussian_kernel1d(sigma, 0, radius)[::-1], the weights gaussian_filter1d correlates with"""
    sigma2 = sigma * sigma
    x = np.arange(-radius, radius + 1)
    phi_x = np.exp(-0.5 / sigma2 * x ** 2)
    phi_x = phi_x / phi_x.sum()
    return np.ascontiguousarray(phi_x[::-1], dtype=np.float64)


def direction_labels(inst, num_angles=8, sigma=2.0, truncate=4.0):
    """DirectionLabelMake after ``_fix_inst``, to_center = True (datasets/ops/direction_map.py:36-193) ->
    dict(dist_gt fp32, point_gt fp32, dir_gt uint8, reg_dir_gt fp32, loss_weight_map fp32 | None (only for 8 angles))."""
    x, was2d = batched(as_input(inst, np.int32))
    N, H, W = x.shape
    radius = int(truncate * float(sigma) + 0.5)
    gw = gaussian_kernel1d(float(sigma), radius)
    dist = empty_like_kind(x, (N, H, W), np.float32)
    point = empty_like_kind(x, (N, H, W), np.float32)
    dirm = empty_like_kind(x, (N, H, W), np.uint8)
    reg = empty_like_kind(x, (N, H, W), np.float32)
    wmap = empty_like_kind(x, (N, H, W), np.float32) if int(num_angles) == 8 else None
    get_ctx(_dev(x)).call("tiseg_direction_labels", ptr(x), N, H, W, int(num_angles), gw.ctypes.data, radius, ptr(dist),
                          ptr(point), ptr(dirm), ptr(reg), ptr(wmap))
    out = dict(dist_gt=dist, point_gt=point, dir_gt=dirm, reg_dir_gt=reg, loss_weight_map=wmap)
    return {k: (_unbatch(v, was2d) if v is not None else None) for k, v in out.items()}
