"""The CDNet and multi-task CDNet tails fed the raw TTA outputs (tiseg_cdnet_refine_tta_typed /
tiseg_mtcdnet_refine_tta_typed): every output equals the window stitch + reverse_tta_transform of the oracle followed by
the entries that take reverse-transformed heads, bit for bit, and the reference-source goldens fed raw."""
import os
import sys
import zlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import tiseg_b200  # noqa: E402,F401
from tiseg_b200 import ops, segmentors  # noqa: E402
from oracle import postprocess as opp  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(os.path.dirname(__file__), "golden")

FLIPS = ["none", "horizontal", "vertical", "diagonal"]
PAIRS = [(r, f) for r in (0, 90, 180, 270) for f in FLIPS]          # every transform the reference's TTA can make
H, W, N = 70, 97, 2                                                 # non-square: 90 / 270 swap the variant's shape


def _windows(Ht, Wt, window, overlap):
    st = window - overlap
    pad_h = st - (Ht - window) % st if Ht - window > 0 else window - Ht
    pad_w = st - (Wt - window) % st if Wt - window > 0 else window - Wt
    return ((Ht + pad_h - window) // st + 1) * ((Wt + pad_w - window) // st + 1)


def _head(rng, C, pairs, window, overlap, dtype, lo=None, hi=None, hw=(H, W)):
    """Raw variants of one head (fp32 values representable in `dtype`) and their stitched, reverse-transformed stack
    [N, T, C, H, W]: the route the existing entries take."""
    import torch
    h, w = hw
    raw, rev = [], []
    for r, f in pairs:
        Ht, Wt = (w, h) if (r // 90) % 2 else (h, w)
        shape = (N, C, Ht, Wt) if window == 0 else (N, _windows(Ht, Wt, window, overlap), C, window, window)
        x = rng.uniform(lo, hi, shape) if lo is not None else rng.standard_normal(shape) * 3
        x = torch.from_numpy(x.astype(np.float32)).to(dtype).float().numpy()
        raw.append(x)
        full = x if window == 0 else np.stack([opp.split_stitch(x[n], Ht, Wt, window, overlap) for n in range(N)])
        rev.append(np.stack([opp.reverse_tta_transform(full[n], r, f) for n in range(N)]))
    return raw, np.ascontiguousarray(np.stack(rev, axis=1))


def _as(x, dtype, device):
    """fp32 numpy -> the library's input kind: numpy (fp32 / fp16) or a torch tensor (bf16 on the host, or on the GPU)."""
    import torch
    if device == "host" and dtype != torch.bfloat16:
        return x.astype(np.float16) if dtype == torch.float16 else x
    return torch.from_numpy(x).to(dtype).to("cuda" if device == "cuda" else "cpu")


def _np(x):
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


def _same(got, want, what):
    assert set(got) == set(want), what
    for k in want:
        a, b = _np(got[k]), _np(want[k])
        assert a.shape == b.shape and a.dtype == b.dtype, "%s %s: %r %s vs %r %s" % (what, k, a.shape, a.dtype, b.shape, b.dtype)
        bad = np.argwhere(a != b)
        assert len(bad) == 0, "%s %s: %d mismatching elements, first at %r: got %r want %r" % (
            what, k, len(bad), tuple(bad[0]), a[tuple(bad[0])], b[tuple(bad[0])])


def _dtypes():
    import torch
    return {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}


# --------------------------------------------------------------------------- 1. bit identity with the existing route
@pytest.mark.parametrize("model", ["cdnet", "mtcdnet", "mtcdnet_reg"])
@pytest.mark.parametrize("window,overlap", [(0, 0), (32, 8)])
@pytest.mark.parametrize("T", [1, 3, 8])
@pytest.mark.parametrize("dt", ["fp32", "fp16", "bf16"])
def test_refine_tta_bit_identical_to_reverse_then_refine(model, window, overlap, T, dt):
    dtype = _dtypes()[dt]
    rng = np.random.default_rng(zlib.crc32(("%s %d %d %s" % (model, window, T, dt)).encode()))
    # T = 8 takes either half of the sixteen transforms, T = 1 / 3 rotate through them: every pair is exercised
    start = {1: 5 * ["cdnet", "mtcdnet", "mtcdnet_reg"].index(model) + window, 3: 3 * ["fp32", "fp16", "bf16"].index(dt) + window, 8: window // 4}[T]
    pairs = [PAIRS[(start + k) % 16] for k in range(T)]
    rots, flips = [p[0] for p in pairs], [p[1] for p in pairs]
    D = 1 if model == "mtcdnet_reg" else 9
    if model == "cdnet":
        heads = [_head(rng, 3, pairs, window, overlap, dtype), _head(rng, D, pairs, window, overlap, dtype),
                 _head(rng, 1, pairs, window, overlap, dtype)]
    else:
        dirh = _head(rng, 1, pairs, window, overlap, dtype, lo=-0.5, hi=7.0) if D == 1 else _head(rng, 9, pairs, window, overlap, dtype)
        heads = [_head(rng, 3, pairs, window, overlap, dtype), _head(rng, 4, pairs, window, overlap, dtype), dirh,
                 _head(rng, 1, pairs, window, overlap, dtype)]
    for if_ddm, device in ((True, "host"), (False, "cuda")):
        raw = [[_as(v, dtype, device) for v in h[0]] for h in heads]
        rev = [_as(h[1], dtype, device) for h in heads]
        what = "%s %s T=%d window=%d if_ddm=%s %s" % (model, dt, T, window, if_ddm, device)
        if model == "cdnet":
            got = ops.cdnet_refine_tta(*raw, rots, flips, (H, W), window, overlap, if_ddm=if_ddm)
            want = ops.cdnet_refine(*rev, if_ddm=if_ddm)
        else:
            got = ops.mtcdnet_refine_tta(*raw, rots, flips, (H, W), window, overlap, if_ddm=if_ddm, want_sem_prob=True)
            want = ops.mtcdnet_refine(*rev, if_ddm=if_ddm, want_sem_prob=True)
        _same(got, want, what)
    if model == "mtcdnet":          # the class maps alone (no semantic probabilities asked for)
        got = ops.mtcdnet_refine_tta(*raw, rots, flips, (H, W), window, overlap)
        want = ops.mtcdnet_refine(*rev)
        _same(got, want, what + " sem_cls only")


def test_refine_tta_window_edges_and_one_pixel_images():
    """Windows larger than the image, an overlap that does not divide, and images one pixel high or wide."""
    import torch
    rng = np.random.default_rng(7)
    pairs = PAIRS[3:11]
    rots, flips = [p[0] for p in pairs], [p[1] for p in pairs]
    for hw, window, overlap in [((70, 97), 48, 17), ((20, 30), 40, 10), ((1, 45), 0, 0), ((37, 1), 0, 0), ((33, 33), 16, 6)]:
        heads = [_head(rng, C, pairs, window, overlap, torch.float32, hw=hw) for C in (3, 9, 1)]
        for if_ddm in (True, False):
            got = ops.cdnet_refine_tta(*[h[0] for h in heads], rots, flips, hw, window, overlap, if_ddm=if_ddm)
            _same(got, ops.cdnet_refine(*[h[1] for h in heads], if_ddm=if_ddm), "cdnet %r window %d" % (hw, window))


def test_refine_tta_argument_checks():
    from tiseg_b200._lib import TisegError
    rng = np.random.default_rng(3)
    import torch
    heads = [_head(rng, C, PAIRS[:2], 0, 0, torch.float32) for C in (3, 9, 1)]
    raw = [h[0] for h in heads]
    with pytest.raises(ValueError):                     # one transform per variant
        ops.cdnet_refine_tta(*raw, [0], ["none"], (H, W))
    with pytest.raises(ValueError):                     # whole variants where windows are announced
        ops.cdnet_refine_tta(*raw, [0, 0], ["none", "horizontal"], (H, W), 32, 8)
    with pytest.raises(TisegError):                     # nine direction classes
        ops.cdnet_refine_tta(raw[0], [x[:, :5] for x in raw[1]], raw[2], [0, 0], ["none", "horizontal"], (H, W))
    with pytest.raises(TisegError):                     # rotations are multiples of 90 degrees
        ops.cdnet_refine_tta(*raw, [0, 45], ["none", "horizontal"], (H, W))
    many = [_head(rng, C, [PAIRS[0]] * 17, 0, 0, torch.float32)[0] for C in (3, 9, 1)]
    with pytest.raises(TisegError):                     # at most sixteen variants
        ops.cdnet_refine_tta(*many, [0] * 17, ["none"] * 17, (H, W))


# --------------------------------------------------------------------------- 2. reference-source goldens, fed raw
def test_cdnet_refine_tta_matches_reference_source_golden():
    """tta_ref.npz c*: CDNet.inference executed from source with flips; the recorded head outputs go in untouched."""
    from test_oracle_golden import _cdnet_case
    m = np.load(os.path.join(G, "tta_ref.npz"))
    for j in range(2):
        flips = [str(f) for f in m["c%d_flips" % j]]
        T = len(flips)
        raw = [[m["c%d_%s%d" % (j, key, t)].astype(np.float32)[None] for t in range(T)] for key in ("sem", "dir", "pt")]
        h, w = raw[0][0].shape[-2:]
        if_ddm = bool(m["c%d_if_ddm" % j])
        r = ops.cdnet_refine_tta(*raw, [0] * T, flips, (h, w), if_ddm=if_ddm)
        assert np.array_equal(r["dir_map"][0], m["c%d_dir_out" % j]), j
        np.testing.assert_allclose(r["sem_prob"][0], m["c%d_sem_out" % j], rtol=1e-5, atol=1e-7)
        sem, dirs, pts, _ = _cdnet_case(m, j)
        _same(r, ops.cdnet_refine(np.stack(sem)[None], np.stack(dirs)[None], np.stack(pts)[None], if_ddm=if_ddm), "golden c%d" % j)


def _mt_golden(m, prefix, j, use_regression):
    from test_gpu_ops import _check_class_map
    T = len(m["%s%d_flips" % (prefix, j)])
    raw = [[m["%s%d_%s%d" % (prefix, j, key, t)].astype(np.float32)[None] for t in range(T)] for key in ("tc", "sem", "dir", "pt")]
    rots, flips = [int(r) for r in m["%s%d_rots" % (prefix, j)]], [str(f) for f in m["%s%d_flips" % (prefix, j)]]
    if_ddm = bool(m["%s%d_if_ddm" % (prefix, j)])
    hh, ww = raw[0][0].shape[-2:]
    h, w = (ww, hh) if (rots[0] // 90) % 2 else (hh, ww)
    r = ops.mtcdnet_refine_tta(*raw, rots, flips, (h, w), if_ddm=if_ddm, want_sem_prob=True)
    # the tolerances of the golden tests of mtcdnet_refine: class maps by _check_class_map, direction maps up to libm ties
    r0 = {k: v[0] for k, v in r.items()}
    _check_class_map(r0["tc_cls"], r0["tc_prob"], m["%s%d_tc_out" % (prefix, j)], "%s%d tc" % (prefix, j))
    _check_class_map(r0["sem_cls"], r0["sem_prob"], m["%s%d_sem_out" % (prefix, j)], "%s%d sem" % (prefix, j))
    assert (r0["dir_map"] != m["%s%d_dir_out" % (prefix, j)]).mean() < 1e-3, (prefix, j)
    rev = [np.stack([opp.reverse_tta_transform(x[0], rr, ff) for x, rr, ff in zip(h_, rots, flips)])[None] for h_ in raw]
    _same(r, ops.mtcdnet_refine(*rev, if_ddm=if_ddm, want_sem_prob=True), "golden %s%d" % (prefix, j))
    seg = segmentors.MultiTaskCDNet(num_classes=raw[1][0].shape[1], if_ddm=if_ddm, use_regression=use_regression,
                                    test_cfg=dict(rotate_degrees=sorted(set(rots), key=rots.index),
                                                  flip_directions=sorted(set(flips), key=flips.index)))
    tcp, sem_cls, dir_map, tc_cls = seg.inference_tail(*raw, ori_hw=(h, w))         # (the goldens' lists are rots x flips)
    _same(dict(tc_prob=tcp, sem_cls=sem_cls, dir_map=dir_map, tc_cls=tc_cls),
          {k: r[k] for k in ("tc_prob", "sem_cls", "dir_map", "tc_cls")}, "MultiTaskCDNet.inference_tail %s%d" % (prefix, j))


def test_mtcdnet_refine_tta_matches_reference_source_golden():
    """r2_ref.npz m*: MultiTaskCDNet.inference executed from source with rotations and flips, fed raw."""
    m = np.load(os.path.join(G, "r2_ref.npz"))
    for j in range(3):
        _mt_golden(m, "m", j, False)


def test_mtcdnet_regression_refine_tta_matches_reference_source_golden():
    """reg_ref.npz g*: the angle head of use_regression = True, fed raw."""
    m = np.load(os.path.join(G, "reg_ref.npz"))
    for j in range(int(m["n_cases"])):
        _mt_golden(m, "g", j, True)


# --------------------------------------------------------------------------- 3. windows and the segmentor API
def test_windows_cut_from_a_whole_variant_equal_whole_inference():
    """Window tensors cut from a full variant image (as split_inference cuts them, base.py:255-295) give the bits of whole
    inference on that image."""
    import torch
    rng = np.random.default_rng(11)
    window, overlap = 32, 8
    st = window - overlap
    pairs = PAIRS[4:12]
    rots, flips = [p[0] for p in pairs], [p[1] for p in pairs]
    whole, cut = [], []
    for C in (3, 9, 1):
        wh, cu = [], []
        for r, f in pairs:
            Ht, Wt = (W, H) if (r // 90) % 2 else (H, W)
            x = (rng.standard_normal((N, C, Ht, Wt)) * 3).astype(np.float32)
            pad_h = st - (Ht - window) % st if Ht - window > 0 else window - Ht
            pad_w = st - (Wt - window) % st if Wt - window > 0 else window - Wt
            H1, W1 = Ht + pad_h, Wt + pad_w
            canvas = np.zeros((N, C, H1, W1), np.float32)
            canvas[:, :, (H1 - Ht) // 2:(H1 - Ht) // 2 + Ht, (W1 - Wt) // 2:(W1 - Wt) // 2 + Wt] = x
            wins = [canvas[:, :, i:i + window, j:j + window] for i in range(0, H1 - overlap, st) for j in range(0, W1 - overlap, st)]
            wh.append(torch.from_numpy(x).cuda())
            cu.append(torch.from_numpy(np.ascontiguousarray(np.stack(wins, axis=1))).cuda())
        whole.append(wh)
        cut.append(cu)
    a = ops.cdnet_refine_tta(*whole, rots, flips, (H, W), if_ddm=True)
    b = ops.cdnet_refine_tta(*cut, rots, flips, (H, W), window, overlap, if_ddm=True)
    _same(b, a, "windows cut from whole variants")


def test_segmentor_inference_tails_with_ori_hw():
    import torch
    rng = np.random.default_rng(12)
    rot_cfg, flip_cfg = [0, 90], FLIPS
    pairs = [(r, f) for r in rot_cfg for f in flip_cfg]             # _tta_lists: rotate_degrees outer, flips inner
    rots, flips = [p[0] for p in pairs], [p[1] for p in pairs]
    for window, overlap in ((0, 0), (32, 8)):
        cd = [[torch.from_numpy(v).cuda() for v in _head(rng, C, pairs, window, overlap, torch.float32)[0]] for C in (3, 9, 1)]
        seg = segmentors.CDNet(num_classes=2, test_cfg=dict(rotate_degrees=rot_cfg, flip_directions=flip_cfg, if_ddm=True))
        prob, dir_map, cls = seg.inference_tail(*cd, ori_hw=(H, W), window=window, overlap=overlap)
        want = ops.cdnet_refine_tta(*cd, rots, flips, (H, W), window, overlap, if_ddm=True)
        _same(dict(sem_prob=prob, dir_map=dir_map, cls=cls), {k: want[k] for k in ("sem_prob", "dir_map", "cls")}, "CDNet")
        for use_regression in (False, True):
            D = 1 if use_regression else 9
            mt = [[torch.from_numpy(v).cuda() for v in _head(rng, C, pairs, window, overlap, torch.float32)[0]] for C in (3, 4, D, 1)]
            seg = segmentors.MultiTaskCDNet(num_classes=4, if_ddm=True, use_regression=use_regression,
                                            test_cfg=dict(rotate_degrees=rot_cfg, flip_directions=flip_cfg))
            tcp, sem_cls, dmap, tc_cls = seg.inference_tail(*mt, ori_hw=(H, W), window=window, overlap=overlap)
            want = ops.mtcdnet_refine_tta(*mt, rots, flips, (H, W), window, overlap, if_ddm=True)
            _same(dict(tc_prob=tcp, sem_cls=sem_cls, dir_map=dmap, tc_cls=tc_cls),
                  {k: want[k] for k in ("tc_prob", "sem_cls", "dir_map", "tc_cls")}, "MultiTaskCDNet reg=%s" % use_regression)
            with pytest.raises(ValueError):
                segmentors.MultiTaskCDNet(num_classes=4, use_regression=not use_regression,
                                          test_cfg=dict(rotate_degrees=rot_cfg, flip_directions=flip_cfg)).inference_tail(
                    *mt, ori_hw=(H, W), window=window, overlap=overlap)
