"""CPU suite: the oracle against the golden vectors produced by the reference's own code
(tests/golden/make_golden.py) and against independent scipy implementations."""
import hashlib
import os

import numpy as np
import pytest
from scipy import ndimage as ndi

from oracle import metrics as om
from oracle import postprocess as opp
from oracle import skimage_port as sk

G = os.path.join(os.path.dirname(__file__), "golden")
import sys
sys.path.insert(0, os.path.dirname(__file__))


@pytest.fixture(scope="module")
def mref():
    return np.load(os.path.join(G, "metrics_ref.npz"))


def _cases(mref):
    return ["c%d" % i for i in range(int(mref["n_cases"]))]


def test_bin_aji_pq_match_reference(mref):
    for n in _cases(mref):
        p, g = mref[n + "_pred"], mref[n + "_gt"]
        for literal in (True, False):
            aji = om.pre_eval_bin_aji(p, g, literal=literal)
            pq = om.pre_eval_bin_pq(p, g, literal=literal)
            assert tuple(np.float64(aji)) == tuple(mref[n + "_bin_aji"]), n
            assert tuple(np.float64(pq)) == tuple(mref[n + "_bin_pq"]), n


def test_multiclass_aji_pq_match_reference(mref):
    C = 4
    for n in _cases(mref):
        p, g = mref[n + "_pred"], mref[n + "_gt"]
        ps, gs = mref[n + "_pred_sem"], mref[n + "_gt_sem"]
        rp, rg = om.re_instance(p), om.re_instance(g)
        assert np.array_equal(rp, mref[n + "_re_pred"]) and rp.dtype == np.int32
        dp = om.assign_sem_class_to_insts(rp, ps, C)
        dg = om.assign_sem_class_to_insts(rg, gs, C)
        flat = np.array([(c, i) for c, ids in dp.items() for i in ids], np.int64).reshape(-1, 2)
        assert np.array_equal(flat, mref[n + "_cls_pred"]), n
        aji = np.stack(om.pre_eval_aji(rp, rg, dp, dg, C, literal=False))
        pq = np.stack(om.pre_eval_pq(rp, rg, dp, dg, C, literal=False))
        assert np.array_equal(aji, mref[n + "_aji"]), n
        assert np.array_equal(pq, mref[n + "_pq"]), n


def test_semantic_counts_match_reference(mref):
    for n in _cases(mref):
        res = np.stack(om.pre_eval_all_semantic_metric(mref[n + "_pred_sem"], mref[n + "_gt_sem"], 4))
        assert np.array_equal(res, mref[n + "_sem"]), n
    res = np.stack(om.pre_eval_all_semantic_metric(mref["c0_pred_sem"], mref["ign_gt_sem"], 4))
    assert np.array_equal(res, mref["ign_sem"])


def test_align_foreground_matches_numba_reference():
    o = np.load(os.path.join(G, "ordered_ref.npz"))
    for j in range(3):
        for key, t in (("out", 20), ("out5", 5)):
            got = sk.align_foreground(o["af%d_seed" % j].copy(), o["af%d_fg" % j], t)
            assert np.array_equal(got, o["af%d_%s" % (j, key)])


def test_ddm_matches_torch_reference():
    o = np.load(os.path.join(G, "ordered_ref.npz"))
    for j in range(3):
        got = opp.direction_differential_map(o["dd%d_dir" % j], 9)
        assert np.array_equal(got, o["dd%d_out" % j])
    assert np.array_equal(opp.direction_differential_map(np.zeros((16, 16), np.int64), 9), o["dd_zero_out"])


# ----------------------------------------------------------------- C restatement vs scipy
def _canon(lab):
    flat = lab.ravel()
    nz = flat > 0
    if not nz.any():
        return lab.astype(np.int64)
    vals, first = np.unique(flat[nz], return_index=True)
    lut = np.zeros(int(flat.max()) + 1, np.int64)
    lut[flat[nz][np.sort(first)]] = np.arange(1, len(vals) + 1)
    return lut[lab]


@pytest.mark.parametrize("conn", [1, 2])
def test_label_binary_matches_scipy(conn):
    rng = np.random.default_rng(conn)
    for shape in [(1, 1), (1, 17), (23, 1), (37, 41), (64, 64)]:
        for dens in (0.2, 0.5, 0.7):
            m = rng.random(shape) < dens
            ref, k = ndi.label(m, ndi.generate_binary_structure(2, conn))
            got, kk = sk.label(m, connectivity=conn, return_num=True)
            assert kk == k and np.array_equal(got, ref)


def test_label_equal_value_and_background():
    rng = np.random.default_rng(5)
    img = rng.integers(0, 4, (40, 50))
    for bg in (0, 2):
        got = sk.label(img, background=bg)
        comp = np.zeros(img.shape, np.int64)
        nxt = 0
        for v in np.unique(img):
            if v == bg:
                continue
            lab, k = ndi.label(img == v, np.ones((3, 3)))
            comp[lab > 0] = lab[lab > 0] + nxt
            nxt += k
        assert np.array_equal(got, _canon(comp))


def test_reconstruction_erosion_fixed_point():
    rng = np.random.default_rng(3)
    x = rng.integers(0, 256, (30, 33)).astype(np.float64)
    seed = np.minimum(255, x + 7)
    r = seed.copy()
    for _ in range(200):
        n = np.maximum(ndi.grey_erosion(r, size=(3, 3)), x)
        if np.array_equal(n, r):
            break
        r = n
    assert np.array_equal(sk.reconstruction_erosion(seed, x), r)


def test_regional_minima_identity():
    """find_maxima (dist.py:60-71) == 8-connected regional-minimum plateaus with value < 255."""
    rng = np.random.default_rng(4)
    x = ndi.uniform_filter(rng.integers(0, 256, (60, 70)).astype(np.float64), 5).astype(np.uint8)
    x[:5] = 255
    res = opp._find_maxima(x, np.ones_like(x), literal=False)
    plate = sk.label(x.astype(np.int64) + 1, background=-1)
    mn = ndi.grey_erosion(x, size=(3, 3))
    has_lower = ndi.maximum(mn < x, plate, np.arange(1, plate.max() + 1)).astype(bool)
    expect = (~has_lower[plate - 1]) & (x < 255)
    assert np.array_equal(res.astype(bool), expect)


def test_watershed_known_answers():
    # two seeds on a flat image: BFS rings, ties resolved by (value, age): seed with lower index first
    img = np.zeros((1, 7))
    mk = np.zeros((1, 7), np.int32); mk[0, 0] = 1; mk[0, 6] = 2
    assert sk.watershed(img, mk).tolist() == [[1, 1, 1, 1, 2, 2, 2]]
    # a ridge keeps basins apart until both sides are flooded
    img = np.array([[0, 1, 2, 9, 2, 1, 0]], np.float64)
    assert sk.watershed(img, mk).tolist() == [[1, 1, 1, 1, 2, 2, 2]]
    # mask stops the flood, markers outside the mask are dropped
    msk = np.array([[1, 1, 0, 1, 1, 1, 0]], np.uint8)
    assert sk.watershed(img, mk, msk).tolist() == [[1, 1, 0, 0, 0, 0, 0]]


def test_literal_and_fast_dist_agree():
    import tiseg_b200  # noqa: F401
    from tiseg_b200 import synth
    t = synth.tile_dist(2, 3, H=120, W=130)
    sp = opp.argmax_classes(opp.softmax(t["sem_logit"]))
    a = opp.dist_postprocess(sp, t["dist_logit"], literal=True)[1]
    b = opp.dist_postprocess(sp, t["dist_logit"], literal=False)[1]
    assert np.array_equal(a, b) and a.max() > 3


def test_opencv_recipes_are_bit_exact():
    """The arithmetic order the HoVer kernels implement (tests/cv_recipes.py) reproduces cv2 bit for bit
    (normalize on fp32 input, Sobel ksize 21 -> CV_64F, GaussianBlur 3x3 on fp64, 5x5 ellipse)."""
    cv2 = pytest.importorskip("cv2")
    import tiseg_b200  # noqa: F401
    from tiseg_b200 import synth
    import cv_recipes as R
    assert np.array_equal(cv2.getStructuringElement(cv2.MORPH_ELLIPSE, (5, 5)), R.ELLIPSE5)
    d, sm = R.deriv_kernels_21()
    kd, ks = cv2.getDerivKernels(1, 0, 21)
    assert np.array_equal(kd.ravel(), d) and np.array_equal(ks.ravel(), sm)
    for seed, (H, W) in enumerate([(48, 48), (64, 100), (250, 131)]):
        t = synth.tile_hover(3, 50 + seed, H=H, W=W)
        for ch in range(2):
            x = np.ascontiguousarray(t["hv_map"][:, :, ch])
            n = cv2.normalize(x, None, alpha=0, beta=1, norm_type=cv2.NORM_MINMAX, dtype=cv2.CV_32F)
            assert np.array_equal(R.normalize_minmax_f32(x), n)
            s = cv2.Sobel(n, cv2.CV_64F, 1 - ch, ch, ksize=21)
            assert np.array_equal(R.sobel21(n, 1 - ch, ch), s)
            assert np.array_equal(R.gaussian_blur3(s), cv2.GaussianBlur(s, (3, 3), 0))
            # fp64 -> fp32 normalize contracts x*a+b into one FMA inside OpenCV; without FMA at most a few
            # pixels next to the minimum differ in the last bit
            sn = cv2.normalize(s, None, alpha=0, beta=1, norm_type=cv2.NORM_MINMAX, dtype=cv2.CV_32F)
            assert (R.normalize_minmax_f32(s) != sn).sum() <= 4


def test_opencv_resize_x2_recipe_is_bit_exact():
    """cv2.resize(x, (0, 0), fx=2, fy=2) of hover_post_proc with scale_factor = 2 (the CoNIC config), and the
    INTER_NEAREST way back: the arithmetic the k_resize_up2 / k_resize_down2_nearest kernels implement."""
    cv2 = pytest.importorskip("cv2")
    import cv_recipes as R
    rng = np.random.default_rng(77)
    for (H, W) in [(1, 1), (1, 5), (3, 1), (2, 2), (7, 9), (64, 64), (100, 131), (256, 256)]:
        x = (rng.standard_normal((H, W)) * 3).astype(np.float32)
        assert np.array_equal(R.resize_up2_linear(x), cv2.resize(x, (0, 0), fx=2, fy=2)), (H, W)
        hv = (rng.random((H, W, 2)) * 2 - 1).astype(np.float32)
        assert np.array_equal(R.resize_up2_linear(hv), cv2.resize(hv, (0, 0), fx=2, fy=2)), (H, W)
        lab = rng.integers(0, 1000, (2 * H, 2 * W)).astype(np.int32)
        assert np.array_equal(cv2.resize(lab, (W, H), interpolation=cv2.INTER_NEAREST), lab[::2, ::2])


def test_mudslide_watershed_matches_numba_reference():
    """oracle mudslide_watershed == the reference's numba get_graph_degree / prepare / mudslide_watershed
    (tests/golden/mudslide_ref.npz, made by tests/golden/make_golden.py from the reference's own file)."""
    m = np.load(os.path.join(G, "mudslide_ref.npz"))
    for j in range(5):
        d = m["m%d_dir" % j].copy()
        pred, boundary = opp.mudslide_watershed(m["m%d_seg" % j].copy(), d, m["m%d_fore" % j].copy())
        assert np.array_equal(pred, m["m%d_pred" % j]) and np.array_equal(boundary, m["m%d_boundary" % j])
        assert np.array_equal(d, m["m%d_dir_after" % j])


def test_label_generation_matches_reference():
    """oracle gen_instance_hv_map / fix_inst + instance_distance_map == datasets/ops/hv_map.py and
    datasets/ops/distance_map.py (DistanceLabelMake) run from the reference's own files (labelgen_ref.npz)."""
    m = np.load(os.path.join(G, "labelgen_ref.npz"))
    for j in range(5):
        inst = m["l%d_inst" % j]
        assert np.array_equal(opp.gen_instance_hv_map(inst), m["l%d_hv" % j])
        fixed = opp.fix_inst(inst)
        for norm in (0, 1):
            assert np.array_equal(opp.instance_distance_map(fixed, bool(norm)), m["l%d_dist%d" % (j, norm)])
        assert np.array_equal(fixed, m["l%d_fixed" % j])
        for tag, radius in (("1", (1, 1)), ("3", (3, 3)), ("21", (2, 1))):
            sem, bound = opp.bound_label(m["l%d_sem" % j], fixed, 4, radius)
            assert np.array_equal(sem, m["l%d_r%s_sem" % (j, tag)])
            assert np.array_equal(bound, m["l%d_r%s_bound" % (j, tag)])
        if j != 2:
            inner, w = opp.unet_weight_map(fixed)
            sem = np.where(fixed == 0, 0, m["l%d_sem" % j])
            assert np.array_equal(np.where(inner == 0, 0, sem), m["l%d_unet_inner" % j])
            assert np.array_equal(w, m["l%d_unet_w" % j])


def test_dist_postprocess_matches_reference_source():
    """oracle dist_postprocess (literal and fast forms) == the reference's own dist.py helpers + DIST.postprocess
    executed from its source text with scikit-image replaced by the port (tests/golden/dist_ref.npz): pins the control
    flow of the restatement."""
    m = np.load(os.path.join(G, "dist_ref.npz"))
    for j in range(4):
        want = m["d%d_out" % j]
        for literal in (True, False):
            got = opp.dist_postprocess(None, m["d%d_in" % j], literal=literal)[1]
            assert np.array_equal(got, want), (j, literal)


def test_segmentor_postprocesses_match_reference_source():
    """oracle restatements == the reference's own method source text (unet.py, cdnet.py, dcan.py, multi_task_*.py,
    hovernet.py) executed with scipy / OpenCV real and scikit-image served by the port (segmentors_ref.npz)."""
    m = np.load(os.path.join(G, "segmentors_ref.npz"))
    for j in range(3):
        sem, inst = opp.unet_family_postprocess(m["u%d_pred" % j].copy(), radius=1)
        assert np.array_equal(sem, m["u%d_sem" % j]) and np.array_equal(inst, m["u%d_inst" % j])
        sem, inst = opp.unet_family_postprocess(m["c%d_pred" % j].copy(), radius=3, edge_id=3)
        assert np.array_equal(sem, m["c%d_sem" % j]) and np.array_equal(inst, m["c%d_inst" % j])
        sem, inst = opp.dcan_postprocess(m["d%d_cell" % j].copy(), m["d%d_cont" % j], radius=3)
        assert np.array_equal(sem, m["d%d_sem" % j]) and np.array_equal(inst, m["d%d_inst" % j])
        for variant, first in (("unet", "inner"), ("cunet", "tc"), ("cdnet", "tc")):
            sem, inst = opp.multitask_postprocess(m["m%d_%s" % (j, first)].copy(), m["m%d_sempred" % j].copy(), variant)
            assert np.array_equal(sem, m["m%d_%s_sem" % (j, variant)]), (j, variant)
            assert np.array_equal(inst, m["m%d_%s_inst" % (j, variant)]), (j, variant)
        out = opp.hover_post_proc(m["h%d_fore" % j].copy(), m["h%d_hv" % j].copy(), fx=1, scale_factor=int(m["h%d_sf" % j]))[0]
        assert np.array_equal(out, m["h%d_out" % j])


def test_dataset_evaluate_matches_reference_source():
    """tiseg_b200.datasets.CustomDataset.evaluate (host arithmetic) on the per-image results the reference's own
    pre_eval produced == the reference's own evaluate (custom.py:307-435 executed from source, dataset_ref.npz)."""
    import torch
    from tiseg_b200 import datasets
    m = np.load(os.path.join(G, "dataset_ref.npz"))
    results = [dict(name=str(m["p%d_name" % j]), bin_aji_pre_eval_res=tuple(m["p%d_bin_aji" % j]),
                    bin_pq_pre_eval_res=tuple(m["p%d_bin_pq" % j]),
                    sem_pre_eval_res=tuple(torch.from_numpy(x) for x in m["p%d_sem" % j])) for j in range(4)]
    ds = datasets.CustomDataset(sem_gts=[None] * 4, inst_gts=[None] * 4, names=["im%d" % j for j in range(4)])
    ev, _ = ds.evaluate(results, logger="silent")
    assert list(ev.keys()) == m["eval_keys"].tolist()
    np.testing.assert_allclose(np.array([float(v) for v in ev.values()]), m["eval_values"], rtol=0, atol=1e-9)


def test_conic_dataset_evaluate_matches_reference_source():
    """CoNICDataset.evaluate on the reference's own per-image results == conic.py:200-323 executed from source (all 67
    entries, including the per-class strings)."""
    import torch
    from tiseg_b200 import datasets
    m = np.load(os.path.join(G, "dataset_ref.npz"))
    results = [dict(bin_aji_pre_eval_res=tuple(m["q%d_bin_aji" % j]), aji_pre_eval_res=tuple(m["q%d_aji" % j]),
                    bin_pq_pre_eval_res=tuple(m["q%d_bin_pq" % j]), pq_pre_eval_res=tuple(m["q%d_pq" % j]),
                    sem_pre_eval_res=tuple(torch.from_numpy(x) for x in m["q%d_sem" % j])) for j in range(3)]
    ds = datasets.CoNICDataset(sem_gts=[None] * 3, inst_gts=[None] * 3)
    ev, _ = ds.evaluate(results, logger="silent")
    assert list(ev.keys()) == m["conic_eval_keys"].tolist()
    assert [isinstance(v, str) for v in ev.values()] == m["conic_eval_isstr"].tolist()
    np.testing.assert_allclose(np.array([float(v) for v in ev.values()]), m["conic_eval_values"], rtol=0, atol=1e-9)


def _tta_case(m, j):
    H, W, window, overlap, C, B, T = (int(v) for v in m["t%d_meta" % j])
    variants = [m["t%d_v%d" % (j, t)].astype(np.float32) / 4.0 for t in range(T)]
    return H, W, window, overlap, B, variants, [int(r) for r in m["t%d_rots" % j]], [str(f) for f in m["t%d_flips" % j]]


def test_tta_stitch_softmax_matches_reference_source():
    """oracle split_stitch + reverse_tta_transform + softmax_tta_mean == BaseSegmentor.inference (base.py:255-381)
    executed from source on recorded window logits (tta_ref.npz); fp32 softmax: 1e-6."""
    m = np.load(os.path.join(G, "tta_ref.npz"))
    for j in range(3):
        H, W, window, overlap, B, variants, rots, flips = _tta_case(m, j)
        for n in range(B):
            rev = []
            for v, r, f in zip(variants, rots, flips):
                Ht, Wt = (W, H) if (r // 90) % 2 else (H, W)
                full = opp.split_stitch(v[n], Ht, Wt, window, overlap) if window else v[n]
                rev.append(opp.reverse_tta_transform(full, r, f))
            np.testing.assert_allclose(opp.softmax_tta_mean(rev), m["t%d_prob" % j][n], rtol=1e-6, atol=1e-7)


def _cdnet_case(m, j):
    flips = [str(f) for f in m["c%d_flips" % j]]
    sem, dirs, pts = [], [], []
    for t, f in enumerate(flips):                      # the recorder saw the logits of the TRANSFORMED image
        sem.append(opp.reverse_tta_transform(m["c%d_sem%d" % (j, t)].astype(np.float32), 0, f))
        dirs.append(opp.reverse_tta_transform(m["c%d_dir%d" % (j, t)].astype(np.float32), 0, f))
        pts.append(opp.reverse_tta_transform(m["c%d_pt%d" % (j, t)].astype(np.float32), 0, f))
    return sem, dirs, pts, bool(m["c%d_if_ddm" % j])


def test_cdnet_inference_tail_matches_reference_source():
    """oracle cdnet_inference_tail == CDNet.inference + _ddm_enhencement executed from source (tta_ref.npz)."""
    m = np.load(os.path.join(G, "tta_ref.npz"))
    for j in range(2):
        sem, dirs, pts, if_ddm = _cdnet_case(m, j)
        got_sem, got_dir, _ = opp.cdnet_inference_tail(sem, dirs, pts, if_ddm=if_ddm)
        assert np.array_equal(got_dir, m["c%d_dir_out" % j])
        np.testing.assert_allclose(got_sem, m["c%d_sem_out" % j], rtol=1e-5, atol=1e-7)


def test_monuseg_debug_evaluate_matches_reference_source():
    """MoNuSegDatasetDebug.evaluate (boundary-class metrics on top of CustomDataset's) on the reference's own per-image
    results == monuseg_debug.py executed from source."""
    import torch
    from tiseg_b200 import datasets
    m = np.load(os.path.join(G, "dataset_ref.npz"))
    results = [dict(name=str(m["d%d_name" % j]), bin_aji_pre_eval_res=tuple(m["d%d_bin_aji" % j]),
                    bin_pq_pre_eval_res=tuple(m["d%d_bin_pq" % j]),
                    bound_sem_pre_eval_res=tuple(torch.from_numpy(x) for x in m["d%d_bound" % j]),
                    sem_pre_eval_res=tuple(torch.from_numpy(x) for x in m["d%d_sem" % j])) for j in range(2)]
    ds = datasets.MoNuSegDatasetDebug(sem_gts=[None] * 2, inst_gts=[None] * 2, names=["m0", "m1"])
    ev, _ = ds.evaluate(results, logger="silent")
    assert list(ev.keys()) == m["monuseg_eval_keys"].tolist()
    np.testing.assert_allclose(np.array([float(v) for v in ev.values()]), m["monuseg_eval_values"], rtol=0, atol=1e-9)


# --------------------------------------------------------------------------- round-2 vectors (r2_ref.npz)
def _r2():
    return np.load(os.path.join(G, "r2_ref.npz"))


def _mt_case(m, j):
    T = len(m["m%d_flips" % j])
    f32 = lambda key: [m["m%d_%s%d" % (j, key, t)].astype(np.float32) for t in range(T)]
    return f32("tc"), f32("sem"), f32("dir"), f32("pt"), bool(m["m%d_if_ddm" % j]), list(m["m%d_rots" % j]), list(m["m%d_flips" % j])


def test_oracle_mtcdnet_tail_matches_reference_source():
    """The restatement of MultiTaskCDNet.inference's tail vs the method executed from source (recorder network)."""
    m = _r2()
    for j in range(3):
        tc, sem, dirs, pts, if_ddm, rots, flips = _mt_case(m, j)
        rev = lambda lst: [opp.reverse_tta_transform(x, int(r), str(f)) for x, r, f in zip(lst, rots, flips)]
        got_tc, got_sem, got_dir, _ = opp.mtcdnet_inference_tail(rev(tc), rev(sem), rev(dirs), rev(pts), if_ddm)
        np.testing.assert_allclose(got_tc, m["m%d_tc_out" % j], rtol=1e-5, atol=1e-7)
        np.testing.assert_allclose(got_sem, m["m%d_sem_out" % j], rtol=1e-5, atol=1e-7)
        assert (got_dir != m["m%d_dir_out" % j]).mean() < 1e-3          # argmax of fp32 products: libm-level ties only


def test_oracle_ddm_enhancement_both_variants():
    m = _r2()
    for j in range(2):
        for key, mode in (("cdnet", 0), ("mtcdnet", 1)):
            got = opp.ddm_enhancement(m["e%d_prob" % j][0], m["e%d_dd" % j][0], m["e%d_pt" % j][0, 0], mode)
            assert np.array_equal(got, m["e%d_%s" % (j, key)][0]), (j, key)


def _reg_inputs(m, name, j):
    """The head outputs make_golden_r2.py's recorder network fed DIST.inference ("d") / HoverNet.inference ("h"), drawn
    again from its seed in its order (per TTA variant: ``calls`` patches, the whole image or split windows; per patch:
    the heads).  The stored digest pins them to what the reference was run on.  -> [head][variant] int8 quarter units"""
    H, W, window, overlap, T = [int(v) for v in m["%s%d_meta" % (name, j)]]
    rots = [int(r) for r in m["%s%d_rots" % (name, j)]]
    chans = (2, 1) if name == "d" else (3, 2, 2)
    rng = np.random.default_rng(9840 + 10 * j + len(chans))
    out = [[] for _ in chans]
    for t in range(T):
        ph, pw = (window, window) if window else ((W, H) if (rots[t] // 90) % 2 else (H, W))
        calls = [[rng.integers(-12, 13, (1, c, ph, pw)).astype(np.int8) for c in chans]
                 for _ in range(int(m["%s%d_calls" % (name, j)]))]
        for h in range(len(chans)):
            w = np.stack([c[h] for c in calls])                                 # [M, 1, C, h, w]
            out[h].append(np.ascontiguousarray(np.moveaxis(w, 1, 0)) if window else w[0])
    digest = hashlib.sha256(b"".join(v.tobytes() for head in out for v in head)).hexdigest()
    assert digest == str(m["%s%d_sha256" % (name, j)]), "%s%d: the seeded draw no longer gives the golden inputs" % (name, j)
    return out


def _reg_case(m, name, j, h):
    H, W, window, overlap, T = [int(v) for v in m["%s%d_meta" % (name, j)]]
    variants = [v.astype(np.float32) / 4.0 for v in _reg_inputs(m, name, j)[h]]
    return H, W, window, overlap, variants, [int(r) for r in m["%s%d_rots" % (name, j)]], [str(f) for f in m["%s%d_flips" % (name, j)]]


def test_oracle_regression_head_tta_mean():
    """dist.py:398-406 (plain mean of the reversed distance maps) and hovernet.py:406 (variant 0 only), from source."""
    m = _r2()
    for j in range(3):
        for name, h, first_only in (("d", 1, False), ("h", 1, True)):
            H, W, window, overlap, variants, rots, flips = _reg_case(m, name, j, h)
            rev = []
            for v, r, f in zip(variants, rots, flips):
                Ht, Wt = (W, H) if (r // 90) % 2 else (H, W)
                full = opp.split_stitch(v[0], Ht, Wt, window, overlap) if window else v[0]
                rev.append(opp.reverse_tta_transform(full, r, f))
            want = m["%s%d_out%d" % (name, j, h)][0]
            got = rev[0] if first_only else opp.tta_plain_mean(rev)
            assert np.array_equal(got, want), (name, j)


def test_oracle_three_class_gt():
    m = _r2()
    for j in range(3):
        assert np.array_equal(opp.three_class_gt(m["g%d_wb" % j], int(m["g%d_nc" % j])), m["g%d_tc" % j])


def _id_dict(m, n, side):
    keys, lens, ids = m[n + "_" + side + "_keys"], m[n + "_" + side + "_lens"], m[n + "_" + side + "_ids"]
    out, o = {}, 0
    for k, l in zip(keys, lens):
        out[int(k)] = [int(v) for v in ids[o:o + l]]
        o += int(l)
    return out


def test_oracle_pre_eval_with_id_dictionaries_and_match_iou():
    """pre_eval_aji / pre_eval_pq called the way conic.py:178-188 calls them, and pre_eval_bin_pq(match_iou > 0.5)."""
    m = _r2()
    for k in range(int(m["n_pair_cases"])):
        n = "p%d" % k
        ip, ig = m[n + "_ip"], m[n + "_ig"]
        dp, dg = _id_dict(m, n, "dp"), _id_dict(m, n, "dg")
        for rz in (True, False):
            got = np.stack(om.pre_eval_aji(ip, ig, dp, dg, 4, reduce_zero_label=rz, literal=False))
            assert np.array_equal(got, m[n + "_aji_rz%d" % rz]), (n, rz)
            got = np.stack(om.pre_eval_pq(ip, ig, dp, dg, 4, reduce_zero_label=rz, literal=False))
            assert np.array_equal(got, m[n + "_pq_rz%d" % rz]), (n, rz)
        for mi in (0.5, 0.6, 0.75, 0.9):
            got = np.array(om.pre_eval_bin_pq(ip, ig, mi, literal=False), np.float64)
            assert np.array_equal(got, m[n + "_binpq_%d" % int(mi * 100)]), (n, mi)



def test_direction_label_make_oracle_vs_reference_golden():
    """oracle.postprocess.direction_label_make against DirectionLabelMake run from the reference's own files
    (tests/golden/make_golden_dir.py, both to_center settings, 4 / 8 / 16 angles): everything that does not pass through the
    float32 convolution is identical (fixed instances, sem_gt, centre points via point_gt, dist_gt); the angle-derived maps
    agree except on a handful of pixels whose gradient component is ~0 (sign of zero decides 0 vs 360 degrees)."""
    g = np.load(os.path.join(G, "dirlabel_ref.npz"))
    for j in range(int(g["n_cases"])):
        p = "d%d_" % j
        A, to_center = int(g[p + "num_angles"]), bool(g[p + "to_center"])
        r = opp.direction_label_make(g[p + "inst"], g[p + "sem"], A, to_center)
        assert np.array_equal(r["inst_gt"], g[p + "fixed"]) and np.array_equal(r["sem_gt"], g[p + "sem_gt"])
        assert np.array_equal(r["dist_gt"], g[p + "dist_gt"]) and r["dist_gt"].dtype == g[p + "dist_gt"].dtype
        assert np.array_equal(r["point_gt"], g[p + "point_gt"])
        fg = int((g[p + "fixed"] > 0).sum())
        assert int((r["dir_gt"] != g[p + "dir_gt"]).sum()) <= max(4, fg // 100)
        d = np.abs(r["reg_dir_gt"].astype(np.float64) - g[p + "reg_dir_gt"])
        d = np.minimum(d, 2 * np.pi - d)
        assert (d > 2e-4).sum() <= max(4, fg // 100)
        assert r["loss_weight_map"].dtype == g[p + "loss_weight_map"].dtype


def _regr_case(m, j):
    T = len(m["g%d_flips" % j])
    f32 = lambda key: [m["g%d_%s%d" % (j, key, t)].astype(np.float32) for t in range(T)]
    return f32("tc"), f32("sem"), f32("dir"), f32("pt"), bool(m["g%d_if_ddm" % j]), list(m["g%d_rots" % j]), list(m["g%d_flips" % j])


def test_oracle_mtcdnet_regression_tail_matches_reference_source():
    """use_regression = True (multi_task_cdnet.py:304-315) vs the method executed from source (make_golden_reg.py): the
    angle head is clamped, binned into eight classes and fed to the same DDM + enhancement; angles exactly on class edges
    and outside [0, 2 pi] are part of the vectors, so the class map must be identical."""
    m = np.load(os.path.join(G, "reg_ref.npz"))
    for j in range(int(m["n_cases"])):
        tc, sem, dirs, pts, if_ddm, rots, flips = _regr_case(m, j)
        rev = lambda lst: [opp.reverse_tta_transform(x, int(r), str(f)) for x, r, f in zip(lst, rots, flips)]
        got_tc, got_sem, got_dir, _ = opp.mtcdnet_inference_tail(rev(tc), rev(sem), rev(dirs), rev(pts), if_ddm, use_regression=True)
        assert np.array_equal(got_dir, m["g%d_dir_out" % j]), j
        np.testing.assert_allclose(got_tc, m["g%d_tc_out" % j], rtol=1e-5, atol=1e-7)
        np.testing.assert_allclose(got_sem, m["g%d_sem_out" % j], rtol=1e-5, atol=1e-7)
