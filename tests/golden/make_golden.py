"""Generate ``tests/golden/*.npz`` by running the REFERENCE's own code (authoring container only).

Imports, by file path, the parts of /root/reference that load in this image:
  tiseg/utils/misc.py + tiseg/utils/inst_metrics.py     (stub ``mmcv``; ``skimage.measure.label``
                                                          replaced by an independent scipy-based
                                                          labelling, since scikit-image is absent)
  tiseg/utils/sem_metrics.py                             (stub ``mmcv``; real torch.histc)
  tiseg/datasets/utils/instance_semantic.py              (stub ``skimage.morphology``)
  tiseg/models/utils/postprocess.py                      (numba align_foreground)
  tiseg/models/utils/direct_diff_map.py                  (torch, CPU)
  tiseg/datasets/ops/{hv_map,distance_map,bound_map,unet_map}.py   (label makers; skimage morphology served by scipy)
and stores seeded inputs together with the reference outputs.  Code that cannot be imported (it lives in modules that
pull in mmcv / the model zoo) is executed FROM ITS SOURCE TEXT instead: the function or method is cut out of the
reference file with ``ast`` and run in a namespace where scipy / OpenCV / torch are the real libraries, scikit-image
calls are served by the oracle's port (``oracle/skimage_port``: this pins control flow, not scikit-image) and ``self``
is a small namespace carrying the attributes the method reads:
  tiseg/models/segmentors/dist.py        helpers :31-131 + DIST.postprocess                      -> dist_ref.npz
  tiseg/models/segmentors/{unet,cdnet,dcan,multi_task_*,hovernet}.py   .postprocess / .hover_post_proc -> segmentors_ref.npz
  tiseg/models/segmentors/base.py        BaseSegmentor.inference (+ split/whole, TTA transforms)  -> tta_ref.npz
  tiseg/models/segmentors/cdnet.py       CDNet.inference tail + _ddm_enhencement                  -> tta_ref.npz
  tiseg/datasets/{custom,monuseg_debug,conic}.py   pre_eval + evaluate (GT files in a temp dir)   -> dataset_ref.npz
/root/reference does not exist on the GPU box, so the tests only read the committed .npz files.

    python tests/golden/make_golden.py
"""
import importlib.util
import os
import sys
import types

import numpy as np
from scipy import ndimage as ndi

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))


def scipy_label(img, background=0, connectivity=None, return_num=False):
    """Independent stand-in for skimage.measure.label: per value, scipy binary labelling, then ids
    renumbered in raster order of first pixel."""
    img = np.asarray(img)
    st = ndi.generate_binary_structure(2, 2 if connectivity in (None, 2) else 1)
    comp = np.zeros(img.shape, np.int64)
    nxt = 0
    for v in np.unique(img):
        if v == background:
            continue
        lab, k = ndi.label(img == v, st)
        comp[lab > 0] = lab[lab > 0] + nxt
        nxt += k
    flat = comp.ravel()
    nz = flat > 0
    _, first = np.unique(flat[nz], return_index=True)
    order = flat[nz][np.sort(first)]
    lut = np.zeros(nxt + 1, np.int64)
    lut[order] = np.arange(1, len(order) + 1)
    out = lut[comp]
    return (out, len(order)) if return_num else out


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def _opp_mod():
    from oracle import postprocess as _opp
    return _opp


def load_reference():
    _stub("mmcv")
    sk = _stub("skimage")
    sk.measure = _stub("skimage.measure", label=scipy_label)
    from oracle import postprocess as _opp          # scikit-image is absent: mudslide_watershed's remove_small_objects
    sk.morphology = _stub("skimage.morphology", remove_small_objects=_opp.remove_small_objects)
    pkg = types.ModuleType("refutils")
    pkg.__path__ = [os.path.join(REF, "tiseg", "utils")]
    sys.modules["refutils"] = pkg

    def load(modname, path, package=None):
        spec = importlib.util.spec_from_file_location(modname, path)
        mod = importlib.util.module_from_spec(spec)
        if package:
            mod.__package__ = package
        sys.modules[modname] = mod
        spec.loader.exec_module(mod)
        return mod

    misc = load("refutils.misc", os.path.join(REF, "tiseg/utils/misc.py"), "refutils")
    inst = load("refutils.inst_metrics", os.path.join(REF, "tiseg/utils/inst_metrics.py"), "refutils")
    sem = load("refutils.sem_metrics", os.path.join(REF, "tiseg/utils/sem_metrics.py"), "refutils")
    isem = load("ref_instance_semantic", os.path.join(REF, "tiseg/datasets/utils/instance_semantic.py"))
    pp = load("ref_postprocess", os.path.join(REF, "tiseg/models/utils/postprocess.py"))
    ddm = load("ref_ddm", os.path.join(REF, "tiseg/models/utils/direct_diff_map.py"))
    return misc, inst, sem, isem, pp, ddm


def main():
    import tiseg_b200  # noqa: F401
    from tiseg_b200 import synth

    misc, inst, sem, isem, pp, ddm = load_reference()
    inst_mod, sem_mod = inst, sem                       # (the names inst / sem are reused for arrays further down)
    import torch

    # ---- instance metrics (binary) on seeded synthetic pairs + hand-made edge cases
    cases = {}
    shapes = [(64, 80), (96, 96), (128, 100), (256, 256)]
    k = 0
    for si, (H, W) in enumerate(shapes):
        for j in range(3):
            t = synth.gt_and_pred(9000 + 10 * si + j, H, W, n=max(3, H * W // 900), num_classes=4)
            cases["c%d" % k] = (t["pred_inst"], t["gt_inst"], t["pred_sem"], t["gt_sem"])
            k += 1
    z = np.zeros((32, 32), np.int32)
    a = z.copy(); a[4:12, 4:12] = 1; a[20:28, 20:30] = 7
    b = z.copy(); b[6:14, 6:14] = 3; b[20:28, 18:26] = 3      # one pred id, two components
    cases["c%d" % k] = (a, b, (a > 0).astype(np.uint8), (b > 0).astype(np.uint8)); k += 1
    cases["c%d" % k] = (z, b, z.astype(np.uint8), (b > 0).astype(np.uint8)); k += 1      # empty pred
    cases["c%d" % k] = (a, z, (a > 0).astype(np.uint8), z.astype(np.uint8)); k += 1      # empty gt
    d1 = z.copy(); d1[5, 5] = 1; d1[6, 6] = 1; d1[10:14, 10:14] = 2; d1[14:18, 14:18] = 2  # diagonal touches
    cases["c%d" % k] = (d1, a, (d1 > 0).astype(np.uint8), (a > 0).astype(np.uint8)); k += 1

    out = {}
    for name, (p, g, ps, gs) in cases.items():
        out[name + "_pred"] = p.astype(np.int32)
        out[name + "_gt"] = g.astype(np.int32)
        out[name + "_pred_sem"] = ps.astype(np.uint8)
        out[name + "_gt_sem"] = gs.astype(np.uint8)
        aji = inst.pre_eval_bin_aji(p, g)
        pq = inst.pre_eval_bin_pq(p, g)
        out[name + "_bin_aji"] = np.array(aji, np.float64)
        out[name + "_bin_pq"] = np.array(pq, np.float64)
        # multi-class (CoNIC path): re_instance -> assign classes -> pre_eval_aji / pre_eval_pq
        C = 4
        rp, rg = isem.re_instance(p), isem.re_instance(g)
        out[name + "_re_pred"] = rp
        dp = isem.assign_sem_class_to_insts(rp, ps, C)
        dg = isem.assign_sem_class_to_insts(rg, gs, C)
        # flatten dicts as (class, id) rows in dict order
        out[name + "_cls_pred"] = np.array([(c, i) for c, ids in dp.items() for i in ids], np.int64).reshape(-1, 2)
        out[name + "_cls_gt"] = np.array([(c, i) for c, ids in dg.items() for i in ids], np.int64).reshape(-1, 2)
        out[name + "_aji"] = np.stack(inst.pre_eval_aji(rp, rg, dp, dg, C))
        out[name + "_pq"] = np.stack(inst.pre_eval_pq(rp, rg, dp, dg, C))
        sres = sem.pre_eval_all_semantic_metric(ps, gs, C)
        out[name + "_sem"] = np.stack([x.numpy() for x in sres])
    gs_ign = cases["c0"][3].copy(); gs_ign[:5] = 255
    out["ign_gt_sem"] = gs_ign
    out["ign_sem"] = np.stack([x.numpy() for x in sem.pre_eval_all_semantic_metric(cases["c0"][2], gs_ign, 4)])
    out["n_cases"] = np.array(k)
    np.savez_compressed(os.path.join(HERE, "metrics_ref.npz"), **out)

    # ---- reducers on the list of per-case results
    names = ["c%d" % i for i in range(k)]
    aji_list = [tuple(out[n + "_bin_aji"]) for n in names]
    pq_list = [tuple(out[n + "_bin_pq"]) for n in names]
    sem_list = [tuple(torch.from_numpy(r) for r in out[n + "_sem"]) for n in names]
    red = dict(
        to_aji=np.float64(inst.pre_eval_to_aji(aji_list)["Aji"]),
        to_bin_aji=np.float64(inst.pre_eval_to_bin_aji(aji_list)["Aji"]),
        to_imw_aji=inst.pre_eval_to_imw_aji(aji_list)["Aji"],
        to_pq=np.array([inst.pre_eval_to_pq(pq_list)[m] for m in ("DQ", "SQ", "PQ")]),
        to_bin_pq=np.array([inst.pre_eval_to_bin_pq(pq_list)[m] for m in ("DQ", "SQ", "PQ")]),
        to_imw_pq=np.stack([inst.pre_eval_to_imw_pq(pq_list)[m] for m in ("DQ", "SQ", "PQ")]),
        to_inst_dice=np.float64(inst.pre_eval_to_inst_dice(pq_list)["InstDice"]),
        to_imw_inst_dice=inst.pre_eval_to_imw_inst_dice(pq_list)["InstDice"],
    )
    sm = sem.pre_eval_to_sem_metrics(sem_list, metrics=["Dice", "Precision", "Recall"])
    red.update({"sem_" + m: sm[m] for m in sm})
    im = sem.pre_eval_to_imw_sem_metrics(sem_list, metrics=["Dice", "Precision", "Recall"])
    red.update({"imw_sem_" + m: im[m] for m in im})
    np.savez_compressed(os.path.join(HERE, "reducers_ref.npz"), **red)

    # ---- align_foreground (numba) and the direction differential map (torch)
    out = {}
    rng = np.random.default_rng(77)
    for j, (H, W) in enumerate([(40, 52), (96, 96), (128, 160)]):
        t = synth.gt_and_pred(9500 + j, H, W, n=max(3, H * W // 700))
        fg = ndi.binary_dilation(t["pred_inst"] > 0, iterations=3) | (rng.random((H, W)) < 0.02)
        seeds = np.where(ndi.binary_erosion(t["pred_inst"] > 0, iterations=2), t["pred_inst"], 0).astype(np.int64)
        seeds = scipy_label(seeds, connectivity=1)
        out["af%d_seed" % j] = seeds.copy()
        out["af%d_fg" % j] = fg
        out["af%d_out" % j] = pp.align_foreground(seeds.copy(), fg, 20)
        out["af%d_out5" % j] = pp.align_foreground(seeds.copy(), fg, 5)
        dl, _ = synth.direction_logits(np.random.default_rng(9600 + j), t["pred_inst"])
        dm = np.argmax(dl, 0).astype(np.int64)
        out["dd%d_dir" % j] = dm
        out["dd%d_out" % j] = ddm.generate_direction_differential_map(torch.from_numpy(dm)[None], 9)[0].numpy()
    zero = np.zeros((16, 16), np.int64)
    out["dd_zero_out"] = ddm.generate_direction_differential_map(torch.from_numpy(zero)[None], 9)[0].numpy()
    np.savez_compressed(os.path.join(HERE, "ordered_ref.npz"), **out)

    # ---- mudslide_watershed (numba get_graph_degree / prepare run by the reference's own file)
    mud = {}
    specs = [(9700, 96, 110, 14, 2, 1, 0.0), (9701, 64, 64, 8, 1, 2, 0.05), (9702, 128, 100, 20, 3, 0, 0.1),
             (9703, 40, 52, 5, 1, 1, 0.3), (9704, 150, 160, 40, 2, 1, 0.02)]
    for j, (seed, H, W, n, ero, dil, noise) in enumerate(specs):
        t = synth.gt_and_pred(seed, H, W, n=n)
        inst = t["pred_inst"]
        r2 = np.random.default_rng(seed)
        fore = ndi.binary_dilation(inst > 0, iterations=dil) if dil else inst > 0
        seg = ndi.binary_erosion(inst > 0, iterations=ero)
        dl, _ = synth.direction_logits(r2, inst)
        dirg = np.argmax(dl, 0).astype(np.int64)
        dirg[r2.random((H, W)) < noise] = r2.integers(0, 9)
        dirg[~fore] = 0
        mud["m%d_seg" % j], mud["m%d_dir" % j], mud["m%d_fore" % j] = seg.copy(), dirg.copy(), fore.copy()
        d_io = dirg.copy()
        pred, boundary = pp.mudslide_watershed(seg.copy(), d_io, fore.copy())
        mud["m%d_pred" % j], mud["m%d_boundary" % j], mud["m%d_dir_after" % j] = pred, boundary, d_io
    np.savez_compressed(os.path.join(HERE, "mudslide_ref.npz"), **mud)

    # ---- train-time label generation: gen_instance_hv_map / DistanceLabelMake run from the reference's own files
    def load(modname, path):
        spec = importlib.util.spec_from_file_location(modname, path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod

    hv = load("ref_hv_map", os.path.join(REF, "tiseg/datasets/ops/hv_map.py"))
    dmap = load("ref_distance_map", os.path.join(REF, "tiseg/datasets/ops/distance_map.py"))
    lab = {}
    for j, (seed, H, W, n) in enumerate([(9900, 64, 80, 10), (9901, 128, 100, 30), (9902, 256, 256, 60),
                                         (9903, 40, 33, 3), (9904, 96, 96, 1)]):
        t = synth.gt_and_pred(seed, H, W, n=n)
        inst = t["gt_inst"].astype(np.int32)
        if j == 4:                                   # one instance covering the whole tile, one thin line
            inst[:] = 1
        if j == 3:
            inst[5, 2:30] = 77
        lab["l%d_inst" % j] = inst
        lab["l%d_hv" % j] = hv.gen_instance_hv_map(inst)
        for norm in (0, 1):
            data = dict(sem_gt=(inst > 0).astype(np.uint8), inst_gt=inst.copy(), seg_fields=[])
            lab["l%d_dist%d" % (j, norm)] = dmap.DistanceLabelMake(inst_norm=bool(norm))(data)["dist_gt"]
    # BoundLabelMake: skimage 0.18's dilation / erosion are ndi.grey_dilation / grey_erosion(footprint=selem)
    sk = sys.modules["skimage"]
    sk.morphology.dilation = lambda image, selem=None: ndi.grey_dilation(image, footprint=selem[::-1, ::-1])
    sk.morphology.erosion = lambda image, selem=None: ndi.grey_erosion(image, footprint=selem)
    sk.morphology.selem = _stub("skimage.morphology.selem", diamond=_opp_mod().diamond)
    bmap = load("ref_bound_map", os.path.join(REF, "tiseg/datasets/ops/bound_map.py"))
    for j in range(5):
        inst = lab["l%d_inst" % j]
        sem = ((inst % 3) + 1).astype(np.uint8) * (inst > 0)
        lab["l%d_sem" % j] = sem
        for radius in (1, 3, (2, 1)):
            data = dict(sem_gt=sem.copy(), inst_gt=inst.copy(), seg_fields=[])
            out = bmap.BoundLabelMake(edge_id=4, selem_radius=radius)(data)
            tag = "l%d_r%s" % (j, "".join(str(r) for r in (radius if isinstance(radius, tuple) else (radius,))))
            lab[tag + "_sem"], lab[tag + "_bound"] = out["sem_gt"], out["sem_gt_w_bound"]
        lab["l%d_fixed" % j] = bmap.BoundLabelMake()._fix_inst(inst)
    # UNetLabelMake (np.PINF left numpy in 2.0: restored for the reference's own line, unet_map.py:77)
    if not hasattr(np, "PINF"):
        np.PINF = np.inf
    umap = load("ref_unet_map", os.path.join(REF, "tiseg/datasets/ops/unet_map.py"))
    for j in (0, 1, 3, 4):
        inst = lab["l%d_inst" % j]
        data = dict(sem_gt=lab["l%d_sem" % j].copy(), inst_gt=inst.copy(), seg_fields=[])
        out = umap.UNetLabelMake(w0=10.0, sigma=5.0)(data)
        lab["l%d_unet_w" % j], lab["l%d_unet_inner" % j] = out["loss_weight_map"], out["sem_gt_inner"]
    np.savez_compressed(os.path.join(HERE, "labelgen_ref.npz"), **lab)

    # ---- DIST post-process: the reference's OWN SOURCE TEXT (dist.py:31-131 helpers + DIST.postprocess :275-284),
    # executed with scikit-image replaced by the oracle's port (scikit-image is absent here).  This pins the control
    # flow of the restatement in oracle/postprocess.py, not scikit-image itself.
    import ast, textwrap
    from oracle import skimage_port as skp
    dsrc = open(os.path.join(REF, "tiseg/models/segmentors/dist.py")).read()
    tree = ast.parse(dsrc)
    wanted = ("prepare_prob", "H_reconstruction_erosion", "find_maxima", "generate_wsl", "arrange_label",
              "dynamic_watershed_alias")
    chunks = [ast.get_source_segment(dsrc, n) for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in wanted]
    cls = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "DIST"][0]
    post = [n for n in cls.body if isinstance(n, ast.FunctionDef) and n.name == "postprocess"][0]
    chunks.append(textwrap.dedent(ast.get_source_segment(dsrc, post, padded=True)))
    morph = types.SimpleNamespace(
        reconstruction=lambda seed, mask, method="erosion": skp.reconstruction_erosion(seed, mask),
        dilation=_opp_mod().dilation, erosion=_opp_mod().erosion, square=_opp_mod().square, disk=_opp_mod().disk,
        watershed=lambda image, markers, mask=None: skp.watershed(image, markers, mask))
    measure = types.SimpleNamespace(label=skp.label)
    class _Numpy1Scalars:
        """numpy as the reference's pinned numpy 1.x sees scalars: ``np.uint8(255) + 1`` inside the np.vectorize'd
        ``making_top_mask`` (dist.py:48-52) promotes to a Python-int sum (256); numpy >= 2 would wrap it to 0."""
        def __getattr__(self, name):
            return getattr(np, name)

        @staticmethod
        def vectorize(f):
            return np.vectorize(lambda x: f(int(x)))
    ns = {"np": _Numpy1Scalars(), "morph": morph, "measure": measure}
    exec(compile("\n\n".join(chunks), "dist.py (reference source)", "exec"), ns)
    dref = {}
    for j, (H, W) in enumerate([(48, 56), (64, 64), (80, 100), (33, 47)]):
        t = synth.tile_dist(2, 40 + j, H=H, W=W)
        d = t["dist_logit"]
        if j == 3:
            d = d * 0 + 7.3                     # one plateau: the background value of arrange_label is the label
        dref["d%d_in" % j] = d
        dref["d%d_out" % j] = ns["postprocess"](None, None, d)[1]
    np.savez_compressed(os.path.join(HERE, "dist_ref.npz"), **dref)

    # ---- the other segmentors' post-processes, same technique: the method's source text out of the reference file,
    # executed with `self` = a namespace carrying the attributes it reads; scipy / OpenCV are the real libraries,
    # scikit-image calls go to the port, align_foreground is the reference's own numba function (loaded above).
    import math
    import cv2
    from scipy.ndimage import binary_fill_holes, measurements

    def ref_method(relpath, cls_name, meth_name, extra):
        src = open(os.path.join(REF, relpath)).read()
        tr = ast.parse(src)
        c = [n for n in tr.body if isinstance(n, ast.ClassDef) and n.name == cls_name][0]
        f = [n for n in c.body if isinstance(n, ast.FunctionDef) and n.name == meth_name][0]
        env = {"np": np, "math": math, "cv2": cv2, "binary_fill_holes": binary_fill_holes, "measurements": measurements,
               "remove_small_objects": _opp_mod().remove_small_objects, "watershed": skp.watershed,
               "measure": types.SimpleNamespace(label=skp.label),
               "morphology": types.SimpleNamespace(dilation=lambda image, selem=None: _opp_mod().dilation(image, selem),
                                                   disk=_opp_mod().disk),
               "align_foreground": pp.align_foreground}
        env.update(extra)
        exec(compile(textwrap.dedent(ast.get_source_segment(src, f, padded=True)), relpath, "exec"), env)
        return env[meth_name]

    seg = {}
    cfg = lambda radius: types.SimpleNamespace(test_cfg={"radius": radius}, num_classes=3)
    unet_pp = ref_method("tiseg/models/segmentors/unet.py", "UNet", "postprocess", {})
    cdnet_pp = ref_method("tiseg/models/segmentors/cdnet.py", "CDNet", "postprocess", {})
    dcan_pp = ref_method("tiseg/models/segmentors/dcan.py", "DCAN", "postprocess", {})
    mt_unet = ref_method("tiseg/models/segmentors/multi_task_unet.py", "MultiTaskUNet", "postprocess", {})
    mt_cunet = ref_method("tiseg/models/segmentors/multi_task_cunet.py", "MultiTaskCUNet", "postprocess", {})
    mt_cdnet = ref_method("tiseg/models/segmentors/multi_task_cdnet.py", "MultiTaskCDNet", "postprocess", {})
    hover = ref_method("tiseg/models/segmentors/hovernet.py", "HoverNet", "hover_post_proc", {})
    for j, (H, W, C) in enumerate([(96, 110, 4), (128, 128, 2), (70, 61, 7)]):
        t = synth.gt_and_pred(9300 + j, H, W, n=max(4, H * W // 600), num_classes=C)
        pred = (t["pred_sem"] if "pred_sem" in t else (t["pred_inst"] > 0)).astype(np.int64)
        pred = np.where(t["pred_inst"] > 0, np.maximum(pred, 1), 0)
        seg["u%d_pred" % j] = pred
        seg["u%d_sem" % j], seg["u%d_inst" % j] = unet_pp(cfg(1), pred.copy())
        tc = synth.three_class_map(t["pred_inst"]).astype(np.int64)             # 0 bg, 1 inside, 2 edge
        edge3 = np.where(tc == 2, 3, pred * (tc == 1)).astype(np.int64)          # classes 1..2 inside, 3 = edge class
        edge3 = np.minimum(edge3, 3)
        seg["c%d_pred" % j] = edge3
        seg["c%d_sem" % j], seg["c%d_inst" % j] = cdnet_pp(cfg(3), edge3.copy())
        cell, cont = (t["pred_inst"] > 0).astype(np.int64), (tc == 2).astype(np.uint8)
        seg["d%d_cell" % j], seg["d%d_cont" % j] = cell, cont
        seg["d%d_sem" % j], seg["d%d_inst" % j] = dcan_pp(cfg(3), cell.copy(), cont)
        inner = (tc == 1).astype(np.int64)
        seg["m%d_inner" % j], seg["m%d_tc" % j], seg["m%d_sempred" % j] = inner, tc, pred
        seg["m%d_unet_sem" % j], seg["m%d_unet_inst" % j] = mt_unet(None, inner.copy(), pred.copy())
        seg["m%d_cunet_sem" % j], seg["m%d_cunet_inst" % j] = mt_cunet(None, tc.copy(), pred.copy())
        seg["m%d_cdnet_sem" % j], seg["m%d_cdnet_inst" % j] = mt_cdnet(None, tc.copy(), pred.copy())
    for j, (H, W, sf) in enumerate([(120, 140, 1), (96, 96, 2), (150, 131, 1)]):
        t = synth.tile_hover(3, 20 + j, H=H, W=W)
        seg["h%d_fore" % j], seg["h%d_hv" % j], seg["h%d_sf" % j] = t["fore_map"], t["hv_map"], np.array(sf)
        seg["h%d_out" % j] = hover(None, t["fore_map"].copy(), t["hv_map"].copy(), fx=1, scale_factor=sf)
    np.savez_compressed(os.path.join(HERE, "segmentors_ref.npz"), **seg)

    # ---- CustomDataset.pre_eval / evaluate (custom.py:219-435) from their source text: ground truth written to a
    # temporary directory in the converted-dataset layout, mmcv.imread served by pillow, the metric functions are the
    # reference's own modules loaded above
    import tempfile, warnings as _warnings, os.path as osp
    from collections import OrderedDict
    from PIL import Image

    class _Table:
        def add_column(self, *a, **k):
            pass

        def get_string(self):
            return ""
    dsenv = {"osp": osp, "os": os, "warnings": _warnings, "OrderedDict": OrderedDict, "PrettyTable": _Table,
             "print_log": lambda *a, **k: None,
             "mmcv": types.SimpleNamespace(imread=lambda f, flag=None, backend=None: np.array(Image.open(f))),
             "re_instance": isem.re_instance}
    for mod in (inst_mod, sem_mod):
        dsenv.update({k: getattr(mod, k) for k in dir(mod) if k.startswith("pre_eval")})
    ds_pre_eval = ref_method("tiseg/datasets/custom.py", "CustomDataset", "pre_eval", dsenv)
    ds_evaluate = ref_method("tiseg/datasets/custom.py", "CustomDataset", "evaluate", dsenv)
    dsr = {}
    with tempfile.TemporaryDirectory() as td:
        infos, preds = [], []
        for j, (H, W) in enumerate([(96, 110), (128, 128), (70, 61), (64, 64)]):
            t = synth.gt_and_pred(9400 + j, H, W, n=max(4, H * W // 600))
            gs = (t["gt_inst"] > 0).astype(np.uint8)
            gi = t["gt_inst"].astype(np.int32) * 3                     # non-contiguous ids: re_instance has work to do
            if j == 3:
                gi[:] = 0; gs[:] = 0                                   # an image without nuclei
            Image.fromarray(gs).save(osp.join(td, "im%d_sem.png" % j))
            np.save(osp.join(td, "im%d_inst.npy" % j), gi)
            infos.append(dict(file_name=osp.join(td, "im%d.tif" % j), sem_file_name=osp.join(td, "im%d_sem.png" % j),
                              inst_file_name=osp.join(td, "im%d_inst.npy" % j)))
            sp, ip = (t["pred_inst"] > 0).astype(np.uint8), t["pred_inst"].astype(np.int32) * 2
            preds.append(dict(sem_pred=sp, inst_pred=ip))
            dsr["p%d_gt_sem" % j], dsr["p%d_gt_inst" % j], dsr["p%d_sem_pred" % j], dsr["p%d_inst_pred" % j] = gs, gi, sp, ip
        me = types.SimpleNamespace(data_infos=infos, sem_suffix="_sem.png", CLASSES=("background", "nuclei"))
        results = ds_pre_eval(me, [dict(p) for p in preds], list(range(4)))
    for j, r in enumerate(results):
        dsr["p%d_name" % j] = np.array(r["name"])
        dsr["p%d_bin_aji" % j] = np.array(r["bin_aji_pre_eval_res"], np.float64)
        dsr["p%d_bin_pq" % j] = np.array(r["bin_pq_pre_eval_res"], np.float64)
        dsr["p%d_sem" % j] = np.stack([x.numpy() for x in r["sem_pre_eval_res"]])
    ev, storage = ds_evaluate(me, results)
    dsr["eval_keys"] = np.array(list(ev.keys()))
    dsr["eval_values"] = np.array([float(v) for v in ev.values()], np.float64)
    # CoNICDataset (conic.py:126-323): per-class AJI / PQ on top of the class assignment
    dsenv["assign_sem_class_to_insts"] = isem.assign_sem_class_to_insts
    cn_pre_eval = ref_method("tiseg/datasets/conic.py", "CoNICDataset", "pre_eval", dsenv)
    cn_evaluate = ref_method("tiseg/datasets/conic.py", "CoNICDataset", "evaluate", dsenv)
    CN = ("background", "neutrophil", "epithelial", "lymphocyte", "plasma", "eosinophil", "connective")
    with tempfile.TemporaryDirectory() as td:
        infos, preds = [], []
        for j, (H, W) in enumerate([(96, 110), (128, 128), (70, 61)]):
            t = synth.gt_and_pred(9450 + j, H, W, n=max(6, H * W // 500), num_classes=7)
            gs, gi = t["gt_sem"].astype(np.uint8), t["gt_inst"].astype(np.int32)
            Image.fromarray(gs).save(osp.join(td, "c%d_sem.png" % j))
            np.save(osp.join(td, "c%d_inst.npy" % j), gi)
            infos.append(dict(sem_file_name=osp.join(td, "c%d_sem.png" % j), inst_file_name=osp.join(td, "c%d_inst.npy" % j)))
            sp, ip = t["pred_sem"].astype(np.uint8), t["pred_inst"].astype(np.int32)
            preds.append(dict(sem_pred=sp, inst_pred=ip))
            dsr["q%d_gt_sem" % j], dsr["q%d_gt_inst" % j], dsr["q%d_sem_pred" % j], dsr["q%d_inst_pred" % j] = gs, gi, sp, ip
        me = types.SimpleNamespace(data_infos=infos, CLASSES=CN)
        cres = cn_pre_eval(me, [dict(p) for p in preds], list(range(3)))
    for j, r in enumerate(cres):
        dsr["q%d_bin_aji" % j] = np.array(r["bin_aji_pre_eval_res"], np.float64)
        dsr["q%d_bin_pq" % j] = np.array(r["bin_pq_pre_eval_res"], np.float64)
        dsr["q%d_aji" % j] = np.stack([np.asarray(x) for x in r["aji_pre_eval_res"]])          # float32, as returned
        dsr["q%d_pq" % j] = np.stack([np.asarray(x) for x in r["pq_pre_eval_res"]])
        dsr["q%d_sem" % j] = np.stack([x.numpy() for x in r["sem_pre_eval_res"]])
    cev, _ = cn_evaluate(me, cres)
    dsr["conic_eval_keys"] = np.array(list(cev.keys()))
    dsr["conic_eval_values"] = np.array([float(v) for v in cev.values()], np.float64)
    dsr["conic_eval_isstr"] = np.array([isinstance(v, str) for v in cev.values()])
    # MoNuSegDatasetDebug (monuseg_debug.py:34-...): the extra boundary-class semantic metrics
    md_pre_eval = ref_method("tiseg/datasets/monuseg_debug.py", "MoNuSegDatasetDebug", "pre_eval", dsenv)
    md_evaluate = ref_method("tiseg/datasets/monuseg_debug.py", "MoNuSegDatasetDebug", "evaluate", dsenv)
    with tempfile.TemporaryDirectory() as td:
        infos, preds = [], []
        for j, (H, W) in enumerate([(96, 110), (80, 64)]):
            t = synth.gt_and_pred(9480 + j, H, W, n=max(4, H * W // 600))
            gs, gi = (t["gt_inst"] > 0).astype(np.uint8), t["gt_inst"].astype(np.int32)
            Image.fromarray(gs).save(osp.join(td, "m%d_sem.png" % j))
            np.save(osp.join(td, "m%d_inst.npy" % j), gi)
            infos.append(dict(file_name=osp.join(td, "m%d.tif" % j), sem_file_name=osp.join(td, "m%d_sem.png" % j),
                              inst_file_name=osp.join(td, "m%d_inst.npy" % j)))
            sp, ip = (t["pred_inst"] > 0).astype(np.uint8), t["pred_inst"].astype(np.int32)
            tcp, tcg = synth.three_class_map(t["pred_inst"]).astype(np.uint8), synth.three_class_map(t["gt_inst"]).astype(np.uint8)
            preds.append(dict(sem_pred=sp, inst_pred=ip, tc_pred=tcp, tc_gt=tcg))
            for key, val in (("gt_sem", gs), ("gt_inst", gi), ("sem_pred", sp), ("inst_pred", ip), ("tc_pred", tcp), ("tc_gt", tcg)):
                dsr["d%d_%s" % (j, key)] = val
        me = types.SimpleNamespace(data_infos=infos, sem_suffix="_sem.png", CLASSES=("background", "nuclei"))
        mres = md_pre_eval(me, [dict(p) for p in preds], list(range(2)))
    for j, r in enumerate(mres):
        dsr["d%d_name" % j] = np.array(r["name"])
        dsr["d%d_bin_aji" % j] = np.array(r["bin_aji_pre_eval_res"], np.float64)
        dsr["d%d_bin_pq" % j] = np.array(r["bin_pq_pre_eval_res"], np.float64)
        dsr["d%d_sem" % j] = np.stack([x.numpy() for x in r["sem_pre_eval_res"]])
        dsr["d%d_bound" % j] = np.stack([x.numpy() for x in r["bound_sem_pre_eval_res"]])
    mev, _ = md_evaluate(me, mres)
    dsr["monuseg_eval_keys"] = np.array(list(mev.keys()))
    dsr["monuseg_eval_values"] = np.array([float(v) for v in mev.values()], np.float64)
    # the convenience scores of tiseg/utils/__init__.py that run in the reference (binary_aggregated_jaccard_index,
    # aggregated_jaccard_index and panoptic_quality raise there: they hand semantic maps to pre_eval_aji / pre_eval_pq,
    # which expect id lists — inst_metrics.py:292, 307, 353)
    for j, (H, W) in enumerate([(96, 110), (64, 80)]):
        t = synth.gt_and_pred(9490 + j, H, W, n=max(4, H * W // 600), num_classes=4)
        ipd, igt = isem.re_instance(t["pred_inst"]), isem.re_instance(t["gt_inst"])
        sp, sg = t["pred_sem"].astype(np.uint8), t["gt_sem"].astype(np.uint8)
        dsr["s%d_inst_pred" % j], dsr["s%d_inst_gt" % j], dsr["s%d_sem_pred" % j], dsr["s%d_sem_gt" % j] = ipd, igt, sp, sg
        dsr["s%d_bin_pq" % j] = np.array(inst_mod.binary_panoptic_quality(ipd, igt), np.float64)
        dsr["s%d_inst_dice" % j] = np.float64(inst_mod.binary_inst_dice(ipd, igt))
        dsr["s%d_dice" % j] = sem_mod.dice_similarity_coefficient(sp, sg, 4)
        pr = sem_mod.precision_recall(sp, sg, 4)
        dsr["s%d_precision" % j], dsr["s%d_recall" % j] = pr[0], pr[1]
    np.savez_compressed(os.path.join(HERE, "dataset_ref.npz"), **dsr)

    # ---- BaseSegmentor.inference (base.py:255-381): window canvas + TTA + reverse + softmax + mean, from source.
    # `self.calculate` is a recorder that returns seeded logits for every window it is asked for; the recorded windows
    # are what the fused kernel (tiseg_softmax_argmax_tta_typed) is given.
    import torch.nn.functional as F
    benv = {"torch": torch, "F": F, "resize": None}
    b_inference = ref_method("tiseg/models/segmentors/base.py", "BaseSegmentor", "inference", benv)
    b_split = ref_method("tiseg/models/segmentors/base.py", "BaseSegmentor", "split_inference", benv)
    b_whole = ref_method("tiseg/models/segmentors/base.py", "BaseSegmentor", "whole_inference", benv)

    def _plain(meth):                                  # the two transforms are @classmethod in the reference
        src = open(os.path.join(REF, "tiseg/models/segmentors/base.py")).read()
        tr = ast.parse(src)
        c = [n for n in tr.body if isinstance(n, ast.ClassDef) and n.name == "BaseSegmentor"][0]
        f = [n for n in c.body if isinstance(n, ast.FunctionDef) and n.name == meth][0]
        f.decorator_list = []
        env = dict(benv)
        exec(compile(ast.Module(body=[f], type_ignores=[]), "base.py", "exec"), env)
        return env[meth]
    b_tta, b_rev = _plain("tta_transform"), _plain("reverse_tta_transform")

    class _Cfg(dict):
        __getattr__ = dict.__getitem__
    tta = {}
    for j, (H, W, window, overlap, C, B, rots, flips) in enumerate([
            (70, 90, 32, 8, 2, 1, [0, 90], ["none", "horizontal", "vertical", "diagonal"]),     # the shipped TTA set
            (48, 56, 24, 8, 3, 2, [90, 180], ["horizontal", "vertical"]),
            (50, 37, 0, 0, 3, 1, [0, 270], ["none", "diagonal"])]):
        rng = np.random.default_rng(9600 + j)
        calls = []

        def calculate(patch):
            out = torch.from_numpy((rng.integers(-12, 13, (patch.shape[0], C, patch.shape[2], patch.shape[3])) / 4.0)
                                   .astype(np.float32))
            calls.append(out.numpy())
            return out
        me = types.SimpleNamespace(num_classes=C, calculate=calculate)
        me.test_cfg = _Cfg(mode="split" if window else "whole", crop_size=(window, window), overlap_size=(overlap, overlap),
                           rotate_degrees=rots, flip_directions=flips)
        me.tta_transform = lambda img, r, f: b_tta(me, img, r, f)
        me.reverse_tta_transform = lambda img, r, f: b_rev(me, img, r, f)
        me.split_inference = lambda img, meta, rescale: b_split(me, img, meta, rescale)
        me.whole_inference = lambda img, meta, rescale: b_whole(me, img, meta, rescale)
        prob = b_inference(me, torch.zeros(B, 3, H, W), None, False).numpy()
        # the recorder saw the windows variant by variant (rotation outer, flip inner), row-major inside a variant
        per = len(calls) // (len(rots) * len(flips))
        for t in range(len(rots) * len(flips)):
            w = np.stack(calls[t * per:(t + 1) * per])                   # [M, B, C, h, w]
            w = np.ascontiguousarray(np.moveaxis(w, 1, 0)) if window else w[0]
            tta["t%d_v%d" % (j, t)] = np.round(w * 4).astype(np.int8)    # the logits are quarter-integers: stored x4 as int8
        tta["t%d_meta" % j] = np.array([H, W, window, overlap, C, B, len(rots) * len(flips)])
        tta["t%d_rots" % j] = np.array([r for r in rots for _ in flips])
        tta["t%d_flips" % j] = np.array([f for _ in rots for f in flips])
        tta["t%d_prob" % j] = prob
    # CDNet.inference (cdnet.py:154-217) + _ddm_enhencement (:354-367) from source, whole-image mode, recorder network
    cenv = dict(benv)
    cenv["generate_direction_differential_map"] = ddm.generate_direction_differential_map
    c_inference = ref_method("tiseg/models/segmentors/cdnet.py", "CDNet", "inference", cenv)
    csrc = open(os.path.join(REF, "tiseg/models/segmentors/cdnet.py")).read()
    cnode = [n for n in ast.parse(csrc).body if isinstance(n, ast.ClassDef) and n.name == "CDNet"][0]
    enh = [n for n in cnode.body if isinstance(n, ast.FunctionDef) and n.name == "_ddm_enhencement"][0]
    enh.decorator_list = []
    exec(compile(ast.Module(body=[enh], type_ignores=[]), "cdnet.py", "exec"), cenv)
    for j, (H, W, flips, if_ddm) in enumerate([(40, 44, ["none", "horizontal", "vertical"], True), (36, 36, ["none"], False)]):
        rng = np.random.default_rng(9700 + j)
        rec = []

        def whole(img, meta, rescale):
            outs = [torch.from_numpy((rng.standard_normal((1, c, img.shape[2], img.shape[3])) * 2).astype(np.float16)
                                     .astype(np.float32)) for c in (3, 9, 1)]
            outs[2] = outs[2].abs()
            rec.append([o.numpy()[0].astype(np.float16) for o in outs])
            return tuple(outs)
        me = types.SimpleNamespace(num_classes=3, num_angles=8, whole_inference=whole)
        me.test_cfg = _Cfg(mode="whole", rotate_degrees=[0], flip_directions=flips, if_ddm=if_ddm)
        me.tta_transform = lambda img, r, f: b_tta(me, img, r, f)
        me.reverse_tta_transform = lambda img, r, f: b_rev(me, img, r, f)
        me._ddm_enhencement = lambda a, b, c: cenv["_ddm_enhencement"](me, a, b, c)
        sem_out, dir_out = c_inference(me, torch.zeros(1, 3, H, W), None, False)
        tta["c%d_flips" % j] = np.array(flips)
        tta["c%d_if_ddm" % j] = np.array(if_ddm)
        for t, (a, b, c) in enumerate(rec):
            tta["c%d_sem%d" % (j, t)], tta["c%d_dir%d" % (j, t)], tta["c%d_pt%d" % (j, t)] = a, b, c
        tta["c%d_sem_out" % j], tta["c%d_dir_out" % j] = sem_out.numpy()[0], dir_out.numpy()[0]
    np.savez_compressed(os.path.join(HERE, "tta_ref.npz"), **tta)
    print("golden vectors written to", HERE)


if __name__ == "__main__":
    main()
