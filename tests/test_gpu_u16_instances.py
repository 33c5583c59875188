"""uint16 instance ground truth read natively.  Every entry point that reads a ground-truth instance map (the multi-class
pair metrics, the class assignment, ``_fix_inst`` and the HV map of the label makers, and the datasets above them) must
return for a uint16 map, bit for bit and with the same dtypes, what it returns for the int32 upcast of that map, and must
hand the uint16 buffer to the library as it is: no widened copy on the host or on the device.  The first tests check the
Python side on the CPU; the others compare the two calls on the GPU."""
import importlib.util
import os
import re
import sys
import zlib
from collections import Counter

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import tiseg_b200  # noqa: E402,F401
from tiseg_b200 import _lib, ops, synth  # noqa: E402

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")
CSRC = os.path.join(ROOT, "tissue-image-segmentation_b200", "csrc")


def _np(a):
    return a.detach().cpu().numpy() if _lib.is_torch(a) else np.asarray(a)


def _same(got, want, what):
    """bit-identical, same dtype, same kind (numpy / torch); floats compared as raw bits"""
    if isinstance(want, dict):
        assert sorted(got) == sorted(want), what
        for k in want:
            _same(got[k], want[k], "%s[%s]" % (what, k))
        return
    if isinstance(want, (list, tuple)):
        assert type(got) is type(want) and len(got) == len(want), what
        for i, (g, w) in enumerate(zip(got, want)):
            _same(g, w, "%s[%d]" % (what, i))
        return
    if want is None or isinstance(want, (str, int, float)):
        assert type(got) is type(want) and (got == want or (got != got and want != want)), (what, got, want)
        return
    assert _lib.is_torch(got) == _lib.is_torch(want), "%s: %s vs %s" % (what, type(got), type(want))
    if _lib.is_torch(want):
        assert got.device == want.device, (what, got.device, want.device)
    g, w = _np(got), _np(want)
    assert type(g) is type(w), (what, type(g), type(w))
    assert g.dtype == w.dtype and g.shape == w.shape, "%s: %s%r vs %s%r" % (what, g.dtype, g.shape, w.dtype, w.shape)
    if g.dtype.kind == "f":
        g, w = g.view("u%d" % g.itemsize), w.view("u%d" % w.itemsize)
    bad = np.argwhere(g != w)
    assert len(bad) == 0, "%s: %d of %d elements differ, first at %r" % (what, len(bad), g.size, tuple(bad[0]))


def _bench():
    spec = importlib.util.spec_from_file_location("_tiseg_bench", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    return b


def _resolves(bench, name):
    try:
        bench.kernel_bytes_per_px(bench.ConicSweep(), name)
        return True
    except KeyError:
        return False


def _spread_ids(inst, seed, top=65535):
    """the same partition with the ids 1..K moved to distinct values in [1, top], `top` itself included"""
    rng = np.random.default_rng(seed)
    ids = np.unique(inst[inst > 0])
    new = np.concatenate([rng.choice(np.arange(1, top), size=len(ids) - 1, replace=False), [top]]) if len(ids) else []
    lut = np.zeros(int(inst.max()) + 1 if inst.size else 1, np.int64)
    lut[ids] = rng.permutation(np.asarray(new, np.int64))
    return lut[inst].astype(np.int32)


def _u16(a):
    a = np.asarray(a)
    assert a.min() >= 0 and a.max() < 65536
    return a.astype(np.uint16)


# --------------------------------------------------------------------------- CPU: dispatch, batching, timing names
class _Recorder:
    def __init__(self):
        self.calls = []

    def call(self, name, *args):
        self.calls.append((name, args))


def test_ops_hand_uint16_ground_truth_to_the_u16_entries_as_it_is(monkeypatch):
    """The operators pick the uint16 twin and pass the caller's own buffer (same address: nothing converted it); int32
    and every other dtype keep going to the int32 entry."""
    import torch
    rec = _Recorder()
    monkeypatch.setattr(ops, "get_ctx", lambda device=None: rec)
    rng = np.random.default_rng(1)
    g16 = rng.integers(0, 65536, (2, 9, 13)).astype(np.uint16)
    t16 = torch.from_numpy(g16.copy())
    sem = rng.integers(0, 3, (2, 9, 13)).astype(np.uint8)
    pred = rng.integers(0, 9, (2, 9, 13)).astype(np.int32)
    P = lambda g, a: a if g.ndim == 3 else a[0]                 # the other arguments, shaped like the ground truth
    calls = [
        (lambda g: ops.pair_metrics_multiclass(P(g, pred), P(g, sem), g, P(g, sem), 3), "tiseg_pair_metrics_multiclass", 2),
        (lambda g: ops.pair_metrics_bin(P(g, pred), g), "tiseg_pair_metrics_bin_iou", 1),
        (lambda g: ops.assign_sem_class(g, P(g, sem), 3), "tiseg_assign_sem_class", 0),
        (lambda g: ops.fix_inst(g), "tiseg_fix_inst", 0),
        (lambda g: ops.gen_instance_hv_map(g), "tiseg_gen_hv_map", 0),
    ]
    u16_names = {"tiseg_pair_metrics_multiclass": "tiseg_pair_metrics_multiclass_u16gt",
                 "tiseg_pair_metrics_bin_iou": "tiseg_pair_metrics_bin_u16gt", "tiseg_assign_sem_class": "tiseg_assign_sem_class_u16",
                 "tiseg_fix_inst": "tiseg_fix_inst_u16", "tiseg_gen_hv_map": "tiseg_gen_hv_map_u16"}
    for fn, name32, slot in calls:
        for g, addr in ((g16, g16.ctypes.data), (t16, t16.data_ptr()), (g16[0], g16.ctypes.data)):
            rec.calls.clear()
            fn(g)
            (name, args), = rec.calls
            assert name == u16_names[name32], (name32, name)
            assert args[slot].value == addr, name
        for g in (g16.astype(np.int32), g16.astype(np.int64), t16.to(torch.int32)):
            rec.calls.clear()
            fn(g)
            assert rec.calls[0][0] == name32


def test_datasets_keep_uint16_groups_uint16():
    """CustomDataset._stack / _gt_batch: a group whose instance maps are all uint16 stays uint16 (numpy and torch);
    one other dtype in the group and the batch is int32, as before."""
    import torch
    from tiseg_b200 import datasets
    rng = np.random.default_rng(2)
    maps = [rng.integers(0, 65536, (7, 5)).astype(np.uint16) for _ in range(3)]
    D = datasets.CustomDataset
    assert D._inst_dtype(maps) == np.uint16
    assert D._inst_dtype(maps[:2] + [maps[2].astype(np.int32)]) == np.int32
    b = D._stack(maps, D._inst_dtype(maps))
    assert b.dtype == np.uint16 and np.array_equal(b, np.stack(maps))
    tm = [torch.from_numpy(m) for m in maps]
    assert D._inst_dtype(tm) == np.uint16
    tb = D._stack(tm, D._inst_dtype(tm))
    assert tb.dtype == torch.uint16 and np.array_equal(tb.numpy(), np.stack(maps))
    sems = [np.zeros((7, 5), np.uint8)] * 3
    ds = datasets.CoNICDataset(sem_gts=sems, inst_gts=maps)
    sg, ig = ds._gt_batch([2, 0, 1])
    assert ig.dtype == np.uint16 and np.array_equal(ig, np.stack([maps[2], maps[0], maps[1]]))
    ds = datasets.CoNICDataset(sem_gts=sems, inst_gts=maps[:2] + [maps[2].astype(np.int64)])
    assert ds._gt_batch([0, 1, 2])[1].dtype == np.int32


def test_uint16_timing_names_resolve_in_the_bench_byte_table():
    """Every uint16 instantiation launched with a TISEG_ID_NAME timing name (and k_eqbits<uint16_t>) resolves in
    bench.py's KERNEL_BYTES prefix lookup wherever its int32 name does; those of the evaluation path all do."""
    bench = _bench()
    found = []
    for f in ("metrics.cu", "labelgen.cu"):
        for name in re.findall(r'TISEG_ID_NAME\(T, "([A-Za-z0-9_]+)"\)', open(os.path.join(CSRC, f)).read()):
            found.append((f, name))
            assert _resolves(bench, name + "<uint16_t>") == _resolves(bench, name), name
            if f == "metrics.cu":
                assert _resolves(bench, name + "<uint16_t>"), name
    assert {n for f, n in found if f == "metrics.cu"} == {"k_max_id", "k_inst_class_hist", "k_comp_class_bits"}
    assert _resolves(bench, "k_eqbits<uint16_t>")


# --------------------------------------------------------------------------- GPU: multi-class metrics
def _multiclass_case(name, C):
    """-> (pred_inst int32, pred_sem, gt_inst int32 with ids < 65536, gt_sem), all [N, H, W]"""
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    if name.startswith("conic"):
        t = [synth.gt_and_pred(7100 + j, 256, 256, num_classes=C) for j in range(5)]
        st = lambda k: np.stack([x[k] for x in t])
        return st("pred_inst"), st("pred_sem"), st("gt_inst"), st("gt_sem")
    if name == "dense_65535":
        H, W = 255, 257                                          # 65535 pixels, every one its own instance, ids 1..65535
        g = rng.permutation(np.arange(1, H * W + 1)).reshape(1, H, W).astype(np.int32)
        p = (np.arange(H)[:, None] // 3 * 100 + np.arange(W)[None, :] // 4 + 1).astype(np.int32)[None]
        p[:, rng.random((H, W)) < 0.1] = 0
        return p, rng.integers(0, C, (1, H, W)).astype(np.uint8), g, rng.integers(0, C, (1, H, W)).astype(np.uint8)
    H, W, n = {"w77": (61, 77, 12), "w19": (40, 19, 4), "big_300": (300, 300, 80)}[name]
    t = [synth.gt_and_pred(7200 + 10 * len(name) + j, H, W, n=n, num_classes=C) for j in range(3)]
    st = lambda k: np.stack([x[k] for x in t])
    gi = st("gt_inst")
    if name == "big_300":                                        # 90000 pixels, ids spread up to 65535
        gi = np.stack([_spread_ids(x, 11 + j) for j, x in enumerate(gi)])
    gi[-1] = 0                                                   # one tile without any ground-truth instance
    return st("pred_inst"), st("pred_sem"), gi, st("gt_sem")


def _misaligned(a16):
    """CUDA uint16 tensor with the values of `a16` whose data starts 2 bytes past an 8-byte boundary (scalar load path)"""
    import torch
    flat = torch.from_numpy(np.concatenate([np.zeros(1, np.uint16), a16.ravel()])).cuda()
    t = flat[1:].view(a16.shape)
    assert t.data_ptr() % 8 == 2 and t.is_contiguous()
    return t


@gpu
@pytest.mark.parametrize("C", [3, 7])
@pytest.mark.parametrize("case", ["conic", "w77", "w19", "dense_65535", "big_300"])
def test_pair_metrics_multiclass_uint16_equals_int32(case, C):
    import torch
    p, ps, g, gs = _multiclass_case(case, C)
    g16 = _u16(g)
    want = ops.pair_metrics_multiclass(p, ps, g, gs, C)
    assert all(want[k] is not None for k in ("aji", "pq", "bin_aji", "bin_pq"))
    _same(ops.pair_metrics_multiclass(p, ps, g16, gs, C), want, "%s C=%d host" % (case, C))
    with _lib.device_outputs():
        got = ops.pair_metrics_multiclass(p, ps, g16, gs, C)
    _same({k: v.cpu().numpy() for k, v in got.items()}, want, "%s C=%d host in, device out" % (case, C))
    cu = lambda a: torch.from_numpy(a).cuda()
    want_d = ops.pair_metrics_multiclass(cu(p), cu(ps), cu(g), cu(gs), C)
    _same(want_d, {k: cu(v) for k, v in want.items()}, "%s C=%d int32 device" % (case, C))
    _same(ops.pair_metrics_multiclass(cu(p), cu(ps), cu(g16), cu(gs), C), want_d, "%s C=%d device" % (case, C))
    _same(ops.pair_metrics_multiclass(cu(p), cu(ps), _misaligned(g16), cu(gs), C), want_d, "%s C=%d misaligned" % (case, C))
    # per-class records only (no binary outputs requested) and a single [H, W] tile
    _same(ops.pair_metrics_multiclass(p, ps, g16, gs, C, want_bin=False), dict(want, bin_aji=None, bin_pq=None), case + " no bin")
    _same(ops.pair_metrics_multiclass(p[0], ps[0], g16[0], gs[0], C), {k: v[0] for k, v in want.items()}, case + " 2-D")


@gpu
def test_pair_metrics_multiclass_uint16_matches_the_oracle():
    from oracle import metrics as om
    C = 7
    tiles = [synth.gt_and_pred(7300 + j, 256, 256, num_classes=C) for j in range(4)]
    st = lambda k: np.stack([t[k] for t in tiles])
    gi = np.stack([_spread_ids(t["gt_inst"], 40 + j) for j, t in enumerate(tiles)])
    r = ops.pair_metrics_multiclass(st("pred_inst"), st("pred_sem"), _u16(gi), st("gt_sem"), C)
    for j, t in enumerate(tiles):
        rp, rg = om.re_instance(t["pred_inst"]), om.re_instance(gi[j])
        dp, dg = om.assign_sem_class_to_insts(rp, t["pred_sem"], C), om.assign_sem_class_to_insts(rg, t["gt_sem"], C)
        assert np.array_equal(r["aji"][j].astype(np.float32).T[:, 1:], np.stack(om.pre_eval_aji(rp, rg, dp, dg, C, literal=False))), j
        assert np.array_equal(r["pq"][j].astype(np.float32).T[:, 1:], np.stack(om.pre_eval_pq(rp, rg, dp, dg, C, literal=False))), j
        assert tuple(r["bin_aji"][j]) == tuple(np.float64(om.pre_eval_bin_aji(rp, rg, literal=False))), j
        assert tuple(r["bin_pq"][j]) == tuple(np.float64(om.pre_eval_bin_pq(rp, rg, literal=False))), j


# --------------------------------------------------------------------------- GPU: class assignment
@gpu
def test_assign_sem_class_uint16_equals_int32():
    import torch
    from tiseg_b200 import metrics as M
    m = np.load(os.path.join(G, "metrics_ref.npz"))
    names = sorted(k[:-len("_cls_pred")] for k in m.files if k.endswith("_cls_pred"))
    for n in names:
        inst, sem = M.re_instance(m[n + "_gt"]), m[n + "_gt_sem"]
        _same(ops.assign_sem_class(_u16(inst), sem, 4), ops.assign_sem_class(inst, sem, 4), n)
        assert M.assign_sem_class_to_insts(_u16(inst), sem, 4) == M.assign_sem_class_to_insts(inst, sem, 4), n
    for case, C in (("big_300", 7), ("dense_65535", 5), ("w19", 3)):
        _, _, g, gs = _multiclass_case(case, C)
        want = ops.assign_sem_class(g, gs, C)
        _same(ops.assign_sem_class(_u16(g), gs, C), want, case)
        _same(ops.assign_sem_class(_misaligned(_u16(g)), torch.from_numpy(gs).cuda(), C), torch.from_numpy(want).cuda(), case + " device")
        for j in range(g.shape[0]):
            assert M.assign_sem_class_to_insts(_u16(g[j]), gs[j], C) == M.assign_sem_class_to_insts(g[j], gs[j], C), (case, j)


@gpu
def test_reference_named_multiclass_metrics_take_uint16():
    """pre_eval_aji / pre_eval_pq with id dictionaries or semantic maps, aggregated_jaccard_index, panoptic_quality"""
    from tiseg_b200 import metrics as M
    C = 7
    t = synth.gt_and_pred(7400, 256, 256, num_classes=C)
    p, ps, gs = t["pred_inst"], t["pred_sem"], t["gt_sem"]
    g = _spread_ids(t["gt_inst"], 5)
    dp, dg = M.assign_sem_class_to_insts(p, ps, C), M.assign_sem_class_to_insts(g, gs, C)
    dg16 = M.assign_sem_class_to_insts(_u16(g), gs, C)
    assert dg16 == dg
    for fn in (M.pre_eval_aji, M.pre_eval_pq):
        _same(fn(p, _u16(g), dp, dg16, C), fn(p, g, dp, dg, C), fn.__name__ + " dicts")
        _same(fn(p, _u16(g), ps, gs, C), fn(p, g, ps, gs, C), fn.__name__ + " maps")
    assert M.aggregated_jaccard_index(p, _u16(g), ps, gs, C) == M.aggregated_jaccard_index(p, g, ps, gs, C)
    _same(M.panoptic_quality(p, _u16(g), ps, gs, C), M.panoptic_quality(p, g, ps, gs, C), "panoptic_quality")


# --------------------------------------------------------------------------- GPU: datasets
def _records_equal(a, b, what):
    import torch
    assert a.dtype == b.dtype == torch.float64 and a.shape == b.shape and a.device == b.device, what
    assert torch.equal(a.view(torch.int64), b.view(torch.int64)), what


@gpu
def test_conic_dataset_uint16_ground_truth_equals_int32(monkeypatch):
    import torch
    from tiseg_b200 import datasets
    m = np.load(os.path.join(G, "dataset_ref.npz"))
    sems, insts = [m["q%d_gt_sem" % j] for j in range(3)], [m["q%d_gt_inst" % j] for j in range(3)]
    preds = [dict(sem_pred=m["q%d_sem_pred" % j], inst_pred=m["q%d_inst_pred" % j]) for j in range(3)]
    seen = []
    real = ops.pair_metrics_multiclass
    monkeypatch.setattr(ops, "pair_metrics_multiclass", lambda ip, sp, ig, sg, *a, **k: seen.append(str(ig.dtype)) or real(ip, sp, ig, sg, *a, **k))
    want = datasets.CoNICDataset(sem_gts=sems, inst_gts=insts).pre_eval(preds, [0, 1, 2])
    ev_want, st_want = datasets.CoNICDataset(sem_gts=sems, inst_gts=insts).evaluate(want, logger="silent")
    assert len(ev_want) == 67 and list(ev_want.keys()) == m["conic_eval_keys"].tolist()
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    feeds = {"numpy": ([_u16(x) for x in insts], sems, "uint16"),
             "cuda": ([cu(_u16(x)) for x in insts], [cu(x) for x in sems], "torch.uint16")}
    for tag, (i16, s, dt) in feeds.items():
        seen.clear()
        ds = datasets.CoNICDataset(sem_gts=s, inst_gts=i16)
        got = ds.pre_eval(preds, [0, 1, 2])
        assert seen and set(seen) == {dt}, (tag, seen)
        _same(got, want, "CoNIC pre_eval " + tag)
        ev, st = ds.evaluate(got, logger="silent")
        _same(ev, ev_want, "CoNIC evaluate " + tag)
        _same(st, st_want, "CoNIC storage " + tag)
    # batched records, ground truth in lists and as one stacked array / tensor, host and device
    C = 7
    tiles = [synth.gt_and_pred(7500 + j, 256, 256, num_classes=C) for j in range(6)]
    gi = np.stack([_spread_ids(t["gt_inst"], 60 + j) for j, t in enumerate(tiles)])
    gsm = np.stack([t["gt_sem"] for t in tiles])
    sp, ip = cu(np.stack([t["pred_sem"] for t in tiles])), cu(np.stack([t["pred_inst"] for t in tiles]))
    idx = list(range(6))
    rec_want = datasets.CoNICDataset(sem_gts=gsm, inst_gts=gi).pre_eval_records(sp, ip, idx)
    for tag, ds in (("stacked numpy", datasets.CoNICDataset(sem_gts=gsm, inst_gts=_u16(gi))),
                    ("stacked cuda", datasets.CoNICDataset(sem_gts=cu(gsm), inst_gts=cu(_u16(gi)))),
                    ("list numpy", datasets.CoNICDataset(sem_gts=list(gsm), inst_gts=list(_u16(gi)))),
                    ("list cuda", datasets.CoNICDataset(sem_gts=[cu(x) for x in gsm], inst_gts=[cu(x) for x in _u16(gi)]))):
        seen.clear()
        _records_equal(ds.pre_eval_records(sp, ip, idx), rec_want, "CoNIC pre_eval_records " + tag)
        assert set(seen) == {"uint16" if "numpy" in tag else "torch.uint16"}, (tag, seen)
        seen.clear()
        _records_equal(ds.pre_eval_records(sp[[4, 1, 3]], ip[[4, 1, 3]], [4, 1, 3]), rec_want[[4, 1, 3]],
                       "CoNIC records, gathered indices " + tag)
        assert set(seen) == {"uint16" if "numpy" in tag else "torch.uint16"}, (tag, seen)


@gpu
def test_custom_dataset_uint16_ground_truth_equals_int32(monkeypatch):
    import torch
    from tiseg_b200 import datasets
    m = np.load(os.path.join(G, "dataset_ref.npz"))
    sems, insts = [m["p%d_gt_sem" % j] for j in range(4)], [m["p%d_gt_inst" % j] for j in range(4)]
    names = ["im%d" % j for j in range(4)]
    preds = [dict(sem_pred=m["p%d_sem_pred" % j], inst_pred=m["p%d_inst_pred" % j]) for j in range(4)]
    seen = []
    real = ops.pair_metrics_bin
    monkeypatch.setattr(ops, "pair_metrics_bin", lambda ip, ig, *a, **k: seen.append(str(ig.dtype)) or real(ip, ig, *a, **k))
    want = datasets.CustomDataset(sem_gts=sems, inst_gts=insts, names=names).pre_eval(preds, list(range(4)))
    ev_want, _ = datasets.CustomDataset(sem_gts=sems, inst_gts=insts, names=names).evaluate(want, logger="silent")
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    for tag, i16, dt in (("numpy", [_u16(x) for x in insts], "uint16"), ("cuda", [cu(_u16(x)) for x in insts], "torch.uint16")):
        seen.clear()
        ds = datasets.CustomDataset(sem_gts=sems, inst_gts=i16, names=names)
        got = ds.pre_eval(preds, list(range(4)))
        assert seen and set(seen) == {dt}, (tag, seen)
        _same(got, want, "pre_eval " + tag)
        _same(ds.evaluate(got, logger="silent")[0], ev_want, "evaluate " + tag)
    tiles = [synth.gt_and_pred(7600 + j, 200, 120) for j in range(5)]
    gi, gsm = np.stack([t["gt_inst"] for t in tiles]), np.stack([t["gt_sem"] for t in tiles])
    sp, ip = cu(np.stack([t["pred_sem"] for t in tiles])), cu(np.stack([t["pred_inst"] for t in tiles]))
    rec_want = datasets.CustomDataset(sem_gts=gsm, inst_gts=gi).pre_eval_records(sp, ip, list(range(5)))
    for ds in (datasets.CustomDataset(sem_gts=cu(gsm), inst_gts=cu(_u16(gi))), datasets.CustomDataset(sem_gts=list(gsm), inst_gts=list(_u16(gi)))):
        _records_equal(ds.pre_eval_records(sp, ip, list(range(5))), rec_want, "CustomDataset pre_eval_records")


# --------------------------------------------------------------------------- GPU: label makers
def _label_inputs():
    """(name, inst int32 with ids < 65536, sem uint8, num_angles) from the label goldens and a 1000^2 synthetic tile"""
    lg, dl = np.load(os.path.join(G, "labelgen_ref.npz")), np.load(os.path.join(G, "dirlabel_ref.npz"))
    out = [("labelgen %d" % j, lg["l%d_inst" % j], lg["l%d_sem" % j], 8) for j in range(5)]
    out += [("dirlabel %d" % j, dl["d%d_inst" % j], dl["d%d_sem" % j], int(dl["d%d_num_angles" % j]))
            for j in range(int(dl["n_cases"])) if int(dl["d%d_to_center" % j])]
    t = synth.gt_and_pred(7700, 1000, 1000)
    out.append(("synthetic 1000^2", _spread_ids(t["gt_inst"], 7), t["gt_sem"], 8))
    return out


@gpu
def test_fix_inst_and_hv_map_uint16_equal_int32():
    import torch
    cases = _label_inputs()
    for name, inst, _, _ in cases:
        i16 = _u16(inst)
        _same(ops.fix_inst(i16), ops.fix_inst(inst), "fix_inst " + name)
        _same(ops.gen_instance_hv_map(i16), ops.gen_instance_hv_map(inst), "hv map " + name)
        want_f, want_h = torch.from_numpy(ops.fix_inst(inst)).cuda(), torch.from_numpy(ops.gen_instance_hv_map(inst)).cuda()
        for tag, d in (("device", torch.from_numpy(i16).cuda()), ("misaligned device", _misaligned(i16))):
            _same(ops.fix_inst(d), want_f, "fix_inst %s %s" % (tag, name))
            _same(ops.gen_instance_hv_map(d), want_h, "hv map %s %s" % (tag, name))
    # a batch, ids up to 65535 in 300 x 301 tiles
    b = np.stack([_spread_ids(synth.gt_and_pred(7800 + j, 300, 301, n=150)["gt_inst"], 90 + j) for j in range(3)])
    _same(ops.fix_inst(_u16(b)), ops.fix_inst(b), "fix_inst batch")
    _same(ops.gen_instance_hv_map(_u16(b)), ops.gen_instance_hv_map(b), "hv map batch")


@gpu
def test_label_makers_uint16_inst_gt_give_identical_data_dicts():
    from tiseg_b200 import label_makers as lm
    makers = [("HV", lambda n: lm.HVLabelMake()), ("Bound", lambda n: lm.BoundLabelMake(edge_id=4, selem_radius=(2, 1))),
              ("Distance", lambda n: lm.DistanceLabelMake(inst_norm=True)), ("UNet", lambda n: lm.UNetLabelMake()),
              ("Direction", lambda n: lm.DirectionLabelMake(num_angles=n))]
    for name, inst, sem, n in _label_inputs():
        for mk, make in makers:
            want = make(n)(dict(sem_gt=sem.copy(), inst_gt=inst.copy(), seg_fields=[]))
            got = make(n)(dict(sem_gt=sem.copy(), inst_gt=_u16(inst), seg_fields=[]))
            assert got["inst_gt"].dtype == np.uint16 and np.array_equal(got["inst_gt"], inst)    # the input is left as given
            _same({k: v for k, v in got.items() if k != "inst_gt"}, {k: v for k, v in want.items() if k != "inst_gt"},
                  "%sLabelMake %s" % (mk, name))


# --------------------------------------------------------------------------- GPU: native reads
def _timed_names(fn):
    ctx = _lib.get_ctx(0)
    ctx.synchronize()
    ctx.timing(True)
    n0 = ctx.launch_count()
    fn()
    ctx.synchronize()
    launches = ctx.launch_count() - n0
    rep = ctx.timing_report()
    ctx.timing(False)
    return rep, launches


@gpu
def test_uint16_calls_launch_the_uint16_instantiations_and_nothing_else(monkeypatch):
    """Device-resident uint16 input: the library receives the tensor's own address, launches the uint16 instantiations
    in place of the int32 ones, launch for launch, and no other kernel; every name of the evaluation call resolves in
    bench.py's KERNEL_BYTES lookup."""
    import torch
    bench = _bench()
    C = 7
    p, ps, g, gs = _multiclass_case("conic", C)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    p, ps, gs, g32, g16 = cu(p), cu(ps), cu(gs), cu(g), cu(_u16(g))
    raw = _spread_ids(synth.gt_and_pred(7900, 320, 300)["gt_inst"], 3)
    raw32, raw16 = cu(raw), cu(_u16(raw))
    calls = {
        "multiclass": lambda g: ops.pair_metrics_multiclass(p, ps, g, gs, C),
        "assign_sem_class": lambda g: ops.assign_sem_class(g, gs, C),
        "fix_inst": lambda g: ops.fix_inst(g),
        "hv_map": lambda g: ops.gen_instance_hv_map(g),
    }
    u16_names = {"k_eqbits<uint16_t>", "k_max_id<uint16_t>", "k_inst_class_hist<uint16_t>", "k_comp_class_bits<uint16_t>",
                 "k_fix_keep<uint16_t>", "k_fix_root_slots<uint16_t>", "k_fix_list<uint16_t>", "k_fix_newid<uint16_t>",
                 "k_inst_stats<uint16_t>", "k_hv_map<uint16_t>"}
    seen_ptrs = []
    real_call = _lib.Context.call
    monkeypatch.setattr(_lib.Context, "call", lambda self, name, *a: seen_ptrs.append((name, [x.value for x in a if hasattr(x, "value")])) or real_call(self, name, *a))
    for what, fn in calls.items():
        src32, src16 = (g32, g16) if what in ("multiclass", "assign_sem_class") else (raw32, raw16)
        rep32, n32 = _timed_names(lambda: fn(src32))
        seen_ptrs.clear()
        rep16, n16 = _timed_names(lambda: fn(src16))
        assert len(seen_ptrs) == 1 and seen_ptrs[0][0].endswith(("_u16", "_u16gt")), seen_ptrs
        assert src16.data_ptr() in seen_ptrs[0][1], what
        assert n16 == n32, (what, n16, n32)
        typed = {k for k in rep16 if "<uint16_t>" in k}
        assert typed and typed <= u16_names, (what, sorted(rep16))
        twin = lambda k: "k_eqbits<int32_t>" if k == "k_eqbits<uint16_t>" else k.replace("<uint16_t>", "")
        back = Counter()
        for k, (cnt, _) in rep16.items():
            back[twin(k)] += cnt
        assert back == Counter({k: cnt for k, (cnt, _) in rep32.items()}), (what, sorted(rep16.items()), sorted(rep32.items()))
        for k in rep16:
            assert _resolves(bench, k) == _resolves(bench, twin(k)), (what, k)
            if what == "multiclass":
                assert _resolves(bench, k), k
    multi16, _ = _timed_names(lambda: calls["multiclass"](g16))
    assert {"k_eqbits<uint16_t>", "k_max_id<uint16_t>", "k_inst_class_hist<uint16_t>", "k_comp_class_bits<uint16_t>"} <= set(multi16)
    assert "k_eqbits<int32_t>" in multi16 and multi16["k_max_id"][0] == 1      # the prediction side stays int32
