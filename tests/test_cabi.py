"""CPU-side checks of the drop-in boundary: the C-ABI library builds for sm_100a, loads, and exports
exactly the symbols include/tiseg_b200.h declares; without a GPU it fails loudly (no CPU fallback)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from tiseg_b200 import _lib
    return _lib


def _declared():
    src = open(os.path.join(ROOT, "include", "tiseg_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(tiseg_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported_and_bound(lib):
    names = _declared()
    assert len(names) >= 20
    so = ctypes.CDLL(lib.SO_PATH)
    for n in names:
        assert hasattr(so, n), "declared in tiseg_b200.h but not exported: " + n
    assert sorted(lib.SIGNATURES) == names, "python binding table and header disagree"
    assert lib.load().tiseg_version() >= 100


def test_no_cpu_fallback(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import numpy as np
    from tiseg_b200 import ops
    with pytest.raises(lib.TisegError, match="no CUDA device|NOGPU|status 3"):
        ops.label(np.zeros((4, 4), np.int32))
    # the product never imports the oracle
    pkg = os.path.join(ROOT, "tissue-image-segmentation_b200")
    for f in os.listdir(pkg):
        if f.endswith(".py"):
            assert "oracle" not in open(os.path.join(pkg, f)).read().replace("CPU oracle", ""), f


def test_label_maker_classes_mirror_the_reference_constructors():
    """Host-side mirror of tiseg/datasets/ops: same class names and constructor arguments; the one configuration the
    reference itself cannot run (UNetLabelMake with class weights, unet_map.py:120-124) is refused, not emulated."""
    import inspect
    from tiseg_b200 import label_makers as lm
    assert list(inspect.signature(lm.BoundLabelMake.__init__).parameters)[1:] == ["edge_id", "selem_radius"]
    assert list(inspect.signature(lm.DistanceLabelMake.__init__).parameters)[1:] == ["inst_norm"]
    assert list(inspect.signature(lm.UNetLabelMake.__init__).parameters)[1:] == ["wc", "w0", "sigma"]
    assert lm.BoundLabelMake(selem_radius=2).radius == (2, 2)
    with pytest.raises(NotImplementedError):
        lm.UNetLabelMake(wc={1: 2.0})


def test_reference_signatures():
    """The reference-named entry points take the reference's parameters, in the reference's order (no GPU needed):
    inst_metrics.py:95,138,232; direct_diff_map.py:95; cdnet.py:354; multi_task_cdnet.py:548,220."""
    import inspect
    import tiseg_b200  # noqa: F401
    from tiseg_b200 import metrics as M, segmentors as S
    names = lambda f: list(inspect.signature(f).parameters)
    assert names(M.pre_eval_aji) == ["inst_pred", "inst_gt", "pred_id_list_per_class", "gt_id_list_per_class", "num_classes",
                                     "reduce_zero_label"]
    assert names(M.pre_eval_pq) == names(M.pre_eval_aji)
    assert names(M.pre_eval_bin_pq) == ["inst_pred", "inst_gt", "match_iou"]
    assert inspect.signature(M.pre_eval_bin_pq).parameters["match_iou"].default == 0.5
    assert names(S.generate_direction_differential_map) == ["dir_map", "direction_classes", "background", "use_reg"]
    for cls in (S.CDNet, S.MultiTaskCDNet):
        assert names(cls._ddm_enhencement) == ["sem_logit", "dd_map", "point_logit"]
    assert names(S.MultiTaskCDNet.postprocess)[1:] == ["inner_pred", "sem_pred"] or names(S.MultiTaskCDNet.postprocess)[1:] == ["tc_pred", "sem_pred"]
    assert names(M.pre_eval_all_semantic_metric)[:4] == ["pred_label", "target_label", "num_classes", "ignore_index"]
    # label makers: constructor arguments and defaults of tiseg/datasets/ops/{direction_map.py:14, distance_map.py:37,
    # bound_map.py:12, unet_map.py:30}
    from tiseg_b200 import label_makers as L
    sig = lambda cls: [(k, v.default) for k, v in inspect.signature(cls.__init__).parameters.items() if k != "self"]
    assert sig(L.DirectionLabelMake) == [("to_center", True), ("num_angles", 8)]
    assert sig(L.DistanceLabelMake) == [("inst_norm", True)]
    assert sig(L.BoundLabelMake) == [("edge_id", 2), ("selem_radius", 3)]
    assert sig(L.UNetLabelMake) == [("wc", None), ("w0", 10.0), ("sigma", 5.0)]
    assert [k for k in inspect.signature(S.MultiTaskCDNet.__init__).parameters][1:] == ["num_classes", "num_angles", "test_cfg", "if_ddm",
                                                                                       "use_regression"]



def test_library_reads_no_environment():
    """The CUDA library's results and launches depend on its arguments alone: no source under csrc/ reads an environment
    variable, so nothing set in a user's shell or a job profile can switch a stage to another implementation."""
    csrc = os.path.join(ROOT, "tissue-image-segmentation_b200", "csrc")
    found = []
    for dirpath, _, files in os.walk(csrc):
        for f in files:
            path = os.path.join(dirpath, f)
            with open(path, encoding="utf-8", errors="replace") as fh:
                found += ["%s:%d" % (os.path.relpath(path, ROOT), i + 1) for i, line in enumerate(fh) if "getenv" in line]
    assert not found, "environment reads in the library: " + ", ".join(found)
