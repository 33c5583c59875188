"""Train-time label makers of ``tiseg/datasets/ops`` on the GPU (SURVEY.md §8f rank 4).

Same class names, constructor arguments and ``data`` dict protocol as the reference (``DistanceLabelMake``:
datasets/ops/distance_map.py:23-142, ``HVLabelMake``: hv_map.py:100-114, ``BoundLabelMake``: bound_map.py:6-89).
``UNetLabelMake``: unet_map.py:7-127, ``DirectionLabelMake``: direction_map.py:11-193 with ``to_center=True``).
``data["inst_gt"]`` may be int32 or uint16; a uint16 map is read as it is and gives the same ``data`` dict.
"""
import numpy as np

from . import ops


class HVLabelMake(object):
    def __call__(self, data):
        hv = ops.gen_instance_hv_map(data["inst_gt"])
        data["hv_gt"] = hv.transpose(2, 0, 1)
        data["seg_fields"].append("hv_gt")
        return data


class BoundLabelMake(object):
    def __init__(self, edge_id=2, selem_radius=3):
        self.edge_id = edge_id
        if isinstance(selem_radius, int):
            selem_radius = (selem_radius, selem_radius)
        self.radius = selem_radius

    def __call__(self, data):
        inst_gt = ops.fix_inst(data["inst_gt"])
        sem_gt, bound = ops.bound_label(data["sem_gt"], inst_gt, self.edge_id, self.radius)
        assert np.array_equal(np.asarray(sem_gt) > 0, np.asarray(inst_gt) > 0)
        data["sem_gt"] = sem_gt.astype(np.asarray(data["sem_gt"]).dtype, copy=False)
        data["sem_gt_w_bound"] = bound.astype(data["sem_gt"].dtype, copy=False)
        data["seg_fields"].append("sem_gt_w_bound")
        return data


class DistanceLabelMake(object):
    def __init__(self, inst_norm=True):
        self.inst_norm = inst_norm

    def __call__(self, data):
        sem_gt = np.asarray(data["sem_gt"])
        inst_gt = ops.fix_inst(data["inst_gt"])
        sem_gt = np.where(inst_gt == 0, 0, sem_gt).astype(sem_gt.dtype)
        data["sem_gt"] = sem_gt
        data["dist_gt"] = ops.instance_distance_map(inst_gt, self.inst_norm)
        data["seg_fields"].append("dist_gt")
        return data


class UNetLabelMake(object):
    def __init__(self, wc=None, w0=10.0, sigma=5.0):
        if wc is not None:
            # unet_map.py:120-124 builds ``np.zeros_like(inst_gt.shape[:2])`` (a length-2 vector) and indexes it with an
            # image-sized mask: the reference itself raises for any wc
            raise NotImplementedError("UNetLabelMake(wc=...) fails in the reference (unet_map.py:121-123)")
        self.wc, self.w0, self.sigma = wc, w0, sigma

    def __call__(self, data):
        sem_gt = np.asarray(data["sem_gt"])
        inst_gt = ops.fix_inst(data["inst_gt"])
        sem_gt = np.where(inst_gt == 0, 0, sem_gt).astype(sem_gt.dtype)
        data["sem_gt"] = sem_gt
        inner, wmap = ops.unet_weight_map(inst_gt, self.w0, self.sigma)
        data["loss_weight_map"] = wmap
        data["sem_gt_inner"] = np.where(inner == 0, 0, sem_gt).astype(sem_gt.dtype)
        data["seg_fields"].append("sem_gt_inner")
        return data


class DirectionLabelMake(object):
    """build direction label & point label for any dataset (direction_map.py:11-84)."""

    def __init__(self, to_center=True, num_angles=8):
        if not to_center:
            # calculate_distance_to_centralridge (direction_map.py:172-183): no config of the reference selects it
            raise NotImplementedError("DirectionLabelMake(to_center=False) is not built")
        self.to_center = to_center
        self.num_angles = num_angles

    def __call__(self, data):
        sem_gt = np.asarray(data["sem_gt"])
        inst_gt = ops.fix_inst(data["inst_gt"])
        data["sem_gt"] = np.where(inst_gt == 0, 0, sem_gt).astype(sem_gt.dtype)
        r = ops.direction_labels(inst_gt, self.num_angles)
        data["dist_gt"] = r["dist_gt"]
        data["point_gt"] = r["point_gt"]
        data["dir_gt"] = r["dir_gt"].astype(np.int64)
        data["reg_dir_gt"] = r["reg_dir_gt"]
        # direction_map.py:73-76: np.zeros_like(dir_map) (int64) unless there are eight angles
        data["loss_weight_map"] = r["loss_weight_map"] if self.num_angles == 8 else np.zeros_like(data["dir_gt"])
        return data
