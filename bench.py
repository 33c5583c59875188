#!/usr/bin/env python
"""bench.py — post-process + evaluation throughput of the tiseg test-time instance pipeline on B200.

A "step" is one pass of the path (segmentor tail -> post-process -> Dataset.pre_eval metrics) over one batch of synthetic
tiles per GPU.  Workloads = the five BASELINE.json configurations (`--workload`, default = configs[1], the 1000x1000
configuration the metric is quoted on):

  dist_monuseg_1000   DIST MoNuSeg 1000^2: argmax of the 2-class head, distance-map markers + ordered watershed
                      (dist.py:275-284), semantic counts + binary AJI / PQ (custom.py:252-283)             22 B/px
  unet_cpm17_256      UNet-VGG16 CPM17 256^2: argmax, fill holes / remove small / label / dilation
                      (unet.py:71-93), semantic counts + binary AJI / PQ                                     18 B/px
  hover_consep_1000   HoVer-Net CoNSeP 1000^2: Sobel-of-HV energy markers + fp64 watershed
                      (hovernet.py:283-365), semantic counts (3 classes) + binary AJI / PQ                   38 B/px
  cdnet_consep_1000   CDNet CoNSeP 1000^2: direction-guided refinement (cdnet.py:183-217, 354-367), CUNet-style
                      post-process radius 3 (cdnet.py:96-119), semantic counts + binary AJI / PQ             62 B/px
  conic_sweep_256     CoNIC-scale sweep, 256^2 tiles, 7 classes: UNet-family post-process + CoNICDataset evaluation
                      (binary AND per-class AJI / PQ, conic.py:157-196); 4981 tiles = 9.7 steps of 512       38 B/px

  python bench.py --gpus N --steps K --warmup W [--workload NAME]     # this repo (CUDA, sm_100a)
  python bench.py --impl reference --gpus N --steps K ...              # the reference's CPU path (oracle port) on host cores

One JSON line on stdout (rank 0).  value = tiles/s with inputs resident in HBM; e2e = tiles/s through the same calls fed
from pinned HOST buffers (H2D of every input + D2H of the metric records inside the timed region).  After the timed
regions the GPU arm re-runs the `--cpu-tiles` tiles that the cpu_baseline leg processes and compares its per-tile records
with the oracle's bit for bit; a mismatch is reported in `check` and makes the exit code 3.

`--dump-outputs DIR` writes what the last timed step computed as DIR/<name>.npy (float32 / float64, at most 64 MB): the
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


# --------------------------------------------------------------------------- workloads
class Workload:
    """One BASELINE configuration: synthetic tiles, the GPU step through the operator API, the same tile through the CPU
    oracle (reference cost profile), and the per-tile metric record both produce."""
    name = metric = None
    H = W = 1000
    C = 2                      # classes of the semantic evaluation
    batch = 64                 # tiles per step per GPU (default)
    pipe_bpp = 0               # algorithmic bytes per pixel of one tile through the whole path (SURVEY.md §8d)
    instances = 900
    config_id = 2
    keys = ()                  # host-fed arrays, in the order they are uploaded
    net_keys = ()              # the subset the CNN would leave on the device
    multi = False              # per-class AJI / PQ as well (CoNIC)
    dihedral = True            # the batch may be filled with rotated / flipped copies of the distinct tiles (not when a
                               # head's CHANNELS mean directions: HV maps, direction classes)

    def make_tile(self, index):
        raise NotImplementedError

    def prep(self, t):
        """tile dict -> the arrays the step consumes (adds the TTA axis where the op wants one)"""
        return {k: t[k] for k in self.keys}

    def gpu_step(self, ops, src):
        """-> dict of per-tile record tensors: aji [B,2], pq [B,4], counts [B,5,C] (+ caji [B,C,2], cpq [B,C,4]), and the
        maps they were computed from: sem [B,H,W] uint8, inst [B,H,W] int32"""
        raise NotImplementedError

    def cpu_tile(self, t, literal=True):
        """the reference path for one tile on the CPU -> the same record as numpy arrays"""
        raise NotImplementedError

    def record_width(self):
        return 6 + 5 * self.C + (6 * self.C if self.multi else 0)

    @staticmethod
    def flat(rec):
        """record dict of batched tensors -> [B, R] float64 tensor (exact: integers and fp64 sums)"""
        import torch
        parts = [rec["aji"], rec["pq"], rec["counts"].reshape(rec["counts"].shape[0], -1).double()]
        if "caji" in rec:         # (the reference accumulates the per-class records in float32 arrays, inst_metrics.py:101-102)
            parts += [rec["caji"].reshape(rec["caji"].shape[0], -1).float().double(),
                      rec["cpq"].reshape(rec["cpq"].shape[0], -1).float().double()]
        return torch.cat(parts, dim=1)

    def _cpu_eval(self, sem, inst, t, literal):
        from oracle import metrics as om
        semres = om.pre_eval_all_semantic_metric(sem, t["gt_sem"], self.C, reduce_zero_label=False)
        ip, ig = om.re_instance(inst), om.re_instance(t["gt_inst"])
        aji = om.pre_eval_bin_aji(ip, ig, literal=literal)
        pq = om.pre_eval_bin_pq(ip, ig, literal=literal)
        tp, tn, fp, fn, pr, gt = [np.asarray(x, np.float64) for x in semres]
        row = [np.float64(aji[0]), np.float64(aji[1]), *[np.float64(v) for v in pq], *np.concatenate([tp, fp, fn, pr, gt])]
        if self.multi:
            dp = om.assign_sem_class_to_insts(ip, sem, self.C)
            dg = om.assign_sem_class_to_insts(ig, t["gt_sem"], self.C)
            caji = om.pre_eval_aji(ip, ig, dp, dg, self.C, reduce_zero_label=False, literal=literal)
            cpq = om.pre_eval_pq(ip, ig, dp, dg, self.C, reduce_zero_label=False, literal=literal)
            row += list(np.stack(caji, 1).astype(np.float64).ravel()) + list(np.stack(cpq, 1).astype(np.float64).ravel())
        return np.array(row, np.float64)


class DistMonuseg(Workload):
    name, metric = "dist_monuseg_1000", "postproc+eval tiles/s @1000x1000 (DIST MoNuSeg config)"
    pipe_bpp, config_id = 22, 2
    keys, net_keys = ("sem_logit", "dist_logit", "gt_inst", "gt_sem"), ("sem_logit", "dist_logit")

    def make_tile(self, index):
        from tiseg_b200 import synth
        return synth.tile_dist(2, index, H=self.H, W=self.W)

    def prep(self, t):
        d = {k: t[k] for k in self.keys}
        d["sem_logit"] = t["sem_logit"][None]                       # [T = 1, C, H, W]
        return d

    def gpu_step(self, ops, src):
        cls = ops.softmax_argmax(src["sem_logit"])
        inst = ops.postproc_dist(src["dist_logit"])
        aji, pq = ops.pair_metrics_bin(inst, src["gt_inst"])
        counts, _ = ops.sem_counts(cls, src["gt_sem"], self.C)
        return dict(aji=aji, pq=pq, counts=counts, sem=cls, inst=inst)

    def cpu_tile(self, t, literal=True):
        from oracle import postprocess as opp
        sem = opp.argmax_classes(opp.softmax(t["sem_logit"]))
        _, inst = opp.dist_postprocess(sem, t["dist_logit"], literal=literal)
        return self._cpu_eval(sem, inst, t, literal)


class UnetCpm17(Workload):
    name, metric = "unet_cpm17_256", "postproc+eval tiles/s @256x256 (UNet-VGG16 CPM17 config)"
    H = W = 256
    batch, pipe_bpp, instances, config_id = 512, 18, 60, 1
    keys, net_keys = ("sem_logit", "gt_inst", "gt_sem"), ("sem_logit",)
    radius, max_class = 1, 1

    def make_tile(self, index):
        from tiseg_b200 import synth
        return synth.tile_unet(self.config_id, index, self.H, self.W, self.C)

    def prep(self, t):
        d = {k: t[k] for k in self.keys}
        d["sem_logit"] = t["sem_logit"][None]
        return d

    def gpu_step(self, ops, src):
        cls = ops.softmax_argmax(src["sem_logit"])
        sem, inst = ops.postproc_unet(cls, self.max_class, self.radius, None)
        counts, _ = ops.sem_counts(sem, src["gt_sem"], self.C)
        if self.multi:
            r = ops.pair_metrics_multiclass(inst, sem, src["gt_inst"], src["gt_sem"], self.C)
            return dict(aji=r["bin_aji"], pq=r["bin_pq"], counts=counts, caji=r["aji"], cpq=r["pq"], sem=sem, inst=inst)
        aji, pq = ops.pair_metrics_bin(inst, src["gt_inst"])
        return dict(aji=aji, pq=pq, counts=counts, sem=sem, inst=inst)

    def cpu_tile(self, t, literal=True):
        from oracle import postprocess as opp
        cls = opp.argmax_classes(opp.softmax(t["sem_logit"]))
        sem, inst = opp.unet_family_postprocess(cls, radius=self.radius)
        return self._cpu_eval(sem, inst, t, literal)


class ConicSweep(UnetCpm17):
    name, metric = "conic_sweep_256", "postproc+eval tiles/s @256x256, 7 classes (CoNIC-scale sweep, per-class AJI/PQ)"
    C, pipe_bpp, config_id, multi, max_class = 7, 38, 5, True, 6


class HoverConsep(Workload):
    name, metric = "hover_consep_1000", "postproc+eval tiles/s @1000x1000 (HoVer-Net CoNSeP config)"
    C, batch, pipe_bpp, config_id, dihedral = 3, 16, 38, 3, False
    keys, net_keys = ("sem_logit", "fore_map", "hv_map", "gt_inst", "gt_sem"), ("sem_logit", "fore_map", "hv_map")

    def make_tile(self, index):
        from tiseg_b200 import synth
        return synth.tile_hover(3, index, H=self.H, W=self.W)

    def prep(self, t):
        d = {k: t[k] for k in self.keys}
        d["sem_logit"] = t["sem_logit"][None]
        return d

    def gpu_step(self, ops, src):
        cls = ops.softmax_argmax(src["sem_logit"])
        inst = ops.postproc_hover(src["fore_map"], src["hv_map"])
        aji, pq = ops.pair_metrics_bin(inst, src["gt_inst"])
        counts, _ = ops.sem_counts(cls, src["gt_sem"], self.C)
        return dict(aji=aji, pq=pq, counts=counts, sem=cls, inst=inst)

    def cpu_tile(self, t, literal=True):
        from oracle import postprocess as opp
        sem = opp.argmax_classes(opp.softmax(t["sem_logit"]))
        inst, _ = opp.hover_post_proc(t["fore_map"], t["hv_map"])
        return self._cpu_eval(sem, inst, t, literal)


class CdnetConsep(Workload):
    name, metric = "cdnet_consep_1000", "postproc+eval tiles/s @1000x1000 (CDNet CoNSeP config, if_ddm)"
    batch, pipe_bpp, config_id, dihedral = 16, 62, 4, False
    keys, net_keys = ("sem_logit", "dir_logit", "point_logit", "gt_inst", "gt_sem"), ("sem_logit", "dir_logit", "point_logit")

    def make_tile(self, index):
        from tiseg_b200 import synth
        return synth.tile_cdnet(4, index, H=self.H, W=self.W, T=1)

    def gpu_step(self, ops, src):
        r = ops.cdnet_refine(src["sem_logit"], src["dir_logit"], src["point_logit"], if_ddm=True)
        sem, inst = ops.postproc_unet(r["cls"], 2, 3, 2)
        aji, pq = ops.pair_metrics_bin(inst, src["gt_inst"])
        counts, _ = ops.sem_counts(sem, src["gt_sem"], self.C)
        return dict(aji=aji, pq=pq, counts=counts, sem=sem, inst=inst)

    def cpu_tile(self, t, literal=True):
        from oracle import postprocess as opp
        prob, _, _ = opp.cdnet_inference_tail(list(t["sem_logit"]), list(t["dir_logit"]), list(t["point_logit"]), if_ddm=True)
        cls = opp.argmax_classes(prob)
        sem, inst = opp.unet_family_postprocess(cls, radius=3, edge_id=2)
        return self._cpu_eval(sem, inst, t, literal)


WORKLOADS = {w.name: w for w in (DistMonuseg, UnetCpm17, HoverConsep, CdnetConsep, ConicSweep)}

# kept for the helper scripts that import this module
H = W = 1000


def make_tiles(n_distinct, seed0, wl=None):
    """n_distinct seeded synthetic tiles of the workload (tiseg_b200.synth, SURVEY.md §8d generator)."""
    import tiseg_b200  # noqa: F401
    wl = wl or DistMonuseg()
    return [wl.prep(wl.make_tile(seed0 + j)) for j in range(n_distinct)]


def stack_batch(tiles, batch, dihedral=True):
    """Fill a batch from the distinct tiles, cycling through the 8 dihedral variants so no two are equal (plain copies
    when the workload's heads carry directions in their channels)."""
    def var(key, a, k):
        a = np.rot90(a, k % 4, axes=(-2, -1))
        if k >= 4:
            a = np.flip(a, axis=-1)
        return np.ascontiguousarray(a)
    keys = list(tiles[0].keys())
    out = {k: [] for k in keys}
    for b in range(batch):
        t = tiles[b % len(tiles)]
        k = (b // len(tiles)) % 8 if dihedral else 0
        for key in keys:
            out[key].append(var(key, t[key], k))
    return {k: np.stack(v) for k, v in out.items()}


DUMP_BYTES = 64 * 10 ** 6          # --dump-outputs writes at most this much


def outputs_to_dump(rec, seed=0):
    """One step's outputs (``Workload.gpu_step``) as host arrays for --dump-outputs: every per-tile record in full
    (float64), and the sem / inst maps of a fixed, seeded sample of the batch's tiles (float32, exact below 2**24) with
    their batch indices in ``sample_tiles``, at most DUMP_BYTES in all."""
    import torch
    out = {k: v.double().cpu().numpy() for k, v in rec.items() if k not in ("sem", "inst")}
    B, H, W = rec["inst"].shape
    if int(rec["inst"].max()) >= 1 << 24:
        raise ValueError("instance ids of 2**24 and above are not exact in float32")
    room = DUMP_BYTES - sum(v.nbytes for v in out.values()) - 8 * B
    idx = np.sort(np.random.default_rng(seed).choice(B, min(B, room // (2 * 4 * H * W)), replace=False))
    sel = torch.from_numpy(idx).to(rec["inst"].device)
    out["sample_tiles"] = idx.astype(np.float64)
    for k in ("sem", "inst"):
        out[k] = rec[k].index_select(0, sel).float().cpu().numpy()
    return out


# Algorithmic bytes per pixel and LAUNCH of every kernel's own inputs + outputs, touched once (DESIGN.md §4); a step's
# bytes are that times the pixels of the batch times the launches of the kernel in the step.  None = the kernel works on
# O(components) / O(words) tables, not on pixels: no per-pixel roofline applies (its time still counts in the step).  A
# kernel name that is not listed is an error: nothing gets a default.
_T = None
KERNEL_BYTES_COMMON = {
    # streaming front
    "k_argmax_logits": "4*C+1", "k_softmax_argmax": "4*C+1+4*C", "k_sem_counts": 2, "memset": _T,
    # bit-plane CCL (bitccl.cuh): planes in, bitmap out
    "k_eqbits": 4 + 5 / 8.0, "k_bitccl_tile": _T, "k_bitccl_border": _T, "k_bitccl_resolve": _T,
    "k_rank_rowtot": _T, "k_rank_rowscan": _T, "k_rank_place_bits": _T, "k_rank_fused": _T, "k_rank_bits": 4,
    # pair metrics
    "k_pair_bits": _T, "k_pair_zero_big": _T, "k_inst_init": _T, "k_pair_best": _T, "k_pair_argbest": _T, "k_aji_gt": _T,
    "k_aji_pred": _T, "k_metrics_final": _T, "k_inst_class_hist": 5, "k_inst_class_pick": _T, "k_comp_class_bits": _T, "k_max_id": 4, "k_zero_class_hist": _T,
    # pixel forests (labelling API, UNet family, HoVer-Net)
    "(k_ccl_local<Img, 2": 8, "(k_ccl_local<Img, 1": 5, "(k_ccl_border": _T, "k_ccl_flatten": 8, "k_apply_rank": 8,
    "k_ccl_areas": 4, "k_keep_large": 5, "k_border_touch": _T, "k_fill_from_forest": 6, "k_grey_morph": 8,
    "k_unet_compose": 13, "k_unet_advance": _T, "k_class_presence": 1, "k_class_mask": 2, "k_zero_class": 1, "k_paint_class": 2,
    "k_zero_prefix_u8": _T, "k_count_seen": _T, "k_mark_values": 4, "k_lookup_values": 8, "k_label_hist": 4,
    "k_drop_small_labels": 8, "k_threshold_ge": 5,
}
KERNEL_BYTES = {
    "dist_monuseg_1000": {
        "k_dist_prep": 4 + 1 + 1 / 8.0, "k_plateau_bits": 1 + 2 / 8.0, "k_filter_root_bits": _T,
        "k_marker_scatter": _T, "k_mask_area": _T, "k_label_clean": _T, "k_dense_tiles": _T, "k_init_label_tables": _T,
        "k_blob_init": _T, "k_blob_roots": _T, "k_blob_mark": _T, "k_blob_runs": _T, "k_huge_clean": _T, "k_flood_count": _T, "k_flood_offsets": _T,
        "k_flood_scatter": _T, "k_ws_flood_par": 1 + 4 + 4,        # level image + seeds in, labels out (mask pixels dominate)
        "k_ws_hist": _T, "k_pick_bg": _T, "k_first_bits": _T, "k_arrange_lut": _T, "k_wsl_remove": 4 + 4,
    },
    "unet_cpm17_256": {}, "conic_sweep_256": {},
    "hover_consep_1000": {
        "k_hv_minmax": 8, "k_hv_normalize": 16, "k_sobel_row": 12, "k_sobel_col": 16, "k_hover_energy": 28, "k_gauss3_row": 16,
        "k_gauss3_col_neg": 16, "k_ellipse5": 2, "k_mm_init": _T, "k_ws_seed": 12, "k_blob_init": _T, "k_blob_roots": _T,
        "k_blob_bbox": 4, "k_blob_offsets": _T, "k_blob_prefix": _T, "k_rank_blobs": 14, "k_flood_count_ranked": _T,
        "k_flood_offsets": _T, "k_flood_scatter_ranked": _T, "(k_ws_flood_ranked": 2 + 4 + 4 + 4, "k_ws_flood_f64": _T,
        "k_resize_up2": 20, "k_resize_down2_nearest": 8,
    },
    "cdnet_consep_1000": {
        "k_dir_map": 36 + 4 + 1, "k_ddm_mm_init": _T, "k_ddm_levels": 2, "k_ddm_mean": 5, "k_key_init": _T, "k_point_mean": 8,
        "k_ddm_enhance": 12 + 8 + 4 + 1,
    },
}


UNKNOWN = []


def kernel_bytes_per_px(wl, name):
    """-> bytes per pixel (float), or None for a table kernel.  Raises on an unknown kernel."""
    for table in (KERNEL_BYTES[wl.name], KERNEL_BYTES_COMMON):
        for prefix, b in table.items():
            if name.startswith(prefix):
                if isinstance(b, str):
                    return float(eval(b, {"C": wl.C}))
                return b
    if os.environ.get("TISEG_BENCH_ALLOW_UNKNOWN"):         # (table maintenance only: lists the names instead of failing)
        UNKNOWN.append(name)
        return None
    raise KeyError("bench.py: kernel %r has no entry in KERNEL_BYTES for workload %s" % (name, wl.name))


# --------------------------------------------------------------------------- reference arm (CPU)
def _cpu_tile(args):
    """The reference's path for one tile, literal cost profile (np.vectorize h-reconstruction, per-instance masks in
    AJI / PQ, which restate inst_metrics.py:25-67 and :150-229 line for line): oracle port."""
    wl_name, index = args
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    import tiseg_b200  # noqa: F401
    wl = WORKLOADS[wl_name]()
    t = wl.make_tile(index)
    t0 = time.perf_counter()
    rec = wl.cpu_tile(t, literal=True)
    return time.perf_counter() - t0, rec


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import multiprocessing as mp
    wl = WORKLOADS[a.workload]()
    cores = os.cpu_count() or 1
    workers = max(1, min(cores, 32))
    per_step = workers * (1 if wl.H >= 1000 else 8)          # one 1000^2 tile (or eight 256^2 tiles) per worker per step
    ctx = mp.get_context("spawn")
    with ctx.Pool(workers) as pool:
        seed = 0
        for _ in range(a.warmup):
            pool.map(_cpu_tile, [(wl.name, seed + i) for i in range(per_step)]); seed += per_step
        t0 = time.perf_counter()
        for _ in range(a.steps):
            pool.map(_cpu_tile, [(wl.name, seed + i) for i in range(per_step)]); seed += per_step
        dt = time.perf_counter() - t0
    value = per_step * a.steps / dt
    line = {
        "impl": "reference", "metric": wl.metric, "value": value, "unit": "tiles/s", "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/int32 labels, fp32 softmax, fp64 IoU", "data": "synthetic",
        "config": {"workload": wl.name, "tile": [wl.H, wl.W], "tiles_per_step": per_step, "instances_per_tile": wl.instances},
        "cpu_baseline": {"value": value, "unit": "tiles/s", "cores": workers, "kind": "port",
                         "sample": "%d tiles per step, one process per tile; oracle port of the reference path: scipy.ndimage / "
                                   "OpenCV are the real libraries, the AJI / PQ part restates inst_metrics.py:25-67, 150-229 line "
                                   "for line, the five scikit-image calls are the C restatement (/root/reference is Python and "
                                   "not importable on this box: mmcv / scikit-image absent)" % per_step},
        "e2e": {"value": value, "unit": "tiles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# --------------------------------------------------------------------------- this repo (CUDA)
class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.QUERY,
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush(); self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(index):
    """Run this rank on the CPU cores next to its GPU, so that the pinned staging buffers (first touch) live in the
    memory of the same socket and host-to-device copies do not cross the inter-socket link.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * w + b for w, m in enumerate(words) for b in range(64) if (m >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if cpus:
            os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:
        return None


def run_b200(a):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    bind_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import tiseg_b200  # noqa: F401
    from tiseg_b200 import _lib, ops, parallel

    wl = WORKLOADS[a.workload]()
    B = a.batch or wl.batch
    R = wl.record_width()
    tiles = make_tiles(a.distinct, seed0=1000 * rank, wl=wl)
    host = stack_batch(tiles, B, wl.dihedral)
    pinned = {k: torch.from_numpy(v).pin_memory() for k, v in host.items()}
    devt = {k: v.to(dev) for k, v in pinned.items()}
    pinned_np = {k: v.numpy() for k, v in pinned.items()}
    ctx = _lib.get_ctx(local)
    acc = torch.zeros(R, dtype=torch.float64, device=dev)
    last = {}                                              # outputs of the latest plain step (--dump-outputs)

    def step(src):
        last["rec"] = wl.gpu_step(ops, src)
        acc.add_(wl.flat(last["rec"]).sum(0))
        return acc

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(src, steps, with_d2h, fork=None, join=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launch_count()
        e0.record()
        if src is devt and join is not None:
            fork()                                         # the value lanes start after the start event
        for _ in range(steps):
            with _lib.device_outputs():
                r = step(src)
            if with_d2h:
                r.cpu()                                    # the step's metric record comes back to the host
        if src is devt and join is not None:
            join()                                         # the value lanes rejoin the timing stream
        if world > 1:
            dist.all_reduce(acc)                           # the only collective: metric accumulators
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), ctx.launch_count() - l0

    # clocks and throttle reasons are sampled from the warm-up to the end of the end-to-end measurement (the timed
    # regions themselves last tens of milliseconds, less than one nvidia-smi sampling period)
    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(max(a.warmup, 3)):
        with _lib.device_outputs():
            step(devt)
    # The resident-input step is a fixed chain of launches with no host decision in it: capture it once into a CUDA graph
    # and replay it (the library's calls are stream-ordered; its workspace and torch's outputs keep their addresses).
    # --no-graph times the plain launches instead.
    launches_per_step = None
    if not a.no_graph:
        # one graph per value lane (own stream, own workspace, own accumulator): successive steps alternate between the
        # lanes, so the latency-bound kernels of one step share the SMs with the streaming kernels of the next.  Every
        # step is still one full pass over one batch.
        VL = max(1, a.value_lanes)
        vstreams = [torch.cuda.Stream(dev) for _ in range(VL)]
        vacc = [torch.zeros(R, dtype=torch.float64, device=dev) for _ in range(VL)]
        vout = [None] * VL                                 # each graph's outputs: rewritten in place by every replay
        graphs = []

        def lane_step(k):
            vout[k] = wl.gpu_step(ops, devt)
            vacc[k].add_(wl.flat(vout[k]).sum(0))

        torch.cuda.synchronize()
        for k in range(VL):
            with _lib.lane(10 + k, vstreams[k]), _lib.device_outputs():
                for _ in range(3):
                    lane_step(k)                                   # grow this lane's workspace before the capture
            torch.cuda.synchronize()
            lctx = None
            with _lib.lane(10 + k):
                lctx = _lib.get_ctx(local)
            l0 = lctx.launch_count()
            gk = torch.cuda.CUDAGraph()
            with _lib.lane(10 + k), _lib.device_outputs():
                with torch.cuda.graph(gk, stream=vstreams[k]):
                    lane_step(k)
            launches_per_step = lctx.launch_count() - l0
            graphs.append(gk)
        _lib.get_ctx(local)                                # re-bind the default context to the ordinary stream
        plain_step = step
        turn = [0]

        def step(src):                                     # noqa: F811  (timed() looks the name up at call time)
            if src is not devt:
                return plain_step(src)
            k = turn[0] % VL
            turn[0] += 1
            with torch.cuda.stream(vstreams[k]):
                graphs[k].replay()
            return acc

        def fork_value_lanes():
            cur = torch.cuda.current_stream(dev)
            for k in range(VL):
                vstreams[k].wait_stream(cur)

        def join_value_lanes():
            cur = torch.cuda.current_stream(dev)
            for k in range(VL):
                cur.wait_stream(vstreams[k])
            acc.add_(torch.stack(vacc).sum(0))
            for v in vacc:
                v.zero_()
        for v in vacc:
            v.zero_()
        fork_value_lanes()
        for _ in range(2 * VL):
            step(devt)
        join_value_lanes()
        turn[0] = 0
    acc.zero_()
    ms, launches = timed(devt, a.steps, with_d2h=False, fork=None if a.no_graph else fork_value_lanes,
                         join=None if a.no_graph else join_value_lanes)
    if launches_per_step is not None:
        launches = launches_per_step * a.steps             # replayed launches are not seen by the library's counter
    value = world * B * a.steps / (ms / 1e3)
    acc_value = acc.clone()
    dump = None
    if a.dump_outputs and rank == 0:
        dump = outputs_to_dump(last["rec"] if a.no_graph else vout[(turn[0] - 1) % VL])

    # e2e: same calls, inputs are pinned host buffers (the library stages them), result record read back.
    # The batch is fed in chunks that alternate between lanes (own stream + own workspace), so the PCIe transfer of one
    # chunk overlaps the kernels of the previous one (tiseg_b200.parallel.HostFeed).
    chunk = a.chunk or max(1, B // 8)
    feed = parallel.HostFeed(local, lanes=a.lanes, chunk=chunk)
    lane_acc = torch.zeros(a.lanes, R, dtype=torch.float64, device=dev)

    def chunk_fn(src, ln):
        lane_acc[ln].add_(wl.flat(wl.gpu_step(ops, src)).sum(0))

    def e2e_step(src):
        feed.run(src, chunk_fn)
        acc.add_(lane_acc.sum(0))
        lane_acc.zero_()
        return acc

    step_resident = step
    step = e2e_step                                        # noqa: F811
    for _ in range(2):
        step(pinned_np)
    torch.cuda.synchronize()
    acc.zero_()
    ms_e2e, _ = timed(pinned_np, a.steps, with_d2h=True)
    e2e = world * B * a.steps / (ms_e2e / 1e3)
    # the same feed with the network outputs already on the device (where the reference's CNN leaves them) and only the
    # ground truth coming from the host: reported beside e2e, not instead of it
    mixed = {k: (devt[k] if k in wl.net_keys else pinned_np[k]) for k in wl.keys}
    step(mixed)
    torch.cuda.synchronize()
    acc.zero_()
    ms_gt, _ = timed(mixed, a.steps, with_d2h=True)
    e2e_gt = world * B * a.steps / (ms_gt / 1e3)
    h2d_gt = int(sum(pinned_np[k].nbytes for k in wl.keys if k not in wl.net_keys))
    # ... and with the instance ground truth stored as uint16 (ids < 65536), the largest evaluation input at half the bytes
    e2e_u16 = None
    if not wl.multi and int(host["gt_inst"].max()) < 65536:
        g16 = torch.from_numpy(host["gt_inst"].astype(np.uint16)).pin_memory().numpy()
        both = dict(pinned_np, gt_inst=g16)
        mixed16 = dict(mixed, gt_inst=g16)
        res16 = {}
        for tag, src in (("all_inputs_from_host", both), ("logits_resident_gt_from_host", mixed16)):
            step(src)
            torch.cuda.synchronize()
            acc.zero_()
            ms16, _ = timed(src, a.steps, with_d2h=True)
            res16[tag] = {"value": world * B * a.steps / (ms16 / 1e3), "unit": "tiles/s", "ms_per_step": ms16 / a.steps,
                          "h2d_bytes_per_step": int(sum(v.nbytes for k, v in src.items() if not hasattr(v, "is_cuda")))}
        e2e_u16 = res16
    step = step_resident
    if sampler and len(open(sampler.f.name).read().splitlines()) < 5:
        # a very short run: keep the same step going until a few samples exist
        t_end = time.perf_counter() + 0.4
        if not a.no_graph:
            fork_value_lanes()
        while time.perf_counter() < t_end:
            step(devt)
        if not a.no_graph:
            join_value_lanes()
        torch.cuda.synchronize()
    clocks = sampler.stop() if sampler else None
    h2d = int(sum(v.nbytes for v in pinned_np.values()))
    d2h = int(acc.numel() * 8)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # roofline leg: per-kernel CUDA-event durations over two more steps on the launching stream
    ctx.timing(True)
    for _ in range(2):
        with _lib.device_outputs():
            (plain_step if not a.no_graph else step)(devt)
    rep = ctx.timing_report()
    ctx.timing(False)
    total_ms = sum(v[1] for v in rep.values())
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    px = wl.H * wl.W * B
    # measured DRAM traffic per kernel for one whole step of this workload (ncu metrics pass, committed under profiles/)
    traffic = {}
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "r2_step_traffic_%s.json" % wl.name)))
        if traffic.get("batch") != B:
            traffic = {}
    except Exception:
        pass
    tk = traffic.get("kernels", {})

    def measured_bytes(name):
        short = name.strip("(").split("<")[0].split("(")[0]
        hits = [v.get("dram_bytes") for k, v in tk.items() if k == short or k.startswith(short + "_") or short.startswith(k + "_")]
        return sum(hits) if hits else None

    per_kernel = {}
    for k, (cnt, kms) in sorted(rep.items(), key=lambda kv: -kv[1][1]):
        bpp = kernel_bytes_per_px(wl, k)                    # KeyError on an unknown kernel: nothing gets a default
        ms_step = kms / 2
        ent = {"ms_per_step": round(ms_step, 4), "launches_per_step": cnt / 2}
        if bpp is not None:
            alg = bpp * px * cnt / 2
            meas = measured_bytes(k)
            used = min(alg, meas) if meas else alg
            ent.update(alg_bytes=alg, dram_bytes=meas, frac=round(used / (ms_step / 1e3) / 1e9 / peak, 4))
        per_kernel[k] = ent
    top_name = max(rep.items(), key=lambda kv: kv[1][1])[0]
    # the dominant kernel for the roofline record: the slowest one that works on pixels
    dom = next(k for k in per_kernel if "frac" in per_kernel[k])
    d = per_kernel[dom]
    achieved = min(d["alg_bytes"], d["dram_bytes"] or d["alg_bytes"]) / (d["ms_per_step"] / 1e3) / 1e9
    step_dram = traffic.get("step_dram_bytes")
    roof = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": d["dram_bytes"], "peak_source": "measured" if peaks else "fallback",
            "bytes_used": "min(algorithmic, measured DRAM) per launch", "alg_bytes_per_launch": d["alg_bytes"],
            "kernel_share_of_step": d["ms_per_step"] * 2 / total_ms, "slowest_kernel": top_name,
            "pipeline_frac": (wl.pipe_bpp * wl.H * wl.W * value / world) / 1e9 / peak,
            "step_dram_bytes": step_dram, "traffic_ratio": (step_dram / (wl.pipe_bpp * px)) if step_dram else None,
            "kernel_sum_ms_per_step": round(total_ms / 2, 4), "per_kernel": per_kernel}
    if UNKNOWN:
        roof["unknown_kernels"] = sorted(set(UNKNOWN))

    # cpu_baseline leg + verification: the same tiles through the oracle (literal cost profile) and through the GPU path
    cpu, check, rc = None, None, 0
    if world == 1 and not a.no_cpu_baseline:
        idx = [900000 + j for j in range(a.cpu_tiles)]
        ts, recs = zip(*[_cpu_tile((wl.name, i)) for i in idx])
        cpu = {"value": len(ts) / sum(ts), "unit": "tiles/s", "cores": 1, "kind": "port",
               "sample": "%d tiles of the same workload, one core, literal oracle port of the reference path (AJI / PQ restate "
                         "inst_metrics.py:25-67, 150-229 line for line)" % len(ts)}
        vt = [wl.prep(wl.make_tile(i)) for i in idx]
        vb = {k: torch.from_numpy(np.stack([t[k] for t in vt])).to(dev) for k in wl.keys}
        with _lib.device_outputs():
            got = wl.flat(wl.gpu_step(ops, vb)).cpu().numpy()
        want = np.stack(recs)
        ok = got.shape == want.shape and np.array_equal(got, want)
        check = {"tiles": len(idx), "records_equal_oracle": bool(ok), "record_width": R}
        if not ok:
            bad = np.argwhere(got != want)[:8].tolist() if got.shape == want.shape else "shape %r vs %r" % (got.shape, want.shape)
            check["mismatch_at"] = bad
            rc = 3
    inter, union = float(acc_value[0]), float(acc_value[1])
    line = {
        "metric": wl.metric, "value": value, "unit": "tiles/s", "n_gpus": world, "steps": a.steps,
        "warmup": max(a.warmup, 3), "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/int32 labels, fp32 softmax, fp64 IoU", "data": "synthetic",
        "config": {"workload": wl.name, "tile": [wl.H, wl.W], "tiles_per_step_per_gpu": B, "instances_per_tile": wl.instances,
                   "distinct_tiles": a.distinct, "l2": "inputs per step (%.0f MB) exceed the 126 MB L2" % (h2d / 1e6),
                   "parallelism": "tiles sharded per GPU, one all-reduce of metric accumulators",
                   "launch": "plain stream launches" if a.no_graph else
                   "CUDA graph replay of the step, steps alternating over %d streams (value); plain launches on %d lanes (e2e)" % (a.value_lanes, a.lanes)},
        "e2e": {"value": e2e, "unit": "tiles/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / a.steps,
                "logits_resident_gt_from_host": {"value": e2e_gt, "unit": "tiles/s", "h2d_bytes_per_step": h2d_gt,
                                                 "ms_per_step": ms_gt / a.steps},
                "gt_inst_as_uint16": e2e_u16},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
        "check": dict(check or {}, aji_of_timed_batch=(inter / union) if union else None),
    }
    if dump is not None:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, arr in dump.items():
            np.save(os.path.join(a.dump_outputs, name + ".npy"), arr)
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return rc


_JSON_FD = None


def guard_stdout():
    """stdout carries exactly ONE JSON line: anything a library prints there (the NCCL version banner does) is sent to
    stderr instead, and the line is written to the real stdout at the end."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _JSON_FD is None:
        os.write(1, data)
    else:
        os.write(_JSON_FD, data)


def main():
    guard_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="dist_monuseg_1000", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="tiles per step per GPU (0 = the workload's default)")
    ap.add_argument("--distinct", type=int, default=8, help="distinct synthetic tiles generated per rank")
    ap.add_argument("--chunk", type=int, default=0, help="e2e: tiles per host-fed chunk (0 = batch / 8)")
    ap.add_argument("--lanes", type=int, default=4, help="e2e: lanes (stream + workspace) the chunks alternate between")
    ap.add_argument("--cpu-tiles", type=int, default=2, help="tiles timed for the cpu_baseline leg (and verified against it)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time plain launches instead of a CUDA-graph replay of the step")
    ap.add_argument("--value-lanes", type=int, default=3, help="resident-input steps alternate between this many streams")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (rank 0) as DIR/<name>.npy: "
                    "the per-tile records, and the sem / inst maps of a seeded sample of the batch's tiles")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    rc = run_reference(a) if a.impl == "reference" else run_b200(a)
    sys.exit(rc or 0)


if __name__ == "__main__":
    main()
