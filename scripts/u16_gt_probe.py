#!/usr/bin/env python
"""What uint16 instance ground truth buys on one GPU.

    python scripts/u16_gt_probe.py [--steps 10] [--rounds 5] [--out FILE]

Evaluation: a CoNIC-shaped batch (512 synthetic 256x256 tiles, C = 7; the bench's conic_sweep_256 inputs) goes through
``CoNICDataset.pre_eval_records`` with the predictions resident on the device and the ground truth
  1. resident int32, 2. resident uint16, 3. from pinned host memory as int32, 4. from pinned host memory as uint16.
Label making: one batch of 16 synthetic 1000x1000 instance maps through ``fix_inst`` -> ``instance_distance_map`` with the
instance map from pinned host memory as int32 and as uint16 (intermediates stay on the device).

For each feed: ms per step (CUDA events around `--steps` steps after a warm-up; the feeds alternate over `--rounds`
rounds, the median round is reported with the spread), host-to-device bytes per step (counted from the host arrays the
library stages), the per-kernel CUDA-event times of the kernels that read an instance map in one step, and the card's name
and power limit.  In the evaluation the prediction is an instance map too: an int32 kernel name counts the launches on both
maps, a ``<uint16_t>`` name only the ground truth's.  The records / label maps of every feed must be bit-identical, or the
script exits with status 1.  L2 is not flushed between steps.  Prints one JSON document.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402

# kernels that read an instance map (the int32 instantiation keeps the plain name, the uint16 one says so)
ID_KERNELS = ("k_eqbits", "k_max_id", "k_inst_class_hist", "k_comp_class_bits", "k_fix_keep", "(k_ccl_local", "(k_ccl_border",
           "k_fix_root_slots", "k_fix_list", "k_fix_newid")


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = [v.strip() for v in q.split(",")[:2]]
    except Exception as e:                                    # the numbers still stand, the card is then named only
        out["power_limit"] = "unavailable (%s)" % type(e).__name__
    return out


def pinned(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()


def time_feeds(feeds, step, steps, rounds):
    """feeds: name -> source; step(src) -> result.  -> name -> {ms_per_step, rounds_ms_per_step}, last results"""
    import torch
    last, per = {}, {k: [] for k in feeds}
    for k, src in feeds.items():                              # warm-up of every shape and workspace
        for _ in range(2):
            last[k] = step(src)
    torch.cuda.synchronize()
    for _ in range(rounds):
        for k, src in feeds.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                last[k] = step(src)
            e1.record()
            torch.cuda.synchronize()
            per[k].append(e0.elapsed_time(e1) / steps)
    return {k: {"ms_per_step": float(np.median(v)), "rounds_ms_per_step": [round(x, 4) for x in v]} for k, v in per.items()}, last


def kernel_times(step, src):
    from tiseg_b200 import _lib
    import torch
    ctx = _lib.get_ctx(0)
    torch.cuda.synchronize()
    ctx.timing(True)
    step(src)
    ctx.synchronize()
    rep = ctx.timing_report()
    ctx.timing(False)
    return {k: {"launches": n, "ms": round(ms, 4)} for k, (n, ms) in sorted(rep.items()) if k.startswith(ID_KERNELS)}


def same_bits(a, b):
    import torch
    a, b = torch.as_tensor(a).cpu(), torch.as_tensor(b).cpu()
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    if a.dtype.is_floating_point:
        a, b = a.view(torch.int64 if a.element_size() == 8 else torch.int32), b.view(torch.int64 if b.element_size() == 8 else torch.int32)
    return bool(torch.equal(a, b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--label-batch", type=int, default=16)
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "u16_gt_probe measures on a CUDA device"
    from tiseg_b200 import _lib, datasets, ops

    # ---- evaluation: CoNIC-shaped batch, predictions resident
    wl = bench.ConicSweep()
    b = bench.stack_batch(bench.make_tiles(64, 0, wl), a.batch)
    assert int(b["gt_inst"].max()) < 65536
    dev = torch.device("cuda:0")
    sem_pred, inst_pred = ops.postproc_unet(ops.softmax_argmax(torch.from_numpy(b["sem_logit"]).to(dev)), wl.max_class, wl.radius, None)
    gi32, gi16, gs = b["gt_inst"].astype(np.int32), b["gt_inst"].astype(np.uint16), b["gt_sem"].astype(np.uint8)
    feeds = {
        "resident_int32": (torch.from_numpy(gi32).to(dev), torch.from_numpy(gs).to(dev)),
        "resident_uint16": (torch.from_numpy(gi16).to(dev), torch.from_numpy(gs).to(dev)),
        "pinned_host_int32": (pinned(gi32), pinned(gs)),
        "pinned_host_uint16": (pinned(gi16), pinned(gs)),
    }
    sets = {k: datasets.CoNICDataset(sem_gts=s, inst_gts=i) for k, (i, s) in feeds.items()}
    idx = list(range(a.batch))
    ev_step = lambda ds: ds.pre_eval_records(sem_pred, inst_pred, idx)
    ev_times, recs = time_feeds(sets, ev_step, a.steps, a.rounds)
    ev = {}
    for k, (i, s) in feeds.items():
        host = not _lib.is_torch(i)
        # the semantic ground truth is staged twice: by the semantic counts and by the pair metrics
        ev[k] = dict(ev_times[k], h2d_bytes_per_step=int(i.nbytes + 2 * s.nbytes) if host else 0,
                     gt_inst_bytes=int(i.nbytes if host else i.numel() * i.element_size()),
                     instance_map_kernels=kernel_times(ev_step, sets[k]))
    ev_equal = all(same_bits(recs[k], recs["resident_int32"]) for k in recs)

    # ---- label making: fix_inst -> instance_distance_map from pinned host memory
    dl = bench.DistMonuseg()
    lb = bench.stack_batch([{"gt_inst": dl.make_tile(j)["gt_inst"]} for j in range(4)], a.label_batch)["gt_inst"]
    assert int(lb.max()) < 65536
    lfeeds = {"pinned_host_int32": pinned(lb.astype(np.int32)), "pinned_host_uint16": pinned(lb.astype(np.uint16))}

    def lab_step(src):
        with _lib.device_outputs():
            fixed = ops.fix_inst(src)
            return fixed, ops.instance_distance_map(fixed, True)
    lab_times, louts = time_feeds(lfeeds, lab_step, a.steps, a.rounds)
    lab = {k: dict(lab_times[k], h2d_bytes_per_step=int(v.nbytes), instance_map_kernels=kernel_times(lab_step, v)) for k, v in lfeeds.items()}
    lab_equal = all(same_bits(louts[k][j], louts["pinned_host_int32"][j]) for k in louts for j in range(2))

    doc = {
        "card": card(),
        "evaluation": {"what": "CoNICDataset.pre_eval_records, %d tiles of 256x256, C = 7, predictions resident" % a.batch,
                       "feeds": ev, "records_equal": ev_equal},
        "label_making": {"what": "fix_inst -> instance_distance_map, %d tiles of 1000x1000, outputs on the device" % a.label_batch,
                         "feeds": lab, "outputs_equal": lab_equal},
        "method": "CUDA events, %d steps per round after 2 warm-up steps per feed, %d rounds alternating the feeds, median "
                  "round; L2 not flushed" % (a.steps, a.rounds),
    }
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    return 0 if ev_equal and lab_equal else 1


if __name__ == "__main__":
    sys.exit(main())
