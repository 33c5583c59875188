"""Per-kernel CUDA-event times of the DIST step on the bench batch (plain launches), plus the wall time of the step.
    python scripts/step_times.py [batch]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import bench
import tiseg_b200
from tiseg_b200 import _lib, ops
B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
tiles = bench.make_tiles(8, 0)
host = bench.stack_batch(tiles, B)
d = {k: torch.from_numpy(v).cuda() for k, v in host.items()}
ctx = _lib.get_ctx(0)
def step():
    cls = ops.softmax_argmax(d["sem_logit"])
    inst = ops.postproc_dist(d["dist_logit"])
    aji, pq = ops.pair_metrics_bin(inst, d["gt_inst"])
    counts, valid = ops.sem_counts(cls, d["gt_sem"], 2)
    return aji, pq, counts
with _lib.device_outputs():
    for _ in range(3):
        r = step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ctx.launch_count()
    e0.record()
    for _ in range(10):
        r = step()
    e1.record(); torch.cuda.synchronize()
    nl = (ctx.launch_count() - l0) / 10
    wall = e0.elapsed_time(e1) / 10
    ctx.timing(True)
    for _ in range(2):
        step()
    rep = ctx.timing_report()
    ctx.timing(False)
tot = sum(v[1] for v in rep.values()) / 2
print("step wall %.3f ms (%.0f tiles/s), %d launches, kernel sum %.3f ms | check aji %.6f pq %s" % (
    wall, B / wall * 1e3, nl, tot, float(r[0][:, 0].sum() / r[0][:, 1].sum()), r[1].sum(0).tolist()))
for k, v in sorted(rep.items(), key=lambda kv: -kv[1][1]):
    if v[1] / 2 >= 0.004:
        print("  %-44s x%-3d %.4f ms" % (k[:44], v[0] // 2, v[1] / 2))
