"""What bf16 network outputs buy on each bench workload: the same step fed fp32 or bf16 network outputs, resident in HBM
or fed from pinned host buffers through parallel.HostFeed.

    python scripts/half_inputs.py --out DIR [--workloads a,b] [--reps 3] [--window 1.0]

Per workload (bench.WORKLOADS, at its bench batch) the network outputs (`net_keys`) are rounded to bf16 after `prep`, and
the fp32 arms are fed their upcast, so every arm computes the same records; the script checks that and exits 1 if not.
Arms:
  fp32_resident        fp32 inputs in HBM
  bf16_resident        bf16 inputs in HBM, read natively
  bf16_upcast_in_step  bf16 inputs in HBM, the caller doing `.float()` inside the step (what a bf16 caller paid before)
  fp32_host            pinned host fp32 inputs through HostFeed (lanes and chunk as bench.py's e2e leg)
  bf16_host            pinned host bf16 network outputs through HostFeed
Every step is a plain stream launch sequence (no CUDA graph, unlike bench.py's value).  Each timed window lasts at least
`--window` seconds; the arms alternate within each of `--reps` rounds.  Writes DIR/half_inputs.json: ms per step and tiles/s
per round, the input bytes per tile of each arm, the per-kernel CUDA-event times (tiseg_timing) of one resident step of each
arm, and the GPU's name, power limit and maximum SM clock."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ARMS = ("fp32_resident", "bf16_resident", "bf16_upcast_in_step", "fp32_host", "bf16_host")


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in q.split(",")]
        info.update(smi_name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:                                # the numbers are still reported, without the limit
        info["nvidia_smi"] = "unavailable: %s" % e
    return info


def run_workload(wl, a):
    import torch
    import bench
    from tiseg_b200 import _lib, ops, parallel
    dev = torch.device("cuda", 0)
    B = wl.batch
    host = bench.stack_batch(bench.make_tiles(a.distinct, 0, wl), B, wl.dihedral)
    bf = {k: torch.from_numpy(host[k]).to(torch.bfloat16) for k in wl.net_keys}
    up = {k: v.float() for k, v in bf.items()}                     # the values every arm computes on
    pin32 = {k: (up[k] if k in wl.net_keys else torch.from_numpy(host[k])).pin_memory() for k in wl.keys}
    src = {
        "fp32_resident": {k: v.to(dev) for k, v in pin32.items()},
        "bf16_host": {k: (bf[k].pin_memory() if k in wl.net_keys else pin32[k].numpy()) for k in wl.keys},
        "fp32_host": {k: v.numpy() for k, v in pin32.items()},
    }
    src["bf16_resident"] = {k: (bf[k].to(dev) if k in wl.net_keys else src["fp32_resident"][k]) for k in wl.keys}
    src["bf16_upcast_in_step"] = src["bf16_resident"]
    in_bytes = {arm: sum(v.numel() * v.element_size() if _lib.is_torch(v) else v.nbytes for v in s.values()) / B
                for arm, s in src.items()}
    feed = parallel.HostFeed(0, lanes=4, chunk=max(1, B // 8))
    R = wl.record_width()
    acc = torch.zeros(R, dtype=torch.float64, device=dev)
    lane_acc = torch.zeros(4, R, dtype=torch.float64, device=dev)

    def records(arm):
        """the flat per-tile records of one pass of the arm, [B, R]"""
        with _lib.device_outputs():
            if arm.endswith("_host"):
                parts = []
                feed.run(src[arm], lambda part, ln: parts.append(wl.flat(wl.gpu_step(ops, part))))
                return torch.cat(parts)
            s = src[arm]
            if arm == "bf16_upcast_in_step":
                s = {k: (v.float() if k in wl.net_keys else v) for k, v in s.items()}
            return wl.flat(wl.gpu_step(ops, s))

    def step(arm):
        with _lib.device_outputs():
            if arm.endswith("_host"):
                feed.run(src[arm], lambda part, ln: lane_acc[ln].add_(wl.flat(wl.gpu_step(ops, part)).sum(0)))
                acc.add_(lane_acc.sum(0))
                lane_acc.zero_()
                acc.cpu()                                          # the record comes back, as in bench.py's e2e leg
            else:
                s = src[arm]
                if arm == "bf16_upcast_in_step":
                    s = {k: (v.float() if k in wl.net_keys else v) for k, v in s.items()}
                acc.add_(wl.flat(wl.gpu_step(ops, s)).sum(0))

    want = records("fp32_resident").cpu().numpy()
    equal = {arm: bool(np.array_equal(records(arm).cpu().numpy(), want)) for arm in ARMS}

    def window(arm, n):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            step(arm)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    steps = {}
    for arm in ARMS:                                               # warm-up, then as many steps as fill the window
        window(arm, 2)
        t = window(arm, 2) / 2
        steps[arm] = max(3, int(np.ceil(a.window * 1e3 / t)))
    runs = {arm: [] for arm in ARMS}
    for r in range(a.reps):
        for arm in (ARMS if r % 2 == 0 else ARMS[::-1]):
            ms = window(arm, steps[arm])
            runs[arm].append({"steps": steps[arm], "window_s": round(ms / 1e3, 3), "ms_per_step": round(ms / steps[arm], 4),
                              "tiles_per_s": round(B * steps[arm] / (ms / 1e3), 1)})
    ctx = _lib.get_ctx(0)
    kernels = {}
    for arm in ARMS[:3]:
        ctx.timing(True)
        step(arm)
        torch.cuda.synchronize()
        kernels[arm] = {k: round(ms, 4) for k, (n, ms) in sorted(ctx.timing_report().items(), key=lambda kv: -kv[1][1])}
        ctx.timing(False)
    med = {arm: float(np.median([x["ms_per_step"] for x in runs[arm]])) for arm in ARMS}
    return {"batch": B, "tile": [wl.H, wl.W], "net_keys": list(wl.net_keys), "records_equal": equal,
            "input_bytes_per_tile": {k: int(v) for k, v in in_bytes.items()}, "runs": runs,
            "median_ms_per_step": {k: round(v, 4) for k, v in med.items()},
            "speedup_vs_fp32": {"resident": round(med["fp32_resident"] / med["bf16_resident"], 3),
                                "resident_vs_upcast_in_step": round(med["bf16_upcast_in_step"] / med["bf16_resident"], 3),
                                "host_fed": round(med["fp32_host"] / med["bf16_host"], 3)},
            "kernel_ms_per_step": kernels}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workloads", default="", help="comma-separated subset of bench.WORKLOADS (default: all five)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--window", type=float, default=1.0, help="seconds per timed window")
    ap.add_argument("--distinct", type=int, default=8)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("half_inputs.py measures on the GPU: no CUDA device")
    import bench
    names = [n for n in a.workloads.split(",") if n] or list(bench.WORKLOADS)
    out = {"gpu": gpu_info(), "arms": list(ARMS), "reps": a.reps, "window_s": a.window,
           "timing": "CUDA events around >= window_s of plain stream launches per arm; arms alternate within each round",
           "workloads": {}}
    ok = True
    for n in names:
        t0 = time.perf_counter()
        res = run_workload(bench.WORKLOADS[n](), a)
        res["wall_s"] = round(time.perf_counter() - t0, 1)
        out["workloads"][n] = res
        ok &= all(res["records_equal"].values())
        print(n, res["median_ms_per_step"], res["records_equal"], file=sys.stderr, flush=True)
        torch.cuda.empty_cache()
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "half_inputs.json"), "w") as f:         # rewritten after every workload
            json.dump(out, f, indent=1)
    if not ok:
        sys.exit("records differ between arms")


if __name__ == "__main__":
    main()
