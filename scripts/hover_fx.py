"""What the HoVer-Net post-process costs at each fx of hover_post_proc (Sobel ksize int(20 * fx + 1), marker obj_size
ceil(10 * fx^2)), and the two ways to run it on 20x data.

    python scripts/hover_fx.py --out DIR [--batch 16] [--reps 3] [--window 1.0]

Arms, each one ops.postproc_hover call on `--batch` synthetic tiles resident in HBM (plain stream launches, no CUDA
graph):
  fx0.5_1000 / fx1.0_1000 / fx1.5_1000   1000 x 1000 tiles at fx 0.5, 1.0 (the benchmark's path) and 1.5
  20x_fx0.5_500                          500 x 500 tiles at fx 0.5, scale_factor 1: 20x data at its native size
  20x_fx1_sf2_500                        the same tiles with scale_factor 2 and fx 1: upsampled, the chain on 4x the pixels
Each timed window lasts at least `--window` seconds; the arms alternate within each of `--reps` rounds.  Before timing, every
arm's instances are checked against the CPU oracle on its first tile (the script exits 1 on a mismatch).  Writes
DIR/hover_fx.json: ms per step and tiles/s per round, the per-kernel CUDA-event times (tiseg_timing) of one step of each arm,
and the GPU's name, power limit and maximum SM clock."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(ROOT))
sys.path.insert(0, ROOT)

# name -> (tile side, fx, scale_factor)
ARMS = {"fx0.5_1000": (1000, 0.5, 1), "fx1.0_1000": (1000, 1.0, 1), "fx1.5_1000": (1000, 1.5, 1),
        "20x_fx0.5_500": (500, 0.5, 1), "20x_fx1_sf2_500": (500, 1.0, 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--window", type=float, default=1.0, help="seconds per timed window")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("hover_fx.py measures on the GPU: no CUDA device")
    from half_inputs import gpu_info
    import tiseg_b200  # noqa: F401
    from tiseg_b200 import _lib, ops, synth
    from oracle import postprocess as opp

    inputs = {}
    for side in sorted({s for s, _, _ in ARMS.values()}):
        ts = [synth.tile_hover(3, i, H=side, W=side) for i in range(a.batch)]
        inputs[side] = (torch.from_numpy(np.stack([t["fore_map"] for t in ts])).cuda(),
                        torch.from_numpy(np.stack([t["hv_map"] for t in ts])).cuda(), ts[0])

    def step(arm):
        side, fx, sf = ARMS[arm]
        fore, hv, _ = inputs[side]
        return ops.postproc_hover(fore, hv, scale_factor=sf, fx=fx)

    equal = {}
    for arm, (side, fx, sf) in ARMS.items():
        t0 = inputs[side][2]
        want, _ = opp.hover_post_proc(t0["fore_map"], t0["hv_map"], fx=fx, scale_factor=sf)
        equal[arm] = bool(np.array_equal(step(arm)[0].cpu().numpy(), want))

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
        steps[arm] = max(3, int(np.ceil(a.window * 1e3 / (window(arm, 2) / 2))))
    names = list(ARMS)
    runs = {arm: [] for arm in names}
    for r in range(a.reps):
        for arm in (names if r % 2 == 0 else names[::-1]):
            ms = window(arm, steps[arm])
            runs[arm].append({"steps": steps[arm], "window_s": round(ms / 1e3, 3), "ms_per_step": round(ms / steps[arm], 4),
                              "tiles_per_s": round(a.batch * steps[arm] / (ms / 1e3), 1)})
    ctx = _lib.get_ctx(0)
    kernels = {}
    for arm in names:
        ctx.timing(True)
        step(arm)
        torch.cuda.synchronize()
        kernels[arm] = {k: round(ms, 4) for k, (n, ms) in sorted(ctx.timing_report().items(), key=lambda kv: -kv[1][1])}
        ctx.timing(False)
    med = {arm: float(np.median([x["ms_per_step"] for x in runs[arm]])) for arm in names}
    out = {"gpu": gpu_info(), "batch": a.batch, "reps": a.reps, "window_s": a.window,
           "arms": {k: {"tile": v[0], "fx": v[1], "scale_factor": v[2], "ksize": int(20 * v[1] + 1)} for k, v in ARMS.items()},
           "timing": "CUDA events around >= window_s of plain stream launches per arm; arms alternate within each round",
           "inst_equal_oracle_tile0": equal, "runs": runs,
           "median_ms_per_step": {k: round(v, 4) for k, v in med.items()},
           "median_tiles_per_s": {k: round(a.batch / (v / 1e3), 1) for k, v in med.items()},
           "kernel_ms_per_step": kernels}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "hover_fx.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"median_ms_per_step": out["median_ms_per_step"], "median_tiles_per_s": out["median_tiles_per_s"],
                      "equal": equal, "gpu": out["gpu"]}))
    if not all(equal.values()):
        sys.exit("instances differ from the oracle")


if __name__ == "__main__":
    main()
