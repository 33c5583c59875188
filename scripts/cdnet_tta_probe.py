#!/usr/bin/env python
"""What feeding the CDNet tails the raw TTA outputs buys on one GPU.

    python scripts/cdnet_tta_probe.py [--tiles 16] [--steps 5] [--rounds 5] [--out FILE]

Workload: CDNet on CoNSeP-sized tiles, 16 tiles of 1000 x 1000, T = 8 variants (rotate [0, 90] x the four flips, the
shipped test config), heads sem 3, dir 9, point 1 channels; whole inference and split inference (window 256, overlap 40:
the split_inference window of base.py), fp32 and bf16; plus one MultiTaskCDNet row (tc 3, sem 4, dir 9, point 1; whole,
fp32).  The head outputs are seeded random normals generated on the device (the kernels' work does not depend on the
values), resident on the device like a network's outputs.

Routes, on the same inputs:
  A       the reference's order in torch: per head and variant the window canvas (split inference), the reverse rotation /
          flip (torch.flip, torch.rot90), torch.stack, then ops.cdnet_refine / ops.mtcdnet_refine
  B       ops.cdnet_refine_tta / ops.mtcdnet_refine_tta on the raw variant lists (this includes the torch.cat that packs
          each head's variants into the library's layout)
  B_entry the C entry on heads already packed in that layout (a network writing its variants into one buffer): the
          fused kernels alone

Method: CUDA events around `--steps` calls after a warm-up of every route, the routes alternate over `--rounds` rounds,
the median round is reported with all rounds.  The inputs (6.6 GB for the fp32 whole-inference case) are far larger than
the 126 MB L2.  Per-kernel CUDA-event times of route B_entry from one extra call.  The outputs of A, B and B_entry must be
equal bit for bit, asserted in the same run.  The card's name and power limit are read in the same run.  Prints one JSON
document.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402

from u16_gt_probe import card, same_bits  # noqa: E402

ROTS, FLIPS = [0, 90], ["none", "horizontal", "vertical", "diagonal"]


def n_windows(H, W, window, overlap):
    st = window - overlap
    pad_h = st - (H - window) % st if H - window > 0 else window - H
    pad_w = st - (W - window) % st if W - window > 0 else window - W
    return H + pad_h, W + pad_w, ((H + pad_h - window) // st + 1) * ((W + pad_w - window) // st + 1)


def stitch(x, H, W, window, overlap):
    """base.py:255-295 in torch: windows [N, M, C, w, w] -> canvas -> centre crop [N, C, H, W]"""
    import torch
    st = window - overlap
    H1, W1, _ = n_windows(H, W, window, overlap)
    canvas = torch.zeros((x.shape[0], x.shape[2], H1, W1), dtype=x.dtype, device=x.device)
    k = 0
    for i in range(0, H1 - overlap, st):
        r_s = i + overlap // 2 if i > 0 else 0
        r_e = i + window - overlap // 2 if i + window < H1 else H1
        for j in range(0, W1 - overlap, st):
            c_s = j + overlap // 2 if j > 0 else 0
            c_e = j + window - overlap // 2 if j + window < W1 else W1
            canvas[:, :, r_s:r_e, c_s:c_e] = x[:, k, :, r_s - i:r_e - i, c_s - j:c_e - j]
            k += 1
    return canvas[:, :, (H1 - H) // 2:(H1 - H) // 2 + H, (W1 - W) // 2:(W1 - W) // 2 + W]


def reverse(x, rot, flip):
    """base.py:365-381 on [N, C, H, W]"""
    import torch
    if flip == "horizontal":
        x = torch.flip(x, [-1])
    elif flip == "vertical":
        x = torch.flip(x, [-2])
    elif flip == "diagonal":
        x = torch.flip(x, [-2, -1])
    return torch.rot90(x, 4 - (rot // 90) % 4, [-2, -1])


def route_a_stack(variants, H, W, window, overlap):
    import torch
    rots = [r for r in ROTS for _ in FLIPS]
    flips = [f for _ in ROTS for f in FLIPS]
    full = []
    for v, r, f in zip(variants, rots, flips):
        Ht, Wt = (W, H) if (r // 90) % 2 else (H, W)
        full.append(reverse(stitch(v, Ht, Wt, window, overlap) if window else v, r, f))
    return torch.stack(full, dim=1)


def make_heads(gen, N, H, W, chans, window, overlap, dtype):
    import torch
    heads = []
    for C in chans:
        vs = []
        for r in ROTS:
            Ht, Wt = (W, H) if (r // 90) % 2 else (H, W)
            shape = (N, C, Ht, Wt) if window == 0 else (N, n_windows(Ht, Wt, window, overlap)[2], C, window, window)
            for _ in FLIPS:
                vs.append((torch.randn(shape, generator=gen, device="cuda") * 3).to(dtype))
        heads.append(vs)
    return heads


def timed(routes, steps, rounds):
    import torch
    last, per = {}, {k: [] for k in routes}
    for k, fn in routes.items():
        for _ in range(2):
            last[k] = fn()
    torch.cuda.synchronize()
    for _ in range(rounds):
        for k, fn in routes.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                last[k] = fn()
            e1.record()
            torch.cuda.synchronize()
            per[k].append(e0.elapsed_time(e1) / steps)
    return {k: {"ms_per_call": round(float(np.median(v)), 4), "rounds_ms": [round(x, 4) for x in v]} for k, v in per.items()}, last


def kernel_times(fn):
    import torch
    from tiseg_b200 import _lib
    ctx = _lib.get_ctx(0)
    torch.cuda.synchronize()
    ctx.timing(True)
    fn()
    ctx.synchronize()
    rep = ctx.timing_report()
    ctx.timing(False)
    return {k: {"launches": n, "ms": round(ms, 4)} for k, (n, ms) in sorted(rep.items())}


def case(model, dt, window, overlap, a, gen):
    import ctypes
    import torch
    from tiseg_b200 import ops
    from tiseg_b200._lib import get_ctx, net_inputs, ptr
    dtype = {"fp32": torch.float32, "bf16": torch.bfloat16}[dt]
    N, H, W = a.tiles, a.size, a.size
    rots = [r for r in ROTS for _ in FLIPS]
    flips = [f for _ in ROTS for f in FLIPS]
    T = len(rots)
    chans = (3, 9, 1) if model == "cdnet" else (3, 4, 9, 1)
    heads = make_heads(gen, N, H, W, chans, window, overlap, dtype)
    in_bytes = sum(v.numel() * v.element_size() for h in heads for v in h)
    packed = [torch.cat([v.reshape(N, -1) for v in h], dim=1) for h in heads]
    crot = (ctypes.c_int * T)(*rots)
    cflip = (ctypes.c_int * T)(*[ops._FLIPS[f] for f in flips])
    _, dcode = net_inputs(packed[0])
    ctx = get_ctx(0)

    def out(shape, dt_):
        return torch.empty(shape, dtype=dt_, device="cuda")

    if model == "cdnet":
        def route_a():
            return ops.cdnet_refine(*[route_a_stack(h, H, W, window, overlap) for h in heads], if_ddm=True)

        def route_b():
            return ops.cdnet_refine_tta(*heads, rots, flips, (H, W), window, overlap, if_ddm=True)

        def route_b_entry():
            r = dict(sem_prob=out((N, 3, H, W), torch.float32), cls=out((N, H, W), torch.uint8), dir_map=out((N, H, W), torch.uint8),
                     dd=out((N, H, W), torch.float32))
            ctx.call("tiseg_cdnet_refine_tta_typed", dcode, *[ptr(p) for p in packed], N, T, 3, 9, H, W, crot, cflip, window, overlap, 1,
                     ptr(r["sem_prob"]), ptr(r["cls"]), ptr(r["dir_map"]), ptr(r["dd"]))
            return r
    else:
        def route_a():
            return ops.mtcdnet_refine(*[route_a_stack(h, H, W, window, overlap) for h in heads], if_ddm=True)

        def route_b():
            return ops.mtcdnet_refine_tta(*heads, rots, flips, (H, W), window, overlap, if_ddm=True)

        def route_b_entry():
            r = dict(tc_prob=out((N, 3, H, W), torch.float32), tc_cls=out((N, H, W), torch.uint8), sem_cls=out((N, H, W), torch.uint8),
                     dir_map=out((N, H, W), torch.uint8), dd=out((N, H, W), torch.float32))
            ctx.call("tiseg_mtcdnet_refine_tta_typed", dcode, *[ptr(p) for p in packed], N, T, 3, 4, 9, H, W, crot, cflip, window, overlap, 1,
                     ptr(r["tc_prob"]), ptr(r["tc_cls"]), None, ptr(r["sem_cls"]), ptr(r["dir_map"]), ptr(r["dd"]))
            return r

    times, last = timed({"A": route_a, "B": route_b, "B_entry": route_b_entry}, a.steps, a.rounds)
    for k in ("B", "B_entry"):
        for name in last["A"]:
            if not same_bits(last[k][name], last["A"][name]):
                sys.stderr.write("%s %s %s window %d: route %s output %s differs from route A\n" % (model, dt, N, window, k, name))
                sys.exit(1)
    res = dict(model=model, dtype=dt, tiles=N, H=H, W=W, T=T, window=window, overlap=overlap,
               head_channels=list(chans), head_input_bytes=int(in_bytes), outputs_equal_bitwise=True, routes=times,
               speedup_B_over_A=round(times["A"]["ms_per_call"] / times["B"]["ms_per_call"], 3),
               speedup_B_entry_over_A=round(times["A"]["ms_per_call"] / times["B_entry"]["ms_per_call"], 3),
               head_read_rate_B_entry_TBps=round(in_bytes / (times["B_entry"]["ms_per_call"] * 1e-3) / 1e12, 3),
               kernels_B_entry=kernel_times(route_b_entry))
    del heads, packed, last
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tiles", type=int, default=16)
    ap.add_argument("--size", type=int, default=1000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "cdnet_tta_probe measures on a CUDA device"
    import tiseg_b200  # noqa: F401
    gen = torch.Generator(device="cuda")
    gen.manual_seed(2024)
    rows = []
    for dt in ("fp32", "bf16"):
        for window, overlap in ((0, 0), (256, 40)):
            rows.append(case("cdnet", dt, window, overlap, a, gen))
    rows.append(case("mtcdnet", "fp32", 0, 0, a, gen))
    doc = dict(probe="cdnet_tta_probe", card=card(), steps=a.steps, rounds=a.rounds,
               l2_note="inputs far larger than the 126 MB L2; L2 not flushed between calls", rows=rows)
    text = json.dumps(doc, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
