"""fp16 / bf16 network outputs read natively.  A call fed half-precision logits, distance / foreground / HV maps or
direction and point heads must return, bit for bit and with the same dtypes, what the same call returns for their fp32
upcast ``x.float()``: the kernels convert at the load (exact) and run the fp32 arithmetic after it.  The first test
checks the Python dispatch on the CPU; the others compare the two calls on the GPU, from the operators up to the
reference-named segmentor tails and the host-fed chunk loop, and check that no fp32 copy of the input is made."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import tiseg_b200  # noqa: E402,F401
from tiseg_b200 import _lib, ops, synth  # noqa: E402

gpu = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
HALF = ("float16", "bfloat16")


def _tdt(name):
    import torch
    return getattr(torch, name)


def _np(a):
    return a.detach().cpu().numpy() if _lib.is_torch(a) else np.asarray(a)


def _same(got, want, what):
    """bit-identical, same dtype, same kind; floats compared as raw bits (NaN payloads and signed zeros included)"""
    if isinstance(want, dict):
        assert sorted(got) == sorted(want), what
        for k in want:
            _same(got[k], want[k], "%s[%s]" % (what, k))
        return
    if isinstance(want, (list, tuple)):
        assert len(got) == len(want), what
        for i, (g, w) in enumerate(zip(got, want)):
            _same(g, w, "%s[%d]" % (what, i))
        return
    if want is None:
        assert got is None, what
        return
    assert _lib.is_torch(got) == _lib.is_torch(want), "%s: %s vs %s" % (what, type(got), type(want))
    g, w = _np(got), _np(want)
    assert g.dtype == w.dtype and g.shape == w.shape, "%s: %s%r vs %s%r" % (what, g.dtype, g.shape, w.dtype, w.shape)
    if g.dtype.kind == "f":
        g, w = g.view("u%d" % g.itemsize), w.view("u%d" % w.itemsize)
    bad = np.argwhere(g != w)
    assert len(bad) == 0, "%s: %d of %d elements differ, first at %r: %r vs %r" % (
        what, len(bad), g.size, tuple(bad[0]), _np(got)[tuple(bad[0])], _np(want)[tuple(bad[0])])


def _rounded(a, dtype, device="cuda"):
    """numpy fp32 array -> (tensor of `dtype` on `device`, its fp32 upcast on the same device)"""
    import torch
    h = torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(device).to(_tdt(dtype))
    return h, h.float()


# --------------------------------------------------------------------------- dispatch (CPU)
def test_net_inputs_dispatch():
    import torch
    a = np.arange(24, dtype=np.float16).reshape(2, 3, 4)
    (x,), code = _lib.net_inputs(a)
    assert code == _lib.DTYPE_F16 == 1 and x.dtype == np.float16 and np.shares_memory(x, a)
    (x, y), code = _lib.net_inputs(a, a[:, ::-1])                  # a strided view is made contiguous, still fp16
    assert code == 1 and y.dtype == np.float16 and y.flags.c_contiguous and np.array_equal(y, a[:, ::-1])
    b = torch.arange(24, dtype=torch.bfloat16).reshape(2, 3, 4)
    (x,), code = _lib.net_inputs(b)
    assert code == _lib.DTYPE_BF16 == 2 and x.dtype == torch.bfloat16 and x.data_ptr() == b.data_ptr()
    (x,), code = _lib.net_inputs(torch.zeros(3, dtype=torch.float16))
    assert code == 1 and x.dtype == torch.float16
    (x,), code = _lib.net_inputs(a.astype(np.float64))
    assert code == _lib.DTYPE_F32 == 0 and x.dtype == np.float32
    (x, y), code = _lib.net_inputs(b, b.float())                   # mixed: today's conversion of everything to fp32
    assert code == 0 and x.dtype == torch.float32 and y.dtype == torch.float32 and torch.equal(x, b.float())
    (x, y), code = _lib.net_inputs(a, b)                           # fp16 with bf16 is mixed too
    assert code == 0 and x.dtype == np.float32 and y.dtype == torch.float32
    (x,), code = _lib.net_inputs([[1.0, 2.0]])
    assert code == 0 and x.dtype == np.float32


# --------------------------------------------------------------------------- softmax / argmax
SHAPES = [(1000, 1000), (33, 257), (1000, 999)]                   # the odd widths take the scalar path


@gpu
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("T,C", [(1, 2), (1, 3), (1, 7), (1, 16), (8, 2), (8, 3), (8, 7), (8, 16)])
def test_softmax_argmax_half_equals_upcast(dtype, T, C):
    """T = 1 without probabilities reaches k_argmax_logits2 (C = 2) and k_argmax_logits<4 / 8 / 16>; the rest
    k_softmax_argmax.  Sources: device tensors, a device view one element off alignment, and host buffers."""
    import torch
    td = _tdt(dtype)
    g = torch.Generator(device="cuda").manual_seed(1000 * T + C)
    for H, W in SHAPES:
        x = (torch.randn((2 if H < 1000 else 1, T, C, H, W), generator=g, device="cuda") * 3).to(td)
        ref = x.float()
        for want_prob in (False, True):
            want = ops.softmax_argmax(ref, want_prob=want_prob)
            _same(ops.softmax_argmax(x, want_prob=want_prob), want, "device %s %dx%d T=%d C=%d" % (dtype, H, W, T, C))
            _same(ops.softmax_argmax(x[0], want_prob=want_prob), ops.softmax_argmax(ref[0], want_prob=want_prob), "single")
            buf = torch.empty(x.numel() + 1, dtype=td, device="cuda")
            view = buf[1:].view(x.shape)
            view.copy_(x)
            assert view.data_ptr() % 8 != 0
            _same(ops.softmax_argmax(view, want_prob=want_prob), want, "misaligned view")
            host_want = tuple(_np(w) for w in want) if want_prob else _np(want)
            pinned = x.cpu().pin_memory()
            _same(ops.softmax_argmax(pinned, want_prob=want_prob), host_want, "pinned host %s" % dtype)
            if dtype == "float16":
                _same(ops.softmax_argmax(x.cpu().numpy(), want_prob=want_prob), host_want, "numpy float16")


def _adversarial_logits(dtype, N, T, C, H, W, seed):
    """logits of `dtype` built from exact ties, +-0, values 1-4 ulps (of the half type) apart around a few bases (near
    1e-6 in fp16, where it is subnormal, near 1e-7 in bf16, and at ordinary magnitudes), and +-inf / NaN in any channel"""
    import torch
    td = _tdt(dtype)
    rng = np.random.default_rng(seed)
    small = 1e-6 if dtype == "float16" else 1e-7
    bases = torch.tensor([small, -small, 0.0, -0.0, 3 * small, 1.0, -2.5, 40.0], dtype=td).view(torch.int16).numpy()
    gi = rng.integers(0, len(bases), (N, T, 1, H, W))
    k = rng.integers(0, 5, (N, T, C, H, W))
    k[rng.random(k.shape) < 0.3] = 0                              # more exact ties
    bits = (bases[gi].astype(np.int32) + k).astype(np.int16)
    x = torch.from_numpy(bits).view(td).clone()
    special = torch.tensor([float("inf"), float("-inf"), float("nan"), 0.0, -0.0], dtype=td)
    pick = torch.from_numpy(rng.integers(0, len(special), x.shape))
    where = torch.from_numpy(rng.random(x.shape) < 0.04)
    x[where] = special[pick[where]]
    return x.cuda()


@gpu
@pytest.mark.parametrize("dtype", HALF)
def test_softmax_argmax_adversarial_ties(dtype):
    """the tie band of the streaming argmax (DESIGN.md §5) runs on the converted values: the same decisions as fp32"""
    for T in (1, 2):
        for C in (2, 3, 5, 16):
            for H, W in ((64, 256), (31, 33)):
                x = _adversarial_logits(dtype, 2, T, C, H, W, 100 * T + C + W)
                for want_prob in (False, True):
                    _same(ops.softmax_argmax(x, want_prob=want_prob), ops.softmax_argmax(x.float(), want_prob=want_prob),
                          "adversarial %s T=%d C=%d %dx%d prob=%s" % (dtype, T, C, H, W, want_prob))


# --------------------------------------------------------------------------- TTA stitch + reverse + mean
def _tta_variants(rng, N, C, H, W, rots, window, overlap):
    out = []
    for r in rots:
        Ht, Wt = (W, H) if (r // 90) % 2 else (H, W)
        if window == 0:
            out.append(rng.standard_normal((N, C, Ht, Wt)).astype(np.float32) * 3)
        else:
            st = window - overlap
            pad_h = st - (Ht - window) % st if Ht - window > 0 else window - Ht
            pad_w = st - (Wt - window) % st if Wt - window > 0 else window - Wt
            M = ((Ht + pad_h - window) // st + 1) * ((Wt + pad_w - window) // st + 1)
            out.append(rng.standard_normal((N, M, C, window, window)).astype(np.float32) * 3)
    return out


@gpu
@pytest.mark.parametrize("dtype", HALF)
def test_tta_half_equals_upcast(dtype):
    """rotations 0 / 90 / 180 / 270 x the four flips, whole and split inference with the window geometry of the
    reference's DIST runs recorded in r2_ref.npz"""
    m = np.load(os.path.join(G, "r2_ref.npz"))
    rots = [r for r in (0, 90, 180, 270) for _ in range(4)]
    flips = ["none", "horizontal", "vertical", "diagonal"] * 4
    for j in range(3):
        H, W, window, overlap, _ = [int(v) for v in m["d%d_meta" % j]]
        for win, ov in ((window, overlap), (0, 0)):
            rng = np.random.default_rng(77 + j + win)
            for C in (2, 7):
                pairs = [_rounded(v, dtype) for v in _tta_variants(rng, 2, C, H, W, rots, win, ov)]
                half, ref = [p[0] for p in pairs], [p[1] for p in pairs]
                what = "%s %dx%d window %d/%d C=%d" % (dtype, H, W, win, ov, C)
                for T in (1, 16):
                    for want_prob in (False, True):
                        _same(ops.softmax_argmax_tta(half[:T], rots[:T], flips[:T], (H, W), win, ov, want_prob=want_prob),
                              ops.softmax_argmax_tta(ref[:T], rots[:T], flips[:T], (H, W), win, ov, want_prob=want_prob),
                              "softmax_argmax_tta " + what)
                    _same(ops.tta_mean(half[:T], rots[:T], flips[:T], (H, W), win, ov),
                          ops.tta_mean(ref[:T], rots[:T], flips[:T], (H, W), win, ov), "tta_mean " + what)
                if dtype == "float16" and C == 2:                 # host variants are packed in fp16 too
                    _same(ops.tta_mean([_np(h) for h in half], rots, flips, (H, W), win, ov),
                          _np(ops.tta_mean(ref, rots, flips, (H, W), win, ov)), "tta_mean numpy " + what)


# --------------------------------------------------------------------------- DIST
@gpu
@pytest.mark.parametrize("dtype", HALF)
def test_postproc_dist_half_equals_upcast(dtype):
    """instances, markers and raw flood, lambda 0 and 3: synthetic distance maps rounded to the dtype and the adversarial
    topologies of tests/topology.py as d = 1 + pattern"""
    from test_gpu_bitccl import PATTERNS, _pattern
    maps = [synth.tile_dist(2, i, H=1000, W=1000)["dist_logit"] for i in range(2)]
    maps.append(np.stack([synth.tile_dist(2, 10 + i, H=257, W=255)["dist_logit"] for i in range(3)]))
    for H, W in ((65, 257), (33, 1000), (256, 256)):
        maps.append(np.stack([1.0 + _pattern(p, H, W) for p in PATTERNS]).astype(np.float32))
    for d in maps:
        half, ref = _rounded(d, dtype)
        for lamb in (0, 3):
            _same(ops.postproc_dist(half, debug=True, lamb=lamb), ops.postproc_dist(ref, debug=True, lamb=lamb),
                  "postproc_dist %s %r lamb=%d" % (dtype, tuple(d.shape), lamb))
    half, ref = _rounded(maps[2], dtype)
    _same(ops.postproc_dist(half.cpu().pin_memory(), debug=True), tuple(_np(x) for x in ops.postproc_dist(ref, debug=True)),
          "postproc_dist pinned host")


# --------------------------------------------------------------------------- HoVer-Net
@gpu
@pytest.mark.parametrize("dtype", HALF)
def test_postproc_hover_half_equals_upcast(dtype):
    """blb mask, fp64 flooded image, markers and instances at scale 1 and 2 (the resize reads the half inputs)"""
    for H, W, n in ((256, 256, 2), (200, 333, 1), (1000, 1000, 1)):
        ts = [synth.tile_hover(3, 40 + i, H=H, W=W) for i in range(n)]
        fh, fr = _rounded(np.stack([t["fore_map"] for t in ts]), dtype)
        hh, hr = _rounded(np.stack([t["hv_map"] for t in ts]), dtype)
        for sf in ((1, 2) if H < 1000 else (1,)):
            _same(ops.postproc_hover(fh, hh, scale_factor=sf, debug=True), ops.postproc_hover(fr, hr, scale_factor=sf, debug=True),
                  "postproc_hover %s %dx%d scale %d" % (dtype, H, W, sf))
    if dtype == "float16":
        _same(ops.postproc_hover(_np(fh[0]), _np(hh[0]), debug=True), tuple(_np(x) for x in ops.postproc_hover(fr[0], hr[0], debug=True)),
              "postproc_hover numpy float16")


# --------------------------------------------------------------------------- CDNet / MultiTaskCDNet
def _cdnet_heads(seed, N, T, H, W, D=9):
    rng = np.random.default_rng(seed)
    tc, sem, dirs, pts = [], [], [], []
    for n in range(N):
        t = synth.gt_and_pred(seed + n, H, W, num_classes=3)
        tc.append(np.stack([synth.sem_logits(rng, synth.three_class_map(t["pred_inst"]), 3) for _ in range(T)]))
        sem.append(np.stack([synth.sem_logits(rng, t["pred_sem"], 3) for _ in range(T)]))
        d, p = zip(*[synth.direction_logits(rng, t["pred_inst"]) for _ in range(T)])
        dirs.append(np.stack(d) if D == 9 else rng.uniform(-1.0, 7.5, (T, 1, H, W)).astype(np.float32))
        pts.append(np.stack(p))
    return [np.stack(a) for a in (tc, sem, dirs, pts)]


@gpu
@pytest.mark.parametrize("dtype", HALF)
def test_cdnet_refine_half_equals_upcast(dtype):
    for T, (H, W) in [(1, (64, 80)), (2, (96, 70)), (2, (256, 256))]:
        tc, _, dirs, pts = _cdnet_heads(8300 + T + H, 3, T, H, W)
        (th, tr), (dh, dr), (ph, pr) = [_rounded(a, dtype) for a in (tc, dirs, pts)]
        for if_ddm in (True, False):
            _same(ops.cdnet_refine(th, dh, ph, if_ddm=if_ddm), ops.cdnet_refine(tr, dr, pr, if_ddm=if_ddm),
                  "cdnet_refine %s T=%d %dx%d ddm=%s" % (dtype, T, H, W, if_ddm))


@gpu
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("D", [9, 1])
def test_mtcdnet_refine_half_equals_upcast(dtype, D):
    for T, (H, W) in [(1, (64, 80)), (2, (96, 70)), (2, (256, 256))]:
        heads = _cdnet_heads(8400 + T + H + D, 3, T, H, W, D)
        half, ref = zip(*[_rounded(a, dtype) for a in heads])
        for if_ddm in (True, False):
            for want_sem_prob in (False, True):
                _same(ops.mtcdnet_refine(*half, if_ddm=if_ddm, want_sem_prob=want_sem_prob),
                      ops.mtcdnet_refine(*ref, if_ddm=if_ddm, want_sem_prob=want_sem_prob),
                      "mtcdnet_refine %s D=%d T=%d %dx%d ddm=%s" % (dtype, D, T, H, W, if_ddm))
    if dtype == "float16":
        _same(ops.mtcdnet_refine(*[_np(h) for h in half]), {k: _np(v) for k, v in ops.mtcdnet_refine(*ref).items()},
              "mtcdnet_refine numpy float16")


# --------------------------------------------------------------------------- the reference-named tails
@gpu
@pytest.mark.parametrize("dtype", HALF)
def test_segmentor_tails_half_equal_upcast(dtype):
    from tiseg_b200 import segmentors
    m = np.load(os.path.join(G, "r2_ref.npz"))
    H, W, window, overlap, _ = [int(v) for v in m["d0_meta"]]
    cfg = dict(rotate_degrees=[0, 90, 180, 270], flip_directions=["none", "horizontal", "vertical", "diagonal"])
    rots = [r for r in cfg["rotate_degrees"] for _ in cfg["flip_directions"]]
    rng = np.random.default_rng(5)
    sv = [_rounded(v, dtype) for v in _tta_variants(rng, 2, 2, H, W, rots, window, overlap)]
    dv = [_rounded(np.abs(v) * 3, dtype) for v in _tta_variants(rng, 2, 1, H, W, rots, window, overlap)]
    seg = segmentors.Dist(2, test_cfg=cfg)
    _same(seg.inference_tail([h for h, _ in sv], [h for h, _ in dv], (H, W), window, overlap),
          seg.inference_tail([r for _, r in sv], [r for _, r in dv], (H, W), window, overlap), "Dist.inference_tail")
    t = synth.tile_dist(2, 3, H=256, W=256)
    (sh, sr), (dh, dr) = _rounded(t["sem_logit"][None], dtype), _rounded(t["dist_logit"], dtype)
    _same(seg.forward_eval(sh, dh), seg.forward_eval(sr, dr), "Dist.forward_eval")

    t = synth.tile_hover(3, 4, H=256, W=256)
    (sh, sr), (hh, hr), (fh, fr) = [_rounded(a, dtype) for a in (t["sem_logit"][None], t["hv_map"], t["fore_map"])]
    for sf in (1, 2):
        hseg = segmentors.HoverNet(3, test_cfg=dict(scale_factor=sf))
        _same(hseg.forward_eval(sh, hh, fh), hseg.forward_eval(sr, hr, fr), "HoverNet.forward_eval scale %d" % sf)

    tc, sem, dirs, pts = _cdnet_heads(8500, 1, 2, 128, 160)
    half, ref = zip(*[_rounded(a[0], dtype) for a in (tc, sem, dirs, pts)])
    cd = segmentors.CDNet(2, test_cfg=dict(if_ddm=True))
    _same(cd.forward_eval(half[0], half[2], half[3]), cd.forward_eval(ref[0], ref[2], ref[3]), "CDNet.forward_eval")
    for if_ddm in (True, False):
        mt = segmentors.MultiTaskCDNet(3, if_ddm=if_ddm)
        _same(mt.forward_eval(*half), mt.forward_eval(*ref), "MultiTaskCDNet.forward_eval ddm=%s" % if_ddm)


# --------------------------------------------------------------------------- host-fed chunks
@gpu
def test_host_feed_pinned_bf16_equals_one_fp32_call():
    """40 tiles of bf16 network outputs in pinned host memory, fed in chunks of 8 over 2 lanes: the per-tile records
    and maps of one fp32 call on the upcast inputs"""
    import torch
    from tiseg_b200 import parallel
    ts = [synth.tile_dist(2, 60 + i, H=256, W=256) for i in range(40)]
    host = {"sem_logit": torch.from_numpy(np.stack([t["sem_logit"][None] for t in ts])).to(torch.bfloat16).pin_memory(),
            "dist_logit": torch.from_numpy(np.stack([t["dist_logit"] for t in ts])).to(torch.bfloat16).pin_memory(),
            "gt_inst": torch.from_numpy(np.stack([t["gt_inst"] for t in ts])).pin_memory(),
            "gt_sem": torch.from_numpy(np.stack([t["gt_sem"] for t in ts])).pin_memory()}

    def step(src):
        cls = ops.softmax_argmax(src["sem_logit"])
        inst = ops.postproc_dist(src["dist_logit"])
        aji, pq = ops.pair_metrics_bin(inst, src["gt_inst"])
        counts, _ = ops.sem_counts(cls, src["gt_sem"], 2)
        return dict(cls=cls, inst=inst, aji=aji, pq=pq, counts=counts)

    parts = []
    parallel.HostFeed(0, lanes=2, chunk=8).run(host, lambda part, ln: parts.append(step(part)))
    torch.cuda.synchronize()
    assert len(parts) == 5 and all(p["inst"].is_cuda for p in parts)
    got = {k: torch.cat([p[k] for p in parts]) for k in parts[0]}
    want = step({k: (v.cuda().float() if v.dtype == torch.bfloat16 else v.cuda()) for k, v in host.items()})
    _same(got, want, "HostFeed bf16 vs one fp32 call")


# --------------------------------------------------------------------------- no conversion, and the dtype code checked
@gpu
def test_half_inputs_make_no_fp32_copy():
    """the peak of torch's allocator grows by the outputs only, never by an fp32 copy of the input"""
    import torch
    x = torch.randn((64, 1, 2, 512, 512), device="cuda").to(torch.bfloat16)
    d = (torch.rand((64, 512, 512), device="cuda") * 12).to(torch.bfloat16)
    for fn, arg, out_bytes in ((ops.softmax_argmax, x, 64 * 512 * 512), (ops.postproc_dist, d, 64 * 512 * 512 * 4)):
        fn(arg)                                                   # library workspace and modules warmed up
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.max_memory_allocated()
        out = fn(arg)
        torch.cuda.synchronize()
        grew = torch.cuda.max_memory_allocated() - base
        assert grew - out_bytes < 4 * arg.numel(), "%s: the peak grew by %d bytes" % (fn.__name__, grew)
        del out


@gpu
def test_dtype_entries_reject_unknown_dtype():
    ctx = _lib.get_ctx()
    typed = ("tiseg_softmax_argmax_typed", "tiseg_softmax_argmax_tta_typed", "tiseg_tta_mean_typed",
             "tiseg_postproc_dist_lambda_typed", "tiseg_postproc_hover_ex", "tiseg_cdnet_refine_typed",
             "tiseg_mtcdnet_refine_typed")
    for name in typed:
        with pytest.raises(_lib.TisegError, match=r"status 2\).*unknown dtype code 7"):
            ctx.call(name, 7, *[0] * (len(_lib.SIGNATURES[name]) - 2))
