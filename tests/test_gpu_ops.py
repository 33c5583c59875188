"""GPU parity tests: every operator of the C-ABI CUDA library against the CPU oracle (and scipy where the
reference calls scipy directly) on seeded inputs.  Integer outputs must be bit-exact."""
import os
import sys

import numpy as np
import pytest
from scipy import ndimage as ndi

pytestmark = pytest.mark.gpu

import tiseg_b200  # noqa: E402,F401
from tiseg_b200 import ops, synth  # noqa: E402
from oracle import metrics as om  # noqa: E402
from oracle import postprocess as opp  # noqa: E402
from oracle import skimage_port as sk  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import topology as T  # noqa: E402

G = os.path.join(os.path.dirname(__file__), "golden")
SHAPES = [(1, 1), (1, 40), (37, 1), (5, 33), (64, 64), (50, 97), (130, 257)]


def _diff(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, "%s: shape %r vs %r" % (what, a.shape, b.shape)
    bad = np.argwhere(a != b)
    assert len(bad) == 0, "%s: %d mismatching elements, first at %r: got %r want %r" % (
        what, len(bad), tuple(bad[0]), a[tuple(bad[0])], b[tuple(bad[0])])


# --------------------------------------------------------------------------- CCL
@pytest.mark.parametrize("conn", [1, 2])
def test_label_binary(conn):
    rng = np.random.default_rng(10 + conn)
    for shape in SHAPES:
        for dens in (0.15, 0.5, 0.62, 0.9):
            m = (rng.random(shape) < dens).astype(np.uint8)
            want, k = sk.label(m, connectivity=conn, return_num=True)
            got, kk = ops.label(m, connectivity=conn, return_num=True)
            _diff(got, want, "label %r dens %.2f conn %d" % (shape, dens, conn))
            assert kk == k


@pytest.mark.parametrize("conn", [1, 2])
def test_label_equal_value_int32_batched(conn):
    rng = np.random.default_rng(20 + conn)
    imgs = rng.integers(0, 5, (6, 70, 101)).astype(np.int32)
    for bg in (0, 3):
        want = np.stack([sk.label(x, background=bg, connectivity=conn) for x in imgs])
        got, cnt = ops.label(imgs, background=bg, connectivity=conn, return_num=True)
        _diff(got, want, "batched equal-value label bg=%d" % bg)
        _diff(cnt, want.reshape(6, -1).max(1), "label counts")


def test_label_adversarial():
    # spiral, checkerboard, comb: long union chains and many diagonal-only contacts
    H = W = 96
    spiral = T.spiral(H, W)
    assert sk.label(spiral, connectivity=1).max() == 1 and spiral.sum() >= 0.45 * H * W and spiral[:, 0].sum() > 1, \
        "one 4-connected spiral that turns at every corner and covers half the tile"
    checker = (T.checkerboard(H, W) == 2).astype(np.uint8)
    comb = T.comb(W, H).T.copy()                       # teeth along rows, spine down the last column
    for name, m in (("spiral", spiral), ("checker", checker), ("comb", comb)):
        for conn in (1, 2):
            _diff(ops.label(m, connectivity=conn), sk.label(m, connectivity=conn), "%s conn %d" % (name, conn))


def test_label_big_tile_and_device_pointers():
    import torch
    t = synth.gt_and_pred(77, 1000, 1000)
    want = sk.label(t["pred_inst"])
    got_host = ops.label(t["pred_inst"])
    _diff(got_host, want, "1000^2 label (host buffers)")
    dev = torch.from_numpy(t["pred_inst"]).cuda()
    got_dev = ops.label(dev)
    assert got_dev.is_cuda
    _diff(got_dev.cpu().numpy(), want, "1000^2 label (device pointers)")


def test_re_instance():
    rng = np.random.default_rng(5)
    img = rng.choice(np.array([0, 3, 9, 10, 500, 60000], np.int32), (3, 40, 50))
    want = np.stack([om.re_instance(x) for x in img])
    _diff(ops.re_instance(img), want, "re_instance")


# --------------------------------------------------------------------------- morphology
def test_fill_holes_remove_small_dilate():
    rng = np.random.default_rng(30)
    for shape in SHAPES:
        for dens in (0.3, 0.55, 0.8):
            m = rng.random(shape) < dens
            _diff(ops.binary_fill_holes(m), ndi.binary_fill_holes(m).astype(np.uint8), "fill_holes %r %.2f" % (shape, dens))
            for conn in (1, 2):
                _diff(ops.remove_small_objects(m, 5, conn).astype(bool), opp.remove_small_objects(m, 5, conn),
                      "remove_small_objects %r conn %d" % (shape, conn))
            lab = sk.label(m).astype(np.int32)
            _diff(ops.remove_small_objects(lab, 10), opp.remove_small_objects(lab, 10), "remove_small labels %r" % (shape,))
            for r in (1, 2, 3):
                _diff(ops.dilation(lab, "disk", r), opp.dilation(lab, opp.disk(r)), "dilation disk %d %r" % (r, shape))
            _diff(ops.dilation(lab, "square", 1), opp.dilation(lab, opp.square(3)), "dilation square3 %r" % (shape,))
            _diff(ops.erosion(lab, "square", 1), opp.erosion(lab, opp.square(3)), "erosion square3 %r" % (shape,))


# --------------------------------------------------------------------------- A1
def _torch_cuda_softmax_cls(lg):
    """The reference expression on the device the reference runs it on (base.py:321-339 + unet.py:62):
    ``sum(F.softmax(v, dim=1) for v in variants) / len(variants)`` then ``argmax(dim=1)``, in torch on the GPU.
    lg [N, T, C, H, W] -> (cls [N, H, W] uint8, prob [N, C, H, W])."""
    import torch
    import torch.nn.functional as F
    x = torch.from_numpy(np.ascontiguousarray(lg)).cuda()
    probs = [F.softmax(x[:, t], dim=1) for t in range(x.shape[1])]
    mean = sum(probs) / len(probs)
    return mean.argmax(dim=1).to(torch.uint8).cpu().numpy(), mean.cpu().numpy()


def _check_class_map(cls, prob, want_p, what):
    """A class map is an exact function (first maximum) of fp32 probabilities that carry the float tolerance:
    (1) the returned map IS the first maximum of the returned probabilities, everywhere;
    (2) the probabilities are within 1e-5 relative of the oracle's (north_star);
    (3) the map equals the oracle's wherever the oracle's top-2 margin exceeds that tolerance."""
    assert np.array_equal(cls, np.argmax(prob, axis=-3).astype(np.uint8)), what + ": cls is not argmax(prob)"
    np.testing.assert_allclose(prob, want_p, rtol=1e-5, atol=1e-7, err_msg=what)
    top2 = np.sort(want_p, axis=-3)[..., -2:, :, :]
    clear = (top2[..., 1, :, :] - top2[..., 0, :, :]) > 1e-6
    assert np.array_equal(cls[clear], np.argmax(want_p, axis=-3).astype(np.uint8)[clear]), what
    return float(clear.mean())


def test_softmax_argmax():
    rng = np.random.default_rng(40)
    for (T, C, H, W) in [(1, 2, 33, 47), (3, 3, 64, 64), (8, 7, 40, 50), (2, 9, 31, 65), (1, 7, 64, 64), (4, 3, 50, 50)]:
        lg = (rng.standard_normal((2, T, C, H, W)) * 3).astype(np.float32)
        cls, prob = ops.softmax_argmax(lg, want_prob=True)
        cls_only = ops.softmax_argmax(lg)                    # T == 1: the streaming path with the tie-band fallback
        assert np.array_equal(cls, cls_only)
        for n in range(2):
            want_p = opp.softmax_tta_mean(list(lg[n]))
            assert _check_class_map(cls[n], prob[n], want_p, "softmax_argmax T=%d C=%d" % (T, C)) > 0.999
            if T == 1:                                       # one variant: no accumulation, the maps must be identical
                assert np.array_equal(cls[n], opp.argmax_classes(want_p).astype(np.uint8))
        if T in (1, 2, 4, 8):      # (torch's CUDA `/ len` multiplies by the reciprocal: identical for powers of two)
            tc, tp = _torch_cuda_softmax_cls(lg)
            assert np.array_equal(cls, tc), "class map differs from torch's CUDA softmax + argmax (T=%d C=%d)" % (T, C)
            assert np.array_equal(prob, tp), "probabilities differ bitwise from torch's CUDA softmax (T=%d C=%d)" % (T, C)


def _ulp_spaced_logits(rng, N, T, C, H, W, magnitude):
    """Adversarial logits: per pixel and variant the classes sit 0..4 ulp apart around a base value (many exact ties
    and 1-ulp gaps), a random subset of the classes pushed far below."""
    base = (rng.uniform(0.5, 1.0, (N, T, 1, H, W)) * magnitude).astype(np.float32)
    k = rng.integers(0, 5, (N, T, C, H, W))
    x = base + np.zeros((1, 1, C, 1, 1), np.float32)
    for _ in range(4):
        x = np.where(k > 0, np.nextafter(x, np.float32(-np.inf)), x).astype(np.float32)
        k = k - 1
    far = rng.random((N, T, C, H, W)) < 0.2
    return np.where(far, x - np.float32(3.0) * np.float32(max(magnitude, 1.0)), x).astype(np.float32)


@pytest.mark.parametrize("C", [2, 3, 7])
@pytest.mark.parametrize("T", [1, 8])
def test_softmax_argmax_tie_band(T, C):
    """The reference's class map is the first maximum of the fp32 PROBABILITIES (base.py:332-336, unet.py:62), not of
    the logits: logits a few ulp below the maximum reach the same probability and an earlier class wins.  Full-map
    equality, no masks, against the numpy oracle and against torch's own CUDA softmax + argmax.

    magnitude 0.05: 4 ulp = 1.5e-8 < 2^-25, exp(-gap) == 1.0f in every libm -> exact probability ties everywhere, the
    first class of the cluster wins: oracle (numpy) == torch CUDA == library.
    Between gaps of ~3e-8 and ~3e-7 the libms themselves disagree (measured on the B200 box, scripts/exp_band_probe.py,
    scripts/tie_debug.py): exp(-1.19e-7) is 1 - 2^-23 (correct) under CUDA's expf and 1 - 2^-24 under numpy's AVX exp, the
    latter making e / s round onto 1 / s for C = 3; exp(-5.96e-8) is 1.0 under CUDA's expf and 1 - 2^-24 under numpy.  The
    reference evaluates F.softmax in torch on the GPU, so in that band the library follows CUDA's expf bit for bit
    (checked at magnitudes 3 and 0.4 against torch's own CUDA softmax + argmax, full map); the numpy oracle is
    compared where it is well defined (magnitude 0.05; magnitude 3 with C = 2, where no rounding tie can arise)."""
    rng = np.random.default_rng(4100 + 10 * T + C)
    for magnitude in (0.05, 3.0, 0.4):
        lg = _ulp_spaced_logits(rng, 2, T, C, 48, 64, magnitude)
        cls, prob = ops.softmax_argmax(lg, want_prob=True)
        assert np.array_equal(cls, ops.softmax_argmax(lg)), "fast path differs from the full softmax (T=%d C=%d)" % (T, C)
        tc, tp = _torch_cuda_softmax_cls(lg)
        assert np.array_equal(cls, tc), "differs from torch CUDA softmax + argmax (T=%d C=%d mag=%g)" % (T, C, magnitude)
        assert np.array_equal(prob, tp)
        if magnitude == 0.05 or (magnitude == 3.0 and T == 1 and C == 2):
            for n in range(2):
                want = opp.argmax_classes(opp.softmax_tta_mean(list(lg[n]))).astype(np.uint8)
                assert np.array_equal(cls[n], want), "differs from the oracle (T=%d C=%d mag=%g)" % (T, C, magnitude)
        if T == 1 and magnitude == 0.05:
            # the point of the test: the logits' own argmax is a different map here
            assert (np.argmax(lg[:, 0], axis=1) != cls).mean() > 0.05


# --------------------------------------------------------------------------- A2
@pytest.mark.parametrize("C,radius,edge", [(2, 1, None), (4, 1, None), (3, 3, 2), (7, 1, None)])
def test_postproc_unet(C, radius, edge):
    for j, (H, W) in enumerate([(64, 80), (128, 100), (256, 256)]):
        t = synth.gt_and_pred(3000 + 10 * C + j, H, W, num_classes=C)
        pred = t["pred_sem"].copy()
        if edge is not None:
            pred = np.where(synth.three_class_map(t["pred_inst"]) == 2, edge, (t["pred_inst"] > 0) * 1).astype(np.uint8)
        want_sem, want_inst = opp.unet_family_postprocess(pred.astype(np.int64), radius=radius, edge_id=edge)
        got_sem, got_inst = ops.postproc_unet(pred.copy(), C - 1 if edge is None else edge, radius, edge)
        _diff(got_inst, want_inst, "unet inst C=%d r=%d %dx%d" % (C, radius, H, W))
        _diff(got_sem, want_sem, "unet sem C=%d r=%d %dx%d" % (C, radius, H, W))


def test_postproc_unet_batched_and_dcan():
    tiles = [synth.gt_and_pred(3100 + j, 96, 96, num_classes=3) for j in range(5)]
    pred = np.stack([t["pred_sem"] for t in tiles])
    got_sem, got_inst = ops.postproc_unet(pred.copy(), 2, 1)
    for j in range(5):
        ws, wi = opp.unet_family_postprocess(pred[j].astype(np.int64), radius=1)
        _diff(got_inst[j], wi, "batched unet inst %d" % j)
        _diff(got_sem[j], ws, "batched unet sem %d" % j)
    cell = (tiles[0]["pred_inst"] > 0).astype(np.uint8)
    cont = (synth.three_class_map(tiles[0]["pred_inst"]) == 2).astype(np.uint8)
    ws, wi = opp.dcan_postprocess(cell.astype(np.int64), cont, radius=3)
    gs, gi = ops.postproc_unet(cell.copy(), 1, 3, None, kill=cont)
    _diff(gi, wi, "dcan inst")
    _diff(gs, ws, "dcan sem")


# --------------------------------------------------------------------------- A10
def _random_ws_case(rng, H, W, levels, nmark):
    img = ndi.uniform_filter(rng.random((H, W)), 5)
    img = np.floor(img / img.max() * (levels - 1)).astype(np.uint8)
    mk = np.zeros((H, W), np.int32)
    ys, xs = rng.integers(0, H, nmark), rng.integers(0, W, nmark)
    mk[ys, xs] = np.arange(1, nmark + 1)
    mk = ndi.grey_dilation(mk, size=(2, 2))
    mask = ndi.binary_opening(rng.random((H, W)) < 0.85, iterations=1) | (mk > 0)
    return img, mk, mask.astype(np.uint8)


def test_watershed_u8():
    rng = np.random.default_rng(50)
    for (H, W, levels, nmark) in [(1, 9, 3, 2), (20, 31, 4, 5), (64, 64, 8, 12), (100, 130, 256, 40), (128, 128, 2, 30),
                                 (20, 31, 256, 5), (40, 40, 64, 6), (60, 70, 31, 9), (60, 70, 33, 9), (200, 300, 20, 50)]:
        img, mk, mask = _random_ws_case(rng, H, W, levels, nmark)
        _diff(ops.watershed(img, mk, mask), sk.watershed(img, mk, mask), "watershed u8 masked %dx%d" % (H, W))
        _diff(ops.watershed(img, mk), sk.watershed(img, mk), "watershed u8 unmasked %dx%d" % (H, W))


def test_watershed_f64():
    rng = np.random.default_rng(51)
    for (H, W, nmark) in [(1, 9, 2), (20, 31, 5), (64, 64, 12), (100, 130, 40), (200, 300, 60)]:
        img, mk, mask = _random_ws_case(rng, H, W, 16, nmark)
        f = -ndi.gaussian_filter(img.astype(np.float64), 1.0)
        f[::3] = np.round(f[::3], 1)          # plateaus of equal doubles
        _diff(ops.watershed(f, mk, mask), sk.watershed(f, mk, mask), "watershed f64 masked %dx%d" % (H, W))
        _diff(ops.watershed(f, mk), sk.watershed(f, mk), "watershed f64 unmasked %dx%d" % (H, W))


# --------------------------------------------------------------------------- A8
@pytest.mark.parametrize("H,W,idx", [(120, 130, 3), (256, 256, 0), (256, 256, 1), (300, 517, 2), (97, 101, 4), (33, 385, 5),
                                     (65, 96, 6), (31, 29, 7)])
def test_postproc_dist(H, W, idx):
    t = synth.tile_dist(2, idx, H=H, W=W)
    _, want = opp.dist_postprocess(None, t["dist_logit"], literal=False)
    got, mk, ws = ops.postproc_dist(t["dist_logit"], debug=True)
    # stage by stage, so a mismatch names the stage
    d = np.clip(t["dist_logit"], 0, 255).astype("int32")
    inv = 255 - d.astype(np.uint8)
    want_mk = sk.label(opp._find_maxima(inv, (d > 0.5) + 0, literal=False))
    _diff(mk, want_mk, "dist markers")
    _diff(ws, sk.watershed(inv, want_mk, mask=(d > 0.5) + 0), "dist raw flood")
    _diff(got, want, "dist inst")
    assert got.max() > (3 if H * W > 10000 else 0)


def test_postproc_dist_full_tile_and_batch():
    tiles = [synth.tile_dist(2, j) for j in range(2)]
    dist = np.stack([t["dist_logit"] for t in tiles])
    got = ops.postproc_dist(dist)
    for j in range(2):
        _, want = opp.dist_postprocess(None, dist[j], literal=False)
        _diff(got[j], want, "dist inst 1000^2 tile %d" % j)


def test_postproc_dist_edge_cases():
    z = np.zeros((40, 50), np.float32)
    _diff(ops.postproc_dist(z), opp.dist_postprocess(None, z, literal=False)[1], "all-background dist")
    full = np.full((40, 50), 7.3, np.float32)          # one plateau covering everything: bg becomes the label
    _diff(ops.postproc_dist(full), opp.dist_postprocess(None, full, literal=False)[1], "all-foreground dist")
    big = np.full((30, 30), 300.0, np.float32); big[0, 0] = -5
    _diff(ops.postproc_dist(big), opp.dist_postprocess(None, big, literal=False)[1], "clipped dist")
    rng = np.random.default_rng(5)
    for (H, W) in [(1, 1), (1, 40), (37, 1), (2, 3), (4, 129)]:          # degenerate geometry, noisy levels
        d = (rng.random((H, W)) * 6).astype(np.float32)
        _diff(ops.postproc_dist(d), opp.dist_postprocess(None, d, literal=False)[1], "dist %dx%d" % (H, W))


def _dense_dist(H, W, seed, floor):
    """a tile whose mask covers nearly everything as ONE blob with many markers (beyond the shared-memory flood: it is
    flooded in global memory, on the label map), with holes that hold small islands (other blobs inside its bounding box:
    single-marker fills, multi-marker floods) — the consumers of the label map that read outside their own writes"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    d = np.full((H, W), floor, np.float32)
    for _ in range(25):
        cy, cx, h, r = rng.integers(10, H - 10), rng.integers(10, W - 10), rng.integers(3, 9), rng.integers(6, 20)
        d = np.maximum(d, floor + h * np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / (2.0 * r * r)))
    for _ in range(6):
        cy, cx, r = rng.integers(30, H - 30), rng.integers(30, W - 30), rng.integers(12, 22)
        rr = np.sqrt((yy - cy) ** 2 + (xx - cx) ** 2)
        d[rr < r] = 0.0                                                    # a hole ...
        d[rr < r - 6] = 2.0 + 3.0 * np.exp(-rr[rr < r - 6] ** 2 / 18.0)        # ... with an island
        if r > 16:                                                         # a second peak: the island is flooded, not filled
            d[(np.abs(yy - cy) < 3) & (np.abs(xx - cx - 5) < 3)] = 6.0
    return d.astype(np.float32)


@pytest.mark.parametrize("H,W,floor", [(400, 400, 3.0), (230, 310, 1.5), (400, 400, 0.0)])
def test_postproc_dist_dense_mask_and_huge_blob(H, W, floor):
    """the label map of the flood is not zero-filled: check the paths that depend on zeros elsewhere — the flood in global
    memory (a blob beyond the CTA-wide slice), the histogram of tiles whose mask covers more than half (background = most
    frequent label), the general relabelling — alone, in a batch with ordinary tiles, and with the debug outputs"""
    d = _dense_dist(H, W, 11, floor)
    _, want = opp.dist_postprocess(None, d, literal=False)
    _diff(ops.postproc_dist(d), want, "dense dist inst")
    got, mk, ws = ops.postproc_dist(d, debug=True)
    _diff(got, want, "dense dist inst (debug outputs)")
    inv = 255 - np.clip(d, 0, 255).astype("int32").astype(np.uint8)
    _diff(ws, sk.watershed(inv, mk, mask=(np.clip(d, 0, 255).astype("int32") > 0.5) + 0), "dense dist raw flood")
    other = synth.tile_dist(2, 3, H=H, W=W)["dist_logit"]
    batch = np.stack([other, d, other[::-1].copy(), d[:, ::-1].copy()])
    got = ops.postproc_dist(batch)
    for j in range(4):
        _diff(got[j], opp.dist_postprocess(None, batch[j], literal=False)[1], "dense dist batch entry %d" % j)


# --------------------------------------------------------------------------- A16 / A17 / A19
def test_pair_metrics_golden():
    mref = np.load(os.path.join(G, "metrics_ref.npz"))
    for i in range(int(mref["n_cases"])):
        n = "c%d" % i
        aji, pq = ops.pair_metrics_bin(mref[n + "_pred"], mref[n + "_gt"])
        assert tuple(aji) == tuple(mref[n + "_bin_aji"]), (n, aji, mref[n + "_bin_aji"])
        assert tuple(pq) == tuple(mref[n + "_bin_pq"]), (n, pq, mref[n + "_bin_pq"])


def test_pair_metrics_batched_vs_oracle():
    tiles = [synth.gt_and_pred(6000 + j, 256, 256) for j in range(8)]
    p = np.stack([t["pred_inst"] for t in tiles]); g = np.stack([t["gt_inst"] for t in tiles])
    aji, pq = ops.pair_metrics_bin(p, g)
    for j in range(8):
        assert tuple(aji[j]) == tuple(np.float64(om.pre_eval_bin_aji(p[j], g[j], literal=False))), j
        assert tuple(pq[j]) == tuple(np.float64(om.pre_eval_bin_pq(p[j], g[j], literal=False))), j


def test_pair_metrics_full_tile_and_noise():
    t = synth.gt_and_pred(6100, 1000, 1000)
    aji, pq = ops.pair_metrics_bin(t["pred_inst"], t["gt_inst"])
    assert tuple(aji) == tuple(np.float64(om.pre_eval_bin_aji(t["pred_inst"], t["gt_inst"], literal=False)))
    assert tuple(pq) == tuple(np.float64(om.pre_eval_bin_pq(t["pred_inst"], t["gt_inst"], literal=False)))
    # pathological: per-pixel random ids overflow the small pair table and take the retry path
    rng = np.random.default_rng(1)
    p = rng.integers(0, 400, (96, 96)).astype(np.int32); g = rng.integers(0, 400, (96, 96)).astype(np.int32)
    aji, pq = ops.pair_metrics_bin(p, g)
    assert tuple(aji) == tuple(np.float64(om.pre_eval_bin_aji(p, g, literal=False)))
    assert tuple(pq) == tuple(np.float64(om.pre_eval_bin_pq(p, g, literal=False)))


def test_sem_counts_golden():
    mref = np.load(os.path.join(G, "metrics_ref.npz"))
    C = 4
    for i in range(int(mref["n_cases"])):
        n = "c%d" % i
        counts, valid = ops.sem_counts(mref[n + "_pred_sem"], mref[n + "_gt_sem"], C)
        tp, fp, fn, pr, gt = (counts[k].astype(np.float32) for k in range(5))
        tn = np.float32(valid) - (tp + fp + fn)
        res = np.stack([tp, tn, fp, fn, pr, gt])[:, 1:]
        assert np.array_equal(res, mref[n + "_sem"]), n
    counts, valid = ops.sem_counts(mref["c0_pred_sem"], mref["ign_gt_sem"], C)
    tp, fp, fn, pr, gt = (counts[k].astype(np.float32) for k in range(5))
    res = np.stack([tp, np.float32(valid) - (tp + fp + fn), fp, fn, pr, gt])[:, 1:]
    assert np.array_equal(res, mref["ign_sem"])


# --------------------------------------------------------------------------- A18
def test_multiclass_metrics_golden_and_oracle():
    mref = np.load(os.path.join(G, "metrics_ref.npz"))
    C = 4
    for i in range(int(mref["n_cases"])):
        n = "c%d" % i
        p, g, ps, gs = mref[n + "_pred"], mref[n + "_gt"], mref[n + "_pred_sem"], mref[n + "_gt_sem"]
        r = ops.pair_metrics_multiclass(p, ps, g, gs, C)
        aji = r["aji"].astype(np.float32).T[:, 1:]            # [2, C-1]
        pq = r["pq"].astype(np.float32).T[:, 1:]              # [4, C-1]
        assert np.array_equal(aji, mref[n + "_aji"]), (n, aji, mref[n + "_aji"])
        assert np.array_equal(pq, mref[n + "_pq"]), (n, pq, mref[n + "_pq"])
        assert tuple(r["bin_aji"]) == tuple(mref[n + "_bin_aji"]), n
        assert tuple(r["bin_pq"]) == tuple(mref[n + "_bin_pq"]), n
        # slot 0 (dropped by reduce_zero_label) against the oracle
        rp, rg = om.re_instance(p), om.re_instance(g)
        dp, dg = om.assign_sem_class_to_insts(rp, ps, C), om.assign_sem_class_to_insts(rg, gs, C)
        wa = np.stack(om.pre_eval_aji(rp, rg, dp, dg, C, reduce_zero_label=False, literal=False))
        wp = np.stack(om.pre_eval_pq(rp, rg, dp, dg, C, reduce_zero_label=False, literal=False))
        assert np.array_equal(r["aji"].astype(np.float32).T, wa), n
        assert np.array_equal(r["pq"].astype(np.float32).T, wp), n


def test_multiclass_metrics_batched_conic_like():
    C = 7
    tiles = [synth.gt_and_pred(7000 + j, 256, 256, num_classes=C) for j in range(6)]
    st = lambda k: np.stack([t[k] for t in tiles])
    r = ops.pair_metrics_multiclass(st("pred_inst"), st("pred_sem"), st("gt_inst"), st("gt_sem"), C)
    for j, t in enumerate(tiles):
        rp, rg = om.re_instance(t["pred_inst"]), om.re_instance(t["gt_inst"])
        dp = om.assign_sem_class_to_insts(rp, t["pred_sem"], C)
        dg = om.assign_sem_class_to_insts(rg, t["gt_sem"], C)
        wa = np.stack(om.pre_eval_aji(rp, rg, dp, dg, C, literal=False))
        wp = np.stack(om.pre_eval_pq(rp, rg, dp, dg, C, literal=False))
        assert np.array_equal(r["aji"][j].astype(np.float32).T[:, 1:], wa), j
        assert np.array_equal(r["pq"][j].astype(np.float32).T[:, 1:], wp), j


# --------------------------------------------------------------------------- A12
def test_ddm_golden_and_cdnet_tail():
    o = np.load(os.path.join(G, "ordered_ref.npz"))
    for j in range(3):
        _diff(ops.ddm(o["dd%d_dir" % j].astype(np.uint8)), o["dd%d_out" % j], "ddm golden %d" % j)
    _diff(ops.ddm(np.zeros((16, 16), np.uint8)), o["dd_zero_out"], "ddm of an all-background map")
    for T, (H, W) in [(1, (64, 80)), (3, (96, 70))]:
        rng = np.random.default_rng(80 + T)
        t = synth.gt_and_pred(8000 + T, H, W)
        tc = synth.three_class_map(t["pred_inst"])
        sem = [synth.sem_logits(rng, tc, 3) for _ in range(T)]
        dirs, pts = zip(*[synth.direction_logits(rng, t["pred_inst"]) for _ in range(T)])
        for if_ddm in (True, False):
            want_sem, want_dir, want_dd = opp.cdnet_inference_tail(sem, list(dirs), list(pts), if_ddm=if_ddm)
            r = ops.cdnet_refine(np.stack(sem), np.stack(dirs), np.stack(pts), if_ddm=if_ddm)
            _diff(r["dir_map"], want_dir, "cdnet dir map T=%d" % T)
            _diff(r["dd"], want_dd, "cdnet dd map T=%d" % T)
            _check_class_map(r["cls"], r["sem_prob"], want_sem, "cdnet_refine T=%d if_ddm=%s" % (T, if_ddm))


# --------------------------------------------------------------------------- A13
def test_align_foreground_golden_and_multitask():
    o = np.load(os.path.join(G, "ordered_ref.npz"))
    for j in range(3):
        for key, tm in (("out", 20), ("out5", 5)):
            got = ops.align_foreground(o["af%d_seed" % j].astype(np.int32), o["af%d_fg" % j], tm)
            _diff(got, o["af%d_%s" % (j, key)], "align_foreground golden %d time %d" % (j, tm))
    for j, variant in enumerate(("unet", "cunet", "cdnet")):
        t = synth.gt_and_pred(8100 + j, 128, 150, num_classes=4)
        inner = synth.three_class_map(t["pred_inst"]) if variant != "unet" else (t["pred_inst"] > 0).astype(np.uint8)
        want_sem, want_inst = opp.multitask_postprocess(inner.astype(np.int64), t["pred_sem"].astype(np.int64), variant)
        canvas, inst = ops.postproc_multitask(inner, t["pred_sem"], 3, None if variant == "unet" else 2)
        _diff(inst, want_inst, "multitask inst (%s)" % variant)
        if variant != "cdnet":
            _diff(canvas, want_sem, "multitask sem canvas (%s)" % variant)


# --------------------------------------------------------------------------- A11
@pytest.mark.parametrize("H,W,idx", [(64, 100, 1), (256, 256, 0), (250, 131, 2), (500, 517, 3)])
def test_postproc_hover(H, W, idx):
    import cv2  # noqa: F401  (the oracle calls OpenCV exactly as the reference does)
    t = synth.tile_hover(3, idx, H=H, W=W)
    want, dbg = opp.hover_post_proc(t["fore_map"], t["hv_map"])
    got, blb, dist, mk = ops.postproc_hover(t["fore_map"], t["hv_map"], debug=True)
    _diff(blb, dbg["blb"], "hover blb")
    _diff(mk, dbg["marker"], "hover markers")
    _diff(dist, dbg["dist"], "hover flooded image (fp64, bit-exact)")
    _diff(got, want, "hover inst")
    assert got.max() > 3


@pytest.mark.parametrize("H,W,idx", [(64, 100, 1), (256, 256, 0), (125, 131, 2), (1, 40, 4), (33, 1, 5)])
def test_postproc_hover_scale2(H, W, idx):
    """The CoNIC configuration: cv2.resize x2 in, the chain at 2H x 2W, INTER_NEAREST back (hovernet.py:286-287, 363)."""
    t = synth.tile_hover(3, idx, H=max(H, 40), W=max(W, 40))
    fore, hv = np.ascontiguousarray(t["fore_map"][:H, :W]), np.ascontiguousarray(t["hv_map"][:H, :W])
    want, dbg = opp.hover_post_proc(fore, hv, scale_factor=2)
    got, blb, dist, mk = ops.postproc_hover(fore, hv, scale_factor=2, debug=True)
    assert blb.shape == (2 * H, 2 * W)
    _diff(blb, dbg["blb"], "hover x2 blb")
    _diff(mk, dbg["marker"], "hover x2 markers")
    _diff(dist, dbg["dist"], "hover x2 flooded image (fp64, bit-exact)")
    _diff(got, want, "hover x2 inst")


def test_postproc_hover_full_tile_batched():
    tiles = [synth.tile_hover(3, j) for j in range(2)]
    got = ops.postproc_hover(np.stack([t["fore_map"] for t in tiles]), np.stack([t["hv_map"] for t in tiles]))
    for j, t in enumerate(tiles):
        want, _ = opp.hover_post_proc(t["fore_map"], t["hv_map"])
        _diff(got[j], want, "hover inst 1000^2 tile %d" % j)


# --------------------------------------------------------------------------- A14
def test_distance_transforms_vs_scipy():
    rng = np.random.default_rng(140)
    cases = [np.ones((4, 5), np.uint8), np.zeros((3, 7), np.uint8)]
    for (H, W) in [(1, 1), (1, 40), (37, 1), (64, 64), (50, 97), (130, 257)]:
        cases.append((rng.random((H, W)) < 0.9).astype(np.uint8))
        m = ndi.binary_dilation(rng.random((H, W)) < 0.02, iterations=3).astype(np.uint8)
        cases.append(m)
    t = synth.tile_dist(2, 5, H=300, W=400)
    cases.append((t["gt_inst"] > 0).astype(np.uint8))
    for m in cases:
        want_e = ndi.distance_transform_edt(m)
        got_e = ops.distance_transform_edt(m)
        assert got_e.dtype == np.float64 and np.array_equal(got_e, want_e), "edt differs for shape %r" % (m.shape,)
        _diff(ops.distance_transform_cdt(m), ndi.distance_transform_cdt(m, metric="chessboard"), "cdt %r" % (m.shape,))
    big = np.stack([(synth.tile_dist(2, j)["gt_inst"] > 0).astype(np.uint8) for j in range(2)])
    got = ops.distance_transform_edt(big)
    for j in range(2):
        assert np.array_equal(got[j], ndi.distance_transform_edt(big[j]))


# --------------------------------------------------------------------------- A9
def test_reconstruction_erosion_vs_oracle():
    rng = np.random.default_rng(90)
    for (H, W, h) in [(1, 1, 3), (1, 40, 5), (37, 1, 2), (30, 33, 7), (64, 64, 1), (130, 257, 20), (200, 300, 60)]:
        x = ndi.uniform_filter(rng.integers(0, 256, (H, W)).astype(np.float64), 3).astype(np.uint8)
        seed = np.minimum(255, x.astype(np.int32) + h).astype(np.uint8)
        want = sk.reconstruction_erosion(seed.astype(np.float64), x.astype(np.float64)).astype(np.uint8)
        _diff(ops.reconstruction(seed, x), want, "reconstruction %dx%d h=%d" % (H, W, h))


@pytest.mark.parametrize("lamb", [1, 2, 5])
def test_postproc_dist_lambda(lamb):
    """dynamic_watershed_alias with lamb > 0 (H-minima reconstruction before the markers and the flood)."""
    t = synth.tile_dist(2, 7, H=200, W=230)
    d = np.clip(t["dist_logit"], 0, 255).astype("int32")
    want = opp.dist_dynamic_watershed(d, float(lamb), 0.5, literal=False)
    _diff(ops.postproc_dist(t["dist_logit"], lamb=lamb), want, "dist inst lambda=%d" % lamb)


# --------------------------------------------------------------------------- window stitch + TTA reverse fused into K1
@pytest.mark.parametrize("H,W,window,overlap", [(40, 52, 0, 0), (100, 131, 0, 0), (100, 131, 40, 16), (64, 64, 64, 20),
                                                (30, 45, 40, 10), (131, 100, 48, 17)])
def test_softmax_argmax_tta_windows(H, W, window, overlap):
    rng = np.random.default_rng(H * 1000 + W + window)
    rots, flips = [0, 0, 0, 0, 90, 90, 90, 90], ["none", "horizontal", "vertical", "diagonal"] * 2   # shipped TTA: 8 variants
    C, N = 3, 2
    variants, want = [], []
    for n in range(N):
        rev = []
        for t, (r, f) in enumerate(zip(rots, flips)):
            Ht, Wt = (W, H) if (r // 90) % 2 else (H, W)
            if window == 0:
                x = rng.standard_normal((C, Ht, Wt)).astype(np.float32) * 3
                full = x
            else:
                st = window - overlap
                pad_h = st - (Ht - window) % st if Ht - window > 0 else window - Ht
                pad_w = st - (Wt - window) % st if Wt - window > 0 else window - Wt
                M = ((Ht + pad_h - window) // st + 1) * ((Wt + pad_w - window) // st + 1)
                x = rng.standard_normal((M, C, window, window)).astype(np.float32) * 3
                full = opp.split_stitch(x, Ht, Wt, window, overlap)
            if n == 0:
                variants.append([x])
            else:
                variants[t].append(x)
            rev.append(opp.reverse_tta_transform(full, r, f))
        want.append(opp.softmax_tta_mean(rev))
    variants = [np.stack(v) for v in variants]
    cls, prob = ops.softmax_argmax_tta(variants, rots, flips, (H, W), window, overlap, want_prob=True)
    want = np.stack(want)
    assert prob.shape == want.shape
    _check_class_map(cls, prob, want, "softmax_argmax_tta")


# --------------------------------------------------------------------------- mudslide_watershed (§8f rank 3)
def test_mudslide_watershed_golden_and_oracle():
    m = np.load(os.path.join(G, "mudslide_ref.npz"))
    for j in range(5):
        d = m["m%d_dir" % j].copy()
        pred, boundary = ops.mudslide_watershed(m["m%d_seg" % j], d, m["m%d_fore" % j])
        _diff(pred, m["m%d_pred" % j], "mudslide pred (golden %d)" % j)
        _diff(boundary, m["m%d_boundary" % j], "mudslide boundary (golden %d)" % j)
        _diff(d, m["m%d_dir_after" % j], "mudslide dir_graph after (golden %d)" % j)
    # a batch of full-size tiles against the oracle
    rng = np.random.default_rng(31)
    segs, dirs, fores = [], [], []
    for j in range(2):
        t = synth.gt_and_pred(9800 + j, 256, 256, n=60)
        inst = t["pred_inst"]
        fore = ndi.binary_dilation(inst > 0, iterations=1)
        seg = ndi.binary_erosion(inst > 0, iterations=2)
        dl, _ = synth.direction_logits(rng, inst)
        dg = np.argmax(dl, 0).astype(np.uint8)
        dg[rng.random(dg.shape) < 0.05] = 3
        dg[~fore] = 0
        segs.append(seg); dirs.append(dg); fores.append(fore)
    dbatch = np.stack(dirs)
    pred, boundary = ops.mudslide_watershed(np.stack(segs), dbatch, np.stack(fores))
    for j in range(2):
        dj = dirs[j].astype(np.int64)
        wp, wb = opp.mudslide_watershed(segs[j].copy(), dj, fores[j].copy())
        _diff(pred[j], wp, "mudslide pred tile %d" % j)
        _diff(boundary[j], wb, "mudslide boundary tile %d" % j)
        _diff(dbatch[j], dj, "mudslide dir_graph tile %d" % j)


def test_assign_sem_class_to_insts_matches_reference():
    """datasets/utils/instance_semantic.py:68-93 against the (class, id) pairs the reference's own function produced
    (tests/golden/metrics_ref.npz), dict order included."""
    from tiseg_b200 import metrics as M
    m = np.load(os.path.join(G, "metrics_ref.npz"))
    names = sorted(k[:-len("_cls_pred")] for k in m.files if k.endswith("_cls_pred"))
    assert names
    for n in names:
        for side in ("pred", "gt"):
            got = M.assign_sem_class_to_insts(M.re_instance(m[n + "_" + side]), m[n + "_" + side + "_sem"], 4)
            flat = np.array([(c, i) for c, ids in got.items() for i in ids], np.int64).reshape(-1, 2)
            assert np.array_equal(flat, m[n + "_cls_" + side]), (n, side)
    assert np.array_equal(M.re_instance(m[names[0] + "_pred"]), m[names[0] + "_re_pred"])


def test_debug_dataset_adds_bound_metrics():
    """monuseg_debug.py:85,133-135: the three-class maps give BoundDice / BoundPrecision / BoundRecall (last class)."""
    import torch
    from tiseg_b200 import datasets, metrics as M
    tiles = [synth.tile_unet(1, 60 + j, 128, 128, 2) for j in range(3)]
    preds = []
    for t in tiles:
        cls = opp.argmax_classes(opp.softmax(t["sem_logit"]))
        sem, inst = opp.unet_family_postprocess(cls, radius=1)
        tc_pred = synth.three_class_map(inst).astype(np.uint8)
        tc_gt = synth.three_class_map(t["gt_inst"]).astype(np.uint8)
        preds.append(dict(sem_pred=sem.astype(np.uint8), inst_pred=inst.astype(np.int32), tc_pred=tc_pred, tc_gt=tc_gt))
    ds = datasets.MoNuSegDatasetDebug(sem_gts=[t["gt_sem"] for t in tiles], inst_gts=[t["gt_inst"] for t in tiles])
    res = ds.pre_eval(preds, [0, 1, 2])
    assert all("bound_sem_pre_eval_res" in r for r in res)
    ev, _ = ds.evaluate(res, logger="silent")
    want = [tuple(torch.from_numpy(x) for x in om.pre_eval_all_semantic_metric(p["tc_pred"], p["tc_gt"], 3)) for p in preds]
    bm = M.pre_eval_to_sem_metrics(want, metrics=["Dice", "Precision", "Recall"])
    for k in ("Dice", "Precision", "Recall"):
        assert ev["Bound" + k] == np.round(np.mean(bm[k][-1]) * 100, 2)
    plain, _ = datasets.MoNuSegDataset(sem_gts=[t["gt_sem"] for t in tiles], inst_gts=[t["gt_inst"] for t in tiles]).evaluate(
        [{k: v for k, v in r.items() if k != "bound_sem_pre_eval_res"} for r in res], logger="silent")
    assert all(ev[k] == v for k, v in plain.items())


# --------------------------------------------------------------------------- label generation (§8f rank 4)
def test_label_generation_golden_and_oracle():
    m = np.load(os.path.join(G, "labelgen_ref.npz"))
    for j in range(5):
        inst = m["l%d_inst" % j]
        hv = ops.gen_instance_hv_map(inst)
        assert hv.shape == m["l%d_hv" % j].shape and hv.dtype == np.float32
        _diff(hv, m["l%d_hv" % j], "hv map (golden %d)" % j)
        fixed = opp.fix_inst(inst)
        for norm in (0, 1):
            _diff(ops.instance_distance_map(fixed, bool(norm)), m["l%d_dist%d" % (j, norm)],
                  "distance map norm=%d (golden %d)" % (norm, j))
    # a batch of larger tiles against the oracle, touching instances included
    insts = np.stack([synth.gt_and_pred(9950 + j, 500, 500, n=250)["gt_inst"].astype(np.int32) for j in range(3)])
    hv = ops.gen_instance_hv_map(insts)
    d1 = ops.instance_distance_map(insts, True)
    d0 = ops.instance_distance_map(insts, False)
    for j in range(3):
        _diff(hv[j], opp.gen_instance_hv_map(insts[j]), "hv map tile %d" % j)
        _diff(d1[j], opp.instance_distance_map(insts[j], True), "distance map (norm) tile %d" % j)
        _diff(d0[j], opp.instance_distance_map(insts[j], False), "distance map tile %d" % j)


def test_fix_inst_and_bound_label_golden_and_oracle():
    m = np.load(os.path.join(G, "labelgen_ref.npz"))
    for j in range(5):
        inst = m["l%d_inst" % j]
        fixed = ops.fix_inst(inst)
        _diff(fixed, m["l%d_fixed" % j], "fix_inst (golden %d)" % j)
        for tag, radius in (("1", 1), ("3", 3), ("21", (2, 1))):
            sem, bound = ops.bound_label(m["l%d_sem" % j], fixed, 4, radius)
            _diff(sem, m["l%d_r%s_sem" % (j, tag)], "bound sem r=%s (golden %d)" % (tag, j))
            _diff(bound, m["l%d_r%s_bound" % (j, tag)], "bound map r=%s (golden %d)" % (tag, j))
    # ids with several pieces, pieces under 5 px, diagonal contacts, ids out of raster order
    rng = np.random.default_rng(77)
    insts = []
    for j in range(3):
        t = synth.gt_and_pred(9960 + j, 300, 340, n=120)["gt_inst"].astype(np.int32)
        perm = rng.permutation(int(t.max()) + 1)
        perm[perm == 0], perm[0] = perm[0], 0
        a = perm[t] // 2 * 3                                     # merges pairs of ids -> multi-piece ids, gaps in the ids
        a[rng.random(a.shape) < 0.02] = 0
        a[rng.random(a.shape) < 0.01] = 5
        insts.append(a.astype(np.int32))
    insts = np.stack(insts)
    fixed = ops.fix_inst(insts)
    for j in range(3):
        want = opp.fix_inst(insts[j])
        _diff(fixed[j], want, "fix_inst tile %d" % j)
        sem = ((want % 2) + 1).astype(np.uint8)
        s2, b2 = ops.bound_label(sem, want, 3, 2)
        ws_, wb = opp.bound_label(sem, want, 3, (2, 2))
        _diff(s2, ws_, "bound sem tile %d" % j)
        _diff(b2, wb, "bound map tile %d" % j)


def test_label_maker_classes_follow_the_reference_protocol():
    from tiseg_b200 import label_makers as lm
    m = np.load(os.path.join(G, "labelgen_ref.npz"))
    inst, sem = m["l1_inst"], m["l1_sem"]
    d = lm.DistanceLabelMake(inst_norm=True)(dict(sem_gt=sem.copy(), inst_gt=inst.copy(), seg_fields=[]))
    _diff(d["dist_gt"], m["l1_dist1"], "DistanceLabelMake dist_gt")
    assert d["seg_fields"] == ["dist_gt"]
    b = lm.BoundLabelMake(edge_id=4, selem_radius=(2, 1))(dict(sem_gt=sem.copy(), inst_gt=inst.copy(), seg_fields=[]))
    _diff(b["sem_gt_w_bound"], m["l1_r21_bound"], "BoundLabelMake sem_gt_w_bound")
    _diff(b["sem_gt"], m["l1_r21_sem"], "BoundLabelMake sem_gt")
    h = lm.HVLabelMake()(dict(inst_gt=inst.copy(), seg_fields=[]))
    _diff(h["hv_gt"], m["l1_hv"].transpose(2, 0, 1), "HVLabelMake hv_gt")


def test_unet_weight_map_golden_and_oracle():
    """UNetLabelMake: eroded instances bit-exact; the fp64 weight map within 1e-12 relative of the reference's (it ends
    in an exp)."""
    from tiseg_b200 import label_makers as lm
    m = np.load(os.path.join(G, "labelgen_ref.npz"))
    for j in (0, 1, 3, 4):
        d = lm.UNetLabelMake()(dict(sem_gt=m["l%d_sem" % j].copy(), inst_gt=m["l%d_inst" % j].copy(), seg_fields=[]))
        _diff(d["sem_gt_inner"], m["l%d_unet_inner" % j], "UNetLabelMake sem_gt_inner (golden %d)" % j)
        assert d["loss_weight_map"].dtype == np.float64
        np.testing.assert_allclose(d["loss_weight_map"], m["l%d_unet_w" % j], rtol=1e-12, atol=0)
    insts = np.stack([opp.fix_inst(synth.gt_and_pred(9970 + j, 200, 260, n=60)["gt_inst"].astype(np.int32)) for j in range(2)])
    inner, w = ops.unet_weight_map(insts, w0=7.5, sigma=3.0)
    for j in range(2):
        wi, ww = opp.unet_weight_map(insts[j], w0=7.5, sigma=3.0)
        _diff(inner[j], wi, "unet inner tile %d" % j)
        np.testing.assert_allclose(w[j], ww, rtol=1e-12, atol=0)


def test_label_makers_degenerate_geometry():
    rng = np.random.default_rng(9)
    for (H, W) in [(1, 1), (1, 40), (37, 1), (2, 3), (6, 65)]:
        inst = (rng.integers(0, 4, (H, W)) * rng.integers(0, 2, (H, W))).astype(np.int32)
        if W >= 8:
            inst[:, W // 4:W // 2], inst[:, W // 2:3 * W // 4] = 5, 6
        if H >= 8:
            inst[H // 4:H // 2], inst[H // 2:3 * H // 4] = 7, 8
        fixed = opp.fix_inst(inst)
        _diff(ops.fix_inst(inst), fixed, "fix_inst %dx%d" % (H, W))
        _diff(ops.gen_instance_hv_map(inst), opp.gen_instance_hv_map(inst), "hv map %dx%d" % (H, W))
        _diff(ops.instance_distance_map(fixed, True), opp.instance_distance_map(fixed, True), "distance map %dx%d" % (H, W))
        sem = (fixed > 0).astype(np.uint8)
        _diff(ops.bound_label(sem, fixed, 2, 3)[1], opp.bound_label(sem, fixed, 2, (3, 3))[1], "bound %dx%d" % (H, W))
        inner, w = ops.unet_weight_map(fixed)
        wi, ww = opp.unet_weight_map(fixed)
        _diff(inner, wi, "unet inner %dx%d" % (H, W))
        np.testing.assert_allclose(w, ww, rtol=1e-12, atol=0)


def test_postproc_dist_matches_reference_source_golden():
    """tiseg_postproc_dist_lambda_typed vs the outputs of the reference's own dist.py source text (tests/golden/dist_ref.npz)."""
    m = np.load(os.path.join(G, "dist_ref.npz"))
    for j in range(4):
        _diff(ops.postproc_dist(m["d%d_in" % j]), m["d%d_out" % j], "dist inst (reference source golden %d)" % j)


def test_segmentor_postprocesses_match_reference_source_golden():
    """The CUDA post-processes vs the outputs of the reference's own method source text (segmentors_ref.npz: unet.py,
    cdnet.py, dcan.py, multi_task_*.py, hovernet.py)."""
    m = np.load(os.path.join(G, "segmentors_ref.npz"))
    for j in range(3):
        pred = m["u%d_pred" % j].astype(np.uint8)
        sem, inst = ops.postproc_unet(pred.copy(), int(pred.max()), 1, None)
        _diff(sem, m["u%d_sem" % j], "unet sem (golden %d)" % j)
        _diff(inst, m["u%d_inst" % j], "unet inst (golden %d)" % j)
        pred = m["c%d_pred" % j].astype(np.uint8)
        sem, inst = ops.postproc_unet(pred.copy(), 3, 3, 3)
        _diff(sem, m["c%d_sem" % j], "cdnet sem (golden %d)" % j)
        _diff(inst, m["c%d_inst" % j], "cdnet inst (golden %d)" % j)
        sem, inst = ops.postproc_unet(m["d%d_cell" % j].astype(np.uint8), 1, 3, None, kill=m["d%d_cont" % j])
        _diff(sem, m["d%d_sem" % j], "dcan sem (golden %d)" % j)
        _diff(inst, m["d%d_inst" % j], "dcan inst (golden %d)" % j)
        sempred = m["m%d_sempred" % j].astype(np.uint8)
        for variant, first, edge in (("unet", "inner", None), ("cunet", "tc", 2), ("cdnet", "tc", 2)):
            canvas, inst = ops.postproc_multitask(m["m%d_%s" % (j, first)].astype(np.uint8), sempred, int(sempred.max()), edge)
            _diff(inst, m["m%d_%s_inst" % (j, variant)], "multitask inst %s (golden %d)" % (variant, j))
            if variant != "cdnet":
                _diff(canvas, m["m%d_%s_sem" % (j, variant)], "multitask canvas %s (golden %d)" % (variant, j))
        out = ops.postproc_hover(m["h%d_fore" % j], m["h%d_hv" % j], scale_factor=int(m["h%d_sf" % j]))
        _diff(out, m["h%d_out" % j], "hover inst (golden %d)" % j)


def test_dataset_pre_eval_matches_reference_source_golden():
    """CustomDataset.pre_eval (one batched CUDA pass per shape) vs the reference's own pre_eval source text run on the
    same predictions and ground truth (dataset_ref.npz), then evaluate on top of it."""
    from tiseg_b200 import datasets
    m = np.load(os.path.join(G, "dataset_ref.npz"))
    ds = datasets.CustomDataset(sem_gts=[m["p%d_gt_sem" % j] for j in range(4)], inst_gts=[m["p%d_gt_inst" % j] for j in range(4)],
                                names=["im%d" % j for j in range(4)])
    preds = [dict(sem_pred=m["p%d_sem_pred" % j], inst_pred=m["p%d_inst_pred" % j]) for j in range(4)]
    res = ds.pre_eval(preds, list(range(4)))
    for j, r in enumerate(res):
        assert r["name"] == str(m["p%d_name" % j])
        _diff(np.array(r["bin_aji_pre_eval_res"], np.float64), m["p%d_bin_aji" % j], "pre_eval bin aji %d" % j)
        _diff(np.array(r["bin_pq_pre_eval_res"], np.float64), m["p%d_bin_pq" % j], "pre_eval bin pq %d" % j)
        _diff(np.stack([np.asarray(x) for x in r["sem_pre_eval_res"]]), m["p%d_sem" % j], "pre_eval sem %d" % j)
    ev, _ = ds.evaluate(res, logger="silent")
    assert list(ev.keys()) == m["eval_keys"].tolist()
    np.testing.assert_allclose(np.array([float(v) for v in ev.values()]), m["eval_values"], rtol=0, atol=1e-9)


def test_conic_dataset_pre_eval_matches_reference_source_golden():
    """CoNICDataset.pre_eval vs conic.py:126-198 executed from source on the same inputs (dataset_ref.npz), values and
    dtypes; then evaluate on top of it: all 67 entries."""
    from tiseg_b200 import datasets
    m = np.load(os.path.join(G, "dataset_ref.npz"))
    ds = datasets.CoNICDataset(sem_gts=[m["q%d_gt_sem" % j] for j in range(3)], inst_gts=[m["q%d_gt_inst" % j] for j in range(3)])
    preds = [dict(sem_pred=m["q%d_sem_pred" % j], inst_pred=m["q%d_inst_pred" % j]) for j in range(3)]
    res = ds.pre_eval(preds, list(range(3)))
    for j, r in enumerate(res):
        _diff(np.array(r["bin_aji_pre_eval_res"], np.float64), m["q%d_bin_aji" % j], "conic bin aji %d" % j)
        _diff(np.array(r["bin_pq_pre_eval_res"], np.float64), m["q%d_bin_pq" % j], "conic bin pq %d" % j)
        for key in ("aji", "pq"):
            got = np.stack([np.asarray(x) for x in r[key + "_pre_eval_res"]])
            assert got.dtype == m["q%d_%s" % (j, key)].dtype, (key, got.dtype)
            _diff(got, m["q%d_%s" % (j, key)], "conic %s %d" % (key, j))
        _diff(np.stack([np.asarray(x) for x in r["sem_pre_eval_res"]]), m["q%d_sem" % j], "conic sem %d" % j)
    ev, _ = ds.evaluate(res, logger="silent")
    assert list(ev.keys()) == m["conic_eval_keys"].tolist()
    np.testing.assert_allclose(np.array([float(v) for v in ev.values()]), m["conic_eval_values"], rtol=0, atol=1e-9)


def test_softmax_argmax_tta_matches_reference_source_golden():
    """The fused stitch + TTA reverse + softmax + mean kernel vs BaseSegmentor.inference executed from source on the same
    recorded window logits (tta_ref.npz)."""
    from test_oracle_golden import _tta_case
    m = np.load(os.path.join(G, "tta_ref.npz"))
    for j in range(3):
        H, W, window, overlap, B, variants, rots, flips = _tta_case(m, j)
        cls, prob = ops.softmax_argmax_tta(variants, rots, flips, (H, W), window, overlap, want_prob=True)
        want = m["t%d_prob" % j]
        assert prob.shape == want.shape
        # (quarter-integer logits permuted over the variants: many class sums are mathematically EQUAL and are decided
        # by the last bit of the libm's exp — the margin condition of _check_class_map is what a float golden can pin)
        _check_class_map(cls, prob, want, "softmax_argmax_tta golden %d" % j)


def test_cdnet_refine_matches_reference_source_golden():
    from test_oracle_golden import _cdnet_case
    m = np.load(os.path.join(G, "tta_ref.npz"))
    for j in range(2):
        sem, dirs, pts, if_ddm = _cdnet_case(m, j)
        r = ops.cdnet_refine(np.stack(sem), np.stack(dirs), np.stack(pts), if_ddm=if_ddm)
        _diff(r["dir_map"], m["c%d_dir_out" % j], "cdnet dir map (reference source golden %d)" % j)
        np.testing.assert_allclose(r["sem_prob"], m["c%d_sem_out" % j], rtol=1e-5, atol=1e-7)


def test_monuseg_debug_pre_eval_matches_reference_source_golden():
    from tiseg_b200 import datasets
    m = np.load(os.path.join(G, "dataset_ref.npz"))
    ds = datasets.MoNuSegDatasetDebug(sem_gts=[m["d%d_gt_sem" % j] for j in range(2)], inst_gts=[m["d%d_gt_inst" % j] for j in range(2)],
                                      names=["m0", "m1"])
    preds = [dict(sem_pred=m["d%d_sem_pred" % j], inst_pred=m["d%d_inst_pred" % j], tc_pred=m["d%d_tc_pred" % j],
                  tc_gt=m["d%d_tc_gt" % j]) for j in range(2)]
    res = ds.pre_eval(preds, [0, 1])
    for j, r in enumerate(res):
        _diff(np.array(r["bin_aji_pre_eval_res"], np.float64), m["d%d_bin_aji" % j], "monuseg bin aji %d" % j)
        _diff(np.array(r["bin_pq_pre_eval_res"], np.float64), m["d%d_bin_pq" % j], "monuseg bin pq %d" % j)
        _diff(np.stack([np.asarray(x) for x in r["sem_pre_eval_res"]]), m["d%d_sem" % j], "monuseg sem %d" % j)
        _diff(np.stack([np.asarray(x) for x in r["bound_sem_pre_eval_res"]]), m["d%d_bound" % j], "monuseg bound %d" % j)
    ev, _ = ds.evaluate(res, logger="silent")
    assert list(ev.keys()) == m["monuseg_eval_keys"].tolist()
    np.testing.assert_allclose(np.array([float(v) for v in ev.values()]), m["monuseg_eval_values"], rtol=0, atol=1e-9)


def test_convenience_scores_match_reference():
    """binary_panoptic_quality / binary_inst_dice / dice_similarity_coefficient / precision_recall (the convenience
    scores of tiseg/utils that run in the reference) vs the reference's own functions (dataset_ref.npz)."""
    from tiseg_b200 import metrics as M
    m = np.load(os.path.join(G, "dataset_ref.npz"))
    for j in range(2):
        ip, ig, sp, sg = (m["s%d_%s" % (j, k)] for k in ("inst_pred", "inst_gt", "sem_pred", "sem_gt"))
        np.testing.assert_allclose(np.array(M.binary_panoptic_quality(ip, ig), np.float64), m["s%d_bin_pq" % j], rtol=1e-12)
        np.testing.assert_allclose(float(M.binary_inst_dice(ip, ig)), float(m["s%d_inst_dice" % j]), rtol=1e-12)
        d = np.asarray(M.dice_similarity_coefficient(sp, sg, 4))
        assert d.dtype == m["s%d_dice" % j].dtype
        _diff(d, m["s%d_dice" % j], "dice_similarity_coefficient %d" % j)
        p, r = M.precision_recall(sp, sg, 4)
        _diff(np.asarray(p), m["s%d_precision" % j], "precision %d" % j)
        _diff(np.asarray(r), m["s%d_recall" % j], "recall %d" % j)


# --------------------------------------------------------------------------- round-2 vectors (r2_ref.npz): the reference's
# own argument shapes through the reference-named entry points
def test_mtcdnet_tail_matches_reference_source_golden():
    """MultiTaskCDNet.inference tail (multi_task_cdnet.py:262-330) + its _ddm_enhencement (:548-564) vs the method executed
    from source; argmax maps as postprocess consumes them."""
    from test_oracle_golden import _mt_case
    from tiseg_b200 import segmentors
    m = np.load(os.path.join(G, "r2_ref.npz"))
    for j in range(3):
        tc, sem, dirs, pts, if_ddm, rots, flips = _mt_case(m, j)
        rev = lambda lst: np.stack([opp.reverse_tta_transform(x, int(r), str(f)) for x, r, f in zip(lst, rots, flips)])
        r = ops.mtcdnet_refine(rev(tc), rev(sem), rev(dirs), rev(pts), if_ddm=if_ddm, want_sem_prob=True)
        _check_class_map(r["tc_cls"], r["tc_prob"], m["m%d_tc_out" % j], "mtcdnet tc %d" % j)
        _check_class_map(r["sem_cls"], r["sem_prob"], m["m%d_sem_out" % j], "mtcdnet sem %d" % j)
        assert (r["dir_map"] != m["m%d_dir_out" % j]).mean() < 1e-3
        seg = segmentors.MultiTaskCDNet(num_classes=sem[0].shape[0], if_ddm=if_ddm)
        tcp, sem_cls, dir_map, tc_cls = seg.inference_tail(rev(tc), rev(sem), rev(dirs), rev(pts))
        assert np.array_equal(tc_cls, r["tc_cls"]) and np.array_equal(sem_cls, r["sem_cls"])
        out = seg.forward_eval(rev(tc), rev(sem), rev(dirs), rev(pts))
        want_sem, want_inst = opp.multitask_postprocess(np.asarray(r["tc_cls"]).astype(np.int64), np.asarray(r["sem_cls"]).astype(np.int64), "cdnet")
        _diff(out[0]["inst_pred"], want_inst, "MultiTaskCDNet.forward_eval inst %d" % j)
        _diff(out[0]["sem_pred"], want_sem, "MultiTaskCDNet.forward_eval sem %d" % j)


def test_mtcdnet_tail_vs_oracle_batched():
    rng = np.random.default_rng(91)
    for T, (H, W) in [(1, (64, 80)), (2, (96, 70))]:
        tiles = []
        for n in range(3):
            t = synth.gt_and_pred(8100 + 10 * T + n, H, W, num_classes=3)
            tc = [synth.sem_logits(rng, synth.three_class_map(t["pred_inst"]), 3) for _ in range(T)]
            sem = [synth.sem_logits(rng, t["pred_sem"], 3) for _ in range(T)]
            dirs, pts = zip(*[synth.direction_logits(rng, t["pred_inst"]) for _ in range(T)])
            tiles.append((np.stack(tc), np.stack(sem), np.stack(dirs), np.stack(pts)))
        batch = [np.stack([t[k] for t in tiles]) for k in range(4)]
        for if_ddm in (True, False):
            r = ops.mtcdnet_refine(*batch, if_ddm=if_ddm, want_sem_prob=True)
            for n in range(3):
                w_tc, w_sem, w_dir, w_dd = opp.mtcdnet_inference_tail(list(tiles[n][0]), list(tiles[n][1]), list(tiles[n][2]),
                                                                      list(tiles[n][3]), if_ddm)
                _diff(r["dir_map"][n], w_dir, "mtcdnet dir map")
                _diff(r["dd"][n], w_dd, "mtcdnet dd")
                _check_class_map(r["tc_cls"][n], r["tc_prob"][n], w_tc, "mtcdnet tc T=%d" % T)
                _check_class_map(r["sem_cls"][n], r["sem_prob"][n], w_sem, "mtcdnet sem T=%d" % T)


def test_ddm_enhencement_reference_argument_shapes():
    """CDNet._ddm_enhencement / MultiTaskCDNet._ddm_enhencement called like the reference: torch tensors [1,C,H,W],
    [1,H,W], [1,1,H,W], in place, on the CPU and on the GPU."""
    import torch
    from tiseg_b200 import segmentors
    m = np.load(os.path.join(G, "r2_ref.npz"))
    for j in range(2):
        for key, cls in (("cdnet", segmentors.CDNet), ("mtcdnet", segmentors.MultiTaskCDNet)):
            for dev in ("cpu", "cuda"):
                prob = torch.from_numpy(m["e%d_prob" % j].copy()).to(dev)
                got = cls._ddm_enhencement(prob, torch.from_numpy(m["e%d_dd" % j]).to(dev), torch.from_numpy(m["e%d_pt" % j]).to(dev))
                assert got is prob                                          # modified in place and returned, like the reference
                np.testing.assert_allclose(got.cpu().numpy(), m["e%d_%s" % (j, key)], rtol=1e-6, atol=0, err_msg="%s %d %s" % (key, j, dev))


def test_generate_direction_differential_map_reference_name():
    import torch
    from tiseg_b200 import segmentors
    o = np.load(os.path.join(G, "ordered_ref.npz"))
    for j in range(3):
        d = o["dd%d_dir" % j]
        got = segmentors.generate_direction_differential_map(torch.from_numpy(d.astype(np.int64))[None].cuda(), 9)
        assert tuple(got.shape) == (1,) + d.shape and got.dtype == torch.float32 and got.is_cuda
        _diff(got[0].cpu().numpy(), o["dd%d_out" % j], "generate_direction_differential_map (cuda tensor) %d" % j)
        got = segmentors.generate_direction_differential_map(d)                 # HxW numpy, like label_to_vector accepts
        _diff(got[0].numpy(), o["dd%d_out" % j], "generate_direction_differential_map (numpy) %d" % j)
    with pytest.raises(NotImplementedError):
        segmentors.generate_direction_differential_map(o["dd0_dir"], 9, use_reg=True)


def test_regression_head_tta_matches_reference_source_golden():
    """DIST.inference / HoverNet.inference executed from source (recorder network, whole and split inference): the
    distance head is the plain TTA mean, the hv head is variant 0, the foreground head a softmax mean."""
    from test_oracle_golden import _reg_case
    from tiseg_b200 import segmentors
    m = np.load(os.path.join(G, "r2_ref.npz"))
    for j in range(3):
        H, W, window, overlap, dv, rots, flips = _reg_case(m, "d", j, 1)
        _, _, _, _, sv, _, _ = _reg_case(m, "d", j, 0)
        seg = segmentors.Dist(2, test_cfg=dict(rotate_degrees=sorted(set(rots), key=rots.index), flip_directions=sorted(set(flips), key=flips.index)))
        sem_pred, dist = seg.inference_tail(sv, dv, (H, W), window, overlap)
        assert np.array_equal(dist, m["d%d_out1" % j][:, 0]), "dist head TTA mean %d" % j        # quarter-integers: exact
        got_mean = ops.tta_mean(dv, rots, flips, (H, W), window, overlap)
        assert np.array_equal(got_mean, m["d%d_out1" % j])
        want_p = m["d%d_out0" % j]
        top2 = np.sort(want_p, axis=1)[:, -2:]
        clear = (top2[:, 1] - top2[:, 0]) > 1e-6
        assert np.array_equal(sem_pred[clear], want_p.argmax(1).astype(np.uint8)[clear])
        # HoVer-Net: hv = variant 0 only
        _, _, _, _, hv, hrots, hflips = _reg_case(m, "h", j, 1)
        _, _, _, _, hs, _, _ = _reg_case(m, "h", j, 0)
        _, _, _, _, hf, _, _ = _reg_case(m, "h", j, 2)
        hseg = segmentors.HoverNet(3, test_cfg=dict(rotate_degrees=sorted(set(hrots), key=hrots.index), flip_directions=sorted(set(hflips), key=hflips.index)))
        sem_pred, hv_map, fore = hseg.inference_tail(hs, hv, hf, (H, W), window, overlap)
        assert np.array_equal(np.moveaxis(hv_map, -1, 1), m["h%d_out1" % j]), "hv head (variant 0) %d" % j
        np.testing.assert_allclose(fore, m["h%d_out2" % j][:, 1], rtol=1e-5, atol=1e-7)


def test_debug_tail_three_class_target():
    from tiseg_b200 import segmentors
    m = np.load(os.path.join(G, "r2_ref.npz"))
    for j in range(3):
        assert np.array_equal(segmentors.three_class_gt(m["g%d_wb" % j], int(m["g%d_nc" % j])), m["g%d_tc" % j])
    t = synth.gt_and_pred(8200, 64, 80, num_classes=3)
    rng = np.random.default_rng(92)
    tc_l = synth.sem_logits(rng, synth.three_class_map(t["pred_inst"]), 3)[None]
    sem_l = synth.sem_logits(rng, t["pred_sem"], 3)[None]
    wb = np.where(synth.three_class_map(t["gt_inst"]) == 2, 2, t["gt_sem"]).astype(np.int64)
    seg = segmentors.MultiTaskCUNetDebug(2)
    out = seg.forward_eval_debug(wb, tc_l, sem_l)
    assert set(out[0]) == {"tc_pred", "tc_gt", "sem_pred", "inst_pred"}
    assert np.array_equal(out[0]["tc_gt"], opp.three_class_gt(wb, 2))
    assert np.array_equal(out[0]["tc_pred"], ops.softmax_argmax(tc_l))


def test_pre_eval_reference_signatures_with_id_dictionaries_and_match_iou():
    """pre_eval_aji / pre_eval_pq fed the exact objects conic.py:178-188 feeds the reference (re_instance'd maps + the two
    id dictionaries), hand-made dictionaries included, and pre_eval_bin_pq with match_iou in (0.5, 1)."""
    from test_oracle_golden import _id_dict
    from tiseg_b200 import metrics as M
    m = np.load(os.path.join(G, "r2_ref.npz"))
    for k in range(int(m["n_pair_cases"])):
        n = "p%d" % k
        ip, ig = m[n + "_ip"], m[n + "_ig"]
        dp, dg = _id_dict(m, n, "dp"), _id_dict(m, n, "dg")
        for rz in (True, False):
            got = M.pre_eval_aji(ip, ig, dp, dg, 4, reduce_zero_label=rz)
            assert all(g.dtype == np.float32 for g in got)
            _diff(np.stack(got), m[n + "_aji_rz%d" % rz], "pre_eval_aji(dicts) %s rz=%s" % (n, rz))
            got = M.pre_eval_pq(ip, ig, dp, dg, 4, reduce_zero_label=rz)
            _diff(np.stack(got), m[n + "_pq_rz%d" % rz], "pre_eval_pq(dicts) %s rz=%s" % (n, rz))
        for mi in (0.5, 0.6, 0.75, 0.9):
            got = M.pre_eval_bin_pq(ip, ig, mi)
            assert tuple(np.float64(v) for v in got) == tuple(m[n + "_binpq_%d" % int(mi * 100)]), (n, mi, got)
        # the library's own class assignment gives the reference's dictionaries back
        if k == 0:
            assert M.assign_sem_class_to_insts(ip, np.zeros_like(ip, np.uint8), 4) == {0: [0] + sorted(set(np.unique(ip)) - {0})}
    with pytest.raises(NotImplementedError):
        M.pre_eval_bin_pq(m["p0_ip"], m["p0_ig"], 0.3)


def test_pair_metrics_uint16_ground_truth():
    """A ground truth shipped as uint16 (ids < 65536) gives the records of the int32 map, host and device buffers."""
    import torch
    tiles = [synth.gt_and_pred(6100 + j, 200, 260) for j in range(4)]
    p = np.stack([t["pred_inst"] for t in tiles]).astype(np.int32)
    g = np.stack([t["gt_inst"] for t in tiles]).astype(np.int32)
    g[1] = np.where(g[1] > 0, g[1] + 60000, 0)                       # large ids still below 65536
    aji, pq = ops.pair_metrics_bin(p, g)
    aji16, pq16 = ops.pair_metrics_bin(p, g.astype(np.uint16))
    assert np.array_equal(aji, aji16) and np.array_equal(pq, pq16)
    a2, q2 = ops.pair_metrics_bin(torch.from_numpy(p).cuda(), torch.from_numpy(g.astype(np.uint16)).cuda(), 0.6)
    a3, q3 = ops.pair_metrics_bin(p, g, 0.6)
    assert np.array_equal(a2.cpu().numpy(), a3) and np.array_equal(q2.cpu().numpy(), q3)
    odd = (np.arange(37 * 53).reshape(37, 53) % 7).astype(np.int32)   # ragged width: the scalar load path
    assert all(np.array_equal(x, y) for x, y in zip(ops.pair_metrics_bin(odd, odd[::-1].copy()),
                                                    ops.pair_metrics_bin(odd, odd[::-1].astype(np.uint16))))



@pytest.mark.parametrize("H,W", [(1, 1), (5, 7), (37, 53), (64, 131), (33, 260), (40, 1000), (3, 257), (70, 252)])
def test_pair_metrics_ragged_shapes_vs_oracle(H, W):
    """the plane builder walks 256-column strips, eight pixels per thread, with vector loads when W % 4 == 0: widths that
    end inside a thread's eight pixels, inside a vector, inside a word, one pixel past a strip; heights below the cluster
    size of the ranking kernel; int32 and uint16 ground truth; batch entries that differ"""
    t = [synth.gt_and_pred(6300 + H + W + k, max(H, 8), max(W, 8), n=max(1, H * W // 600)) for k in range(3)]
    p = np.stack([x["pred_inst"][:H, :W] for x in t]).astype(np.int32)
    g = np.stack([x["gt_inst"][:H, :W] for x in t]).astype(np.int32)
    g[2] = p[2]                                        # identical maps: every pair matches
    p[1, :, -1] = 9                                    # a one-pixel-wide instance on the last column
    aji, pq = ops.pair_metrics_bin(p, g)
    aji16, pq16 = ops.pair_metrics_bin(p, g.astype(np.uint16))
    assert np.array_equal(aji, aji16) and np.array_equal(pq, pq16)
    for n in range(3):
        assert tuple(aji[n]) == tuple(np.float64(om.pre_eval_bin_aji(p[n], g[n], literal=False))), (H, W, n)
        assert tuple(pq[n]) == tuple(np.float64(om.pre_eval_bin_pq(p[n], g[n], literal=False))), (H, W, n)
    # the other streaming passes of the headline step on the same shapes
    rng = np.random.default_rng(H * 1000 + W)
    lg = (rng.standard_normal((3, 1, 2, H, W)) * 2).astype(np.float32)
    lg[0, 0, 1] = lg[0, 0, 0]                          # exact ties everywhere: the tie-band path of the two-class argmax
    cls = ops.softmax_argmax(lg)
    for n in range(3):
        assert np.array_equal(cls[n], opp.argmax_classes(opp.softmax(lg[n, 0])).astype(np.uint8)), (H, W, n)
    sp, sg = (p > 0).astype(np.uint8), (g > 0).astype(np.uint8)
    sg[0, 0, 0] = 255                                  # ignore_index in a two-class map: the generic counting path
    counts, valid = ops.sem_counts(sp, sg, 2)
    for n in range(3):
        ok = sg[n] != 255
        want = [[((sp[n] == c) & (sg[n] == c) & ok).sum() for c in range(2)], [((sp[n] == c) & (sg[n] != c) & ok).sum() for c in range(2)],
                [((sp[n] != c) & (sg[n] == c) & ok).sum() for c in range(2)], [((sp[n] == c) & ok).sum() for c in range(2)],
                [((sg[n] == c) & ok).sum() for c in range(2)]]
        assert np.array_equal(np.asarray(counts[n]), np.array(want)) and int(valid[n]) == int(ok.sum()), (H, W, n)


# --------------------------------------------------------------------------- (f)4 DirectionLabelMake
def _dir_case(g, j):
    p = "d%d_" % j
    return p, int(g[p + "num_angles"]), bool(g[p + "to_center"])


def test_direction_label_make_matches_reference_golden():
    """DirectionLabelMake run from the reference's own files (tests/golden/make_golden_dir.py): the centre points, dist_gt
    and point_gt are reproduced bit for bit; the 11x11 gradient is a float32 sum whose order in the reference is torch's
    convolution backend's, so reg_dir_gt agrees to 2e-4 rad (circular) wherever the gradient is not ~0, dir_gt wherever the
    angle is not within 0.01 degrees of a class edge, and loss_weight_map away from those pixels."""
    from tiseg_b200 import label_makers
    g = np.load(os.path.join(G, "dirlabel_ref.npz"))
    checked = 0
    for j in range(int(g["n_cases"])):
        p, A, to_center = _dir_case(g, j)
        if not to_center:
            with pytest.raises(NotImplementedError):
                label_makers.DirectionLabelMake(to_center=False)
            continue
        data = dict(sem_gt=g[p + "sem"].copy(), inst_gt=g[p + "inst"].copy(), seg_fields=[])
        out = label_makers.DirectionLabelMake(num_angles=A)(data)
        fixed = g[p + "fixed"]
        assert np.array_equal(out["sem_gt"], g[p + "sem_gt"]) and out["sem_gt"].dtype == g[p + "sem_gt"].dtype
        assert out["dist_gt"].dtype == np.float32 and np.array_equal(out["dist_gt"], g[p + "dist_gt"]), "dist_gt case %d" % j
        assert out["point_gt"].dtype == np.float32 and np.array_equal(out["point_gt"], g[p + "point_gt"]), "point_gt case %d" % j
        assert out["dir_gt"].dtype == g[p + "dir_gt"].dtype and out["loss_weight_map"].dtype == g[p + "loss_weight_map"].dtype
        # conditioning of the angle, from the oracle's restatement of the same arithmetic
        o = opp.direction_label_make(g[p + "inst"], g[p + "sem"], A, True)
        step = 360.0 / A
        edge = np.abs(((o["angle"].astype(np.float64) + 180.0 - step / 2) / step) - np.round((o["angle"] + 180.0 - step / 2) / step)) * step
        soft = (np.abs(o["grad"]).max(-1) < 1e-4) | (edge < 0.01) | (fixed == 0)
        d = np.abs(out["reg_dir_gt"].astype(np.float64) - g[p + "reg_dir_gt"])
        d = np.minimum(d, 2 * np.pi - d)
        assert d[~soft].max() < 2e-4, ("reg_dir_gt", j, d[~soft].max())
        assert np.all(out["reg_dir_gt"][fixed == 0] == 0) and np.all(out["dir_gt"][fixed == 0] == 0)
        bad = out["dir_gt"] != g[p + "dir_gt"]
        assert not np.any(bad & ~soft), ("dir_gt", j, int((bad & ~soft).sum()))
        assert bad.sum() <= max(4, 0.01 * (fixed > 0).sum())
        if A == 8:
            near = ndi.binary_dilation(bad, structure=np.ones((3, 3), bool), iterations=2) if bad.any() else bad
            dw = np.abs(out["loss_weight_map"].astype(np.float64) - g[p + "loss_weight_map"])
            if not bad.any():
                assert dw.max() < 1e-5, ("loss_weight_map", j, dw.max())
            else:       # (the DDM is normalised by its tile extrema: a flipped class can only matter next to it)
                assert dw[~near].max() < 1e-5, ("loss_weight_map", j, dw[~near].max())
        else:
            assert not out["loss_weight_map"].any()
        checked += 1
    assert checked >= 5


def test_direction_labels_vs_oracle_batch():
    """a batch of larger tiles against the oracle restatement (same tolerances), incl. an instance that touches the border"""
    tiles = [synth.gt_and_pred(9960 + k, 128, 128, n=30)["gt_inst"].astype(np.int32) for k in range(3)]
    tiles[2][0:20, 100:128] = 500
    fixed = np.stack([opp.fix_inst(t) for t in tiles])
    assert np.array_equal(ops.fix_inst(np.stack(tiles)), fixed)
    r = ops.direction_labels(fixed, 8)
    for k in range(3):
        o = opp.direction_label_make(tiles[k], (tiles[k] > 0).astype(np.uint8), 8, True)
        assert np.array_equal(r["dist_gt"][k], o["dist_gt"]), k
        assert np.array_equal(r["point_gt"][k], o["point_gt"]), k
        soft = (np.abs(o["grad"]).max(-1) < 1e-4) | (fixed[k] == 0)
        d = np.abs(r["reg_dir_gt"][k].astype(np.float64) - o["reg_dir_gt"])
        d = np.minimum(d, 2 * np.pi - d)
        assert d[~soft].max() < 2e-4, (k, d[~soft].max())
        assert (r["dir_gt"][k] != o["dir_gt"]).sum() <= 0.01 * (fixed[k] > 0).sum()


def test_mtcdnet_regression_tail_matches_reference_source_golden():
    """MultiTaskCDNet(use_regression=True): the one-channel angle head (multi_task_cdnet.py:304-315) vs the method executed
    from source; direction classes identical (the vectors hold angles on class edges, below 0 and above 2 pi)."""
    from test_oracle_golden import _regr_case
    from tiseg_b200 import segmentors
    m = np.load(os.path.join(G, "reg_ref.npz"))
    for j in range(int(m["n_cases"])):
        tc, sem, dirs, pts, if_ddm, rots, flips = _regr_case(m, j)
        rev = lambda lst: np.stack([opp.reverse_tta_transform(x, int(r), str(f)) for x, r, f in zip(lst, rots, flips)])
        r = ops.mtcdnet_refine(rev(tc), rev(sem), rev(dirs), rev(pts), if_ddm=if_ddm, want_sem_prob=True)
        # (the background of the direction map is the argmax of the mean tc probabilities: compare where that is clear-cut)
        w_tc, _, w_dir, w_dd = opp.mtcdnet_inference_tail(list(rev(tc)), list(rev(sem)), list(rev(dirs)), list(rev(pts)), if_ddm,
                                                          use_regression=True)
        assert np.array_equal(w_dir, m["g%d_dir_out" % j])
        assert (r["dir_map"] != m["g%d_dir_out" % j]).mean() < 1e-3, j
        _check_class_map(r["tc_cls"], r["tc_prob"], m["g%d_tc_out" % j], "mtcdnet regression tc %d" % j)
        _check_class_map(r["sem_cls"], r["sem_prob"], m["g%d_sem_out" % j], "mtcdnet regression sem %d" % j)
        seg = segmentors.MultiTaskCDNet(num_classes=sem[0].shape[0], if_ddm=if_ddm, use_regression=True)
        _, sem_cls, dir_map, tc_cls = seg.inference_tail(rev(tc), rev(sem), rev(dirs), rev(pts))
        assert np.array_equal(tc_cls, r["tc_cls"]) and np.array_equal(dir_map, r["dir_map"])
        with pytest.raises(ValueError):
            segmentors.MultiTaskCDNet(num_classes=sem[0].shape[0], use_regression=False).inference_tail(rev(tc), rev(sem), rev(dirs), rev(pts))
