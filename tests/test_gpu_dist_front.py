"""The front of the DIST post-process (csrc/dist.cu): k_dist_prep walks 128-column strips down bands of FR_BAND rows and
builds, in one pass over the distance map, the level image, the mask plane, the marker-candidate planes and the mask
area per tile; with lambda > 0 k_plateau_bits runs the same stencil on the H-reconstructed image.  Every case compares
markers, raw flood and instances of ops.postproc_dist bit for bit with the oracle, at the shapes, alignments and values
where the walk changes path: strip and band edges (whose halo comes from the lanes 0 / 31 and from the rows above and
below the band), widths off the four-pixel vector path, unaligned inputs, NaN / inf / out-of-range values, fp32 / fp16 /
bf16 inputs, lambda 0 and 2, and tiles whose mask covers more than half of them."""
import os
import re
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import tiseg_b200  # noqa: E402,F401
from tiseg_b200 import ops  # noqa: E402
from oracle import postprocess as opp  # noqa: E402
from oracle import skimage_port as sk  # noqa: E402

gpu = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tissue-image-segmentation_b200", "csrc", "dist.cu")
BAND = int(re.search(r"#define FR_BAND (\d+)", open(SRC).read()).group(1))     # rows per warp band
STRIP = 128                                                                      # columns per warp strip
DTYPES = ("float32", "float16", "bfloat16")

WS = (1, 2, 3, 5, 127, 128, 129, 130, 131, 255, 257, 1000, 1001)
HS = tuple(k * BAND + e for k in (1, 2) for e in (-2, -1, 0, 1, 2))
# every width at two heights, every height at two or three widths
SHAPES = [(HS[(i + j * 5) % len(HS)], W) for i, W in enumerate(WS) for j in (0, 1)]


def _diff(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, "%s: shape %r vs %r" % (what, a.shape, b.shape)
    bad = np.argwhere(a != b)
    assert len(bad) == 0, "%s: %d mismatching elements, first at %r: got %r want %r" % (
        what, len(bad), tuple(bad[0]), a[tuple(bad[0])], b[tuple(bad[0])])


def _want(d, lamb):
    """dist.py:275-284 and 114-129 for one fp32 map at `lamb`: (markers, raw flood, instances)"""
    x = np.copy(d)
    with np.errstate(invalid="ignore"):
        x[x > 255] = 255
        x[x < 0] = 0
        di = x.astype("int32")
    mask = (di > 0.5) + 0
    h = opp._h_reconstruction_erosion(255 - di.astype(np.uint8), lamb, literal=False)
    mk = sk.label(opp._find_maxima(h, mask, literal=False))
    return mk, sk.watershed(h, mk, mask=mask), opp.dist_dynamic_watershed(di, lamb, 0.5, literal=False)


def _as(d, dtype, offset=0):
    """fp32 numpy [N, H, W] -> a CUDA tensor of `dtype` starting `offset` elements into its storage, and the fp32 values
    it holds (the oracle's input)"""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(d, np.float32)).to(getattr(torch, dtype))
    if offset:
        buf = torch.zeros(t.numel() + offset, dtype=t.dtype, device="cuda")
        x = buf[offset:].view(t.shape)
        x.copy_(t)
    else:
        x = t.cuda()
    return x, t.float().numpy()


def _check(d, what, dtypes=("float32",), lambs=(0, 2), offset=0):
    d = np.asarray(d, np.float32)
    if d.ndim == 2:
        d = d[None]
    for dtype in dtypes:
        x, ref = _as(d, dtype, offset)
        if offset:
            assert x.data_ptr() % (4 * x.element_size()) != 0, "the view must defeat the vector path"
        for lamb in lambs:
            got = [a.cpu().numpy() for a in ops.postproc_dist(x, debug=True, lamb=lamb)]
            for n in range(d.shape[0]):
                mk, ws, inst = _want(ref[n], lamb)
                tag = "%s %s lamb=%d entry %d" % (what, dtype, lamb, n)
                _diff(got[1][n], mk, tag + ": markers")
                _diff(got[2][n], ws, tag + ": raw flood")
                _diff(got[0][n], inst, tag + ": instances")


def _blocky(H, W, seed, levels=7, size=3):
    """plateaus of `size`-pixel blocks at integer levels plus a fraction that truncation drops, with a sprinkle of
    single-pixel bumps: minimum plateaus, spoiled plateaus and background, everywhere in the tile"""
    rng = np.random.default_rng(seed)
    b = rng.integers(0, levels, ((H + size - 1) // size, (W + size - 1) // size))
    d = np.kron(b, np.ones((size, size)))[:H, :W] + rng.random((H, W)) * 0.9
    bump = rng.random((H, W)) < 0.01
    d[bump] += 1
    return d.astype(np.float32)


# --------------------------------------------------------------------------- CPU
def test_shapes_straddle_every_edge():
    assert BAND % 4 == 0 and BAND >= 8
    assert {W % STRIP for W in WS} >= {0, 1, 2, 3, STRIP - 1}, "widths at and around the strip width"
    assert {W % 4 for W in WS} == {0, 1, 2, 3}, "widths on and off the four-pixel vector path"
    assert sorted({H for H, _ in SHAPES}) == sorted(HS), "every height around the first two band edges"
    assert sorted({W for _, W in SHAPES}) == sorted(WS)


# --------------------------------------------------------------------------- GPU
@gpu
@pytest.mark.parametrize("H,W", SHAPES)
def test_shapes(H, W):
    _check(_blocky(H, W, H * 7919 + W), "%dx%d" % (H, W))


@gpu
def test_batches_and_dtypes():
    """N > 1 at a ragged and at a vector-path width, every input dtype"""
    for H, W in ((BAND + 1, 257), (2 * BAND - 2, 1000)):
        d = np.stack([_blocky(H, W, 100 + n) for n in range(3)])
        _check(d, "batch %dx%d" % (H, W), dtypes=DTYPES)


@gpu
@pytest.mark.parametrize("W", (128, 1000, 1001))
def test_unaligned_inputs(W):
    """a view one element into its storage: the scalar load path on a width the vector path would take"""
    H = BAND + 2
    d = np.stack([_blocky(H, W, 7 + W), _blocky(H, W, 8 + W)])
    _check(d, "unaligned %dx%d" % (H, W), dtypes=DTYPES, offset=1)


def _edge_plateaus(H, W, ys, xs, spoil):
    """one plateau of level 5 on a background of 3 for every edge column in `xs` / edge row in `ys`, ending on one side
    of it; `spoil` = 0: nothing else (a maximum plateau across the edge); 1 / 2: a pixel of 6 one / two pixels beyond
    the edge, so the plateau is not a maximum — with 2 the plateau's pixel next to the edge is a plain equal-valued
    non-candidate, and the flag has to come from the stencil of the stencil across the edge"""
    d = np.full((H, W), 3.0, np.float32)
    for x in xs:
        for side in (-1, 1):                                      # plateau left of the edge, or right of it
            y0 = 4 if side < 0 else H // 2 + 2
            if side < 0:
                px = slice(x - 6, x + (spoil == 2))
            else:
                px = slice(x - (spoil == 2), x + 6)
            d[y0:y0 + 5, px] = 5
            if spoil:
                sx = x + spoil - 1 if side < 0 else x - spoil
                d[y0 + 2, sx] = 6
    for y in ys:
        for side in (-1, 1):                                      # plateau above the edge, or below it
            x0 = 10 if side < 0 else W // 2 + 10
            if side < 0:
                py = slice(y - 6, y + (spoil == 2))
            else:
                py = slice(y - (spoil == 2), y + 6)
            d[py, x0:x0 + 5] = 5
            if spoil:
                sy = y + spoil - 1 if side < 0 else y - spoil
                d[sy, x0 + 2] = 6
    return d


@gpu
@pytest.mark.parametrize("spoil", (0, 1, 2))
def test_plateaus_across_strip_and_band_edges(spoil):
    H, W = 2 * BAND + 20, 3 * STRIP + 40
    d = _edge_plateaus(H, W, (BAND, 2 * BAND), (STRIP, 2 * STRIP, 3 * STRIP), spoil)
    _check(d, "plateaus at the edges, spoil %d" % spoil, dtypes=DTYPES)
    mk = ops.postproc_dist(d, debug=True)[1]
    if spoil == 0:
        assert mk.max() == 10, "each plateau is one maximum"
    else:
        # only the spoiling pixels are maxima: every plateau they touch is dropped
        assert mk.max() == 10 and (mk > 0).sum() == 10, (mk.max(), (mk > 0).sum())
    # the same plateaus on the corner where a strip edge meets a band edge
    c = np.full((H, W), 3.0, np.float32)
    c[BAND - 3:BAND + 3, STRIP - 3:STRIP + 3] = 5
    if spoil:
        c[BAND + spoil - 1, STRIP + spoil - 1] = 6
    _check(c, "plateau on a strip / band corner, spoil %d" % spoil)


@gpu
def test_value_extremes():
    H, W = BAND + 3, 2 * STRIP + 3
    d = _blocky(H, W, 5)
    rng = np.random.default_rng(6)
    specials = np.array([np.nan, np.inf, -np.inf, -3.5, -0.0, 255.0, 300.0, 1e30, 0.5, 254.99, 1.0, 0.49], np.float32)
    pick = rng.random((H, W)) < 0.08
    d[pick] = rng.choice(specials, int(pick.sum()))
    # specials on the strip edges and the band edge, where the halo is loaded separately
    for x in (STRIP - 2, STRIP - 1, STRIP, STRIP + 1, 2 * STRIP - 1, 2 * STRIP, 0, W - 1):
        d[::3, x] = specials[(x + np.arange(len(d[::3, x]))) % len(specials)]
    d[BAND - 1] = np.nan
    d[BAND, ::2] = 255.0
    for dt in DTYPES:
        _check(d, "extremes", dtypes=(dt,))
    _check(d[:, :2 * STRIP], "extremes, vector path", dtypes=DTYPES)


@gpu
def test_dense_masks_pick_the_background():
    """tiles whose mask covers more than half of them: the mask area of the front decides whether the label histogram
    runs, and there the largest flood region can outnumber the background"""
    H, W = BAND + 7, STRIP + 5
    sparse = _blocky(H, W, 11)
    sparse[sparse < 4] = 0                                         # well under half the tile in the mask
    dense = np.full((H, W), 9.0, np.float32)                       # one big plateau: one region, larger than the rest
    dense[H // 2, W // 2] = 10
    dense[:, :3] = 0
    half = _blocky(H, W, 12) + 1                                   # everything in the mask, many regions
    half[::5, ::7] = 0
    d = np.stack([sparse, dense, half])
    assert (d[0] >= 1).mean() < 0.5 < (d[1] >= 1).mean() and (d[2] >= 1).mean() > 0.5
    _check(d, "dense masks", dtypes=DTYPES)
