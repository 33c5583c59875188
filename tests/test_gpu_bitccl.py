"""The bit-plane labeller (csrc/bitccl.cuh) at its tile, word and strip boundaries, through its three consumers:
  DIST markers      8-connected components of the candidate plane, with the plateau flags carried to the final roots
  DIST mask blobs   4-connected components of the mask plane (planes derived from F by shifts)
  pair metrics      8-connected equal-value components of gt and pred (k_eqbits planes, one batch of 2N entries)
Each is compared bit for bit with the CPU oracle on the adversarial topologies of tests/topology.py: union chains that
cross many tiles, diagonal-only contacts on word / tile-column / tile-row / tile-corner edges, flagged plateaus whose
local root is not the final root.  The generators' own topology is checked first, on the CPU."""
import functools
import os
import sys

import numpy as np
import pytest
from scipy import ndimage as ndi

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import tiseg_b200  # noqa: E402,F401
from tiseg_b200 import ops  # noqa: E402
from oracle import metrics as om  # noqa: E402
from oracle import postprocess as opp  # noqa: E402
from oracle import skimage_port as sk  # noqa: E402
import topology as T  # noqa: E402

gpu = pytest.mark.gpu

# H around the 32-row tile height, W around the 32-pixel word and the 256-pixel tile / strip width; the odd widths take
# the scalar load path of k_eqbits and k_plateau_bits (W % 4 != 0)
SHAPES = [(1, 1000), (31, 257), (32, 256), (33, 513), (65, 255), (65, 1000), (33, 31), (31, 33), (65, 33)]


@functools.lru_cache(maxsize=None)
def _spiral(H, W):
    return T.spiral(H, W)


def _pattern(name, H, W):
    """binary pattern `name` at H x W (uint8)"""
    if name == "spiral":
        return _spiral(H, W).copy()
    if name == "comb":
        return T.comb(H, W)
    if name == "checker":
        return (T.checkerboard(H, W) == 2).astype(np.uint8)
    if name == "stairs":
        return T.staircase(H, W, 5) | T.staircase(H, W, 7, anti=True)
    if name == "perc8":
        return T.percolation(H, W, 0.41, H * 7919 + W)
    if name == "perc4":
        return T.percolation(H, W, 0.59, H * 7919 + W + 1)
    raise ValueError(name)


PATTERNS = ("spiral", "comb", "checker", "stairs", "perc8", "perc4")


def _diff(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, "%s: shape %r vs %r" % (what, a.shape, b.shape)
    bad = np.argwhere(a != b)
    assert len(bad) == 0, "%s: %d mismatching elements, first at %r: got %r want %r" % (
        what, len(bad), tuple(bad[0]), a[tuple(bad[0])], b[tuple(bad[0])])


# --------------------------------------------------------------------------- the generators (CPU)
def test_generators_have_the_claimed_topology():
    for H, W in [(1, 1), (1, 40), (2, 5), (31, 33), (65, 257), (96, 600)]:
        s = T.spiral(H, W)
        assert sk.label(s, connectivity=1).max() == 1, ("spiral", H, W)
        assert s.sum() >= 0.45 * H * W, ("spiral coverage", H, W, int(s.sum()))
        # one pixel wide: a simple path, every pixel has at most two 4-neighbours on it and exactly two are its ends
        p = np.pad(s, 1).astype(int)
        nb = (p[:-2, 1:-1] + p[2:, 1:-1] + p[1:-1, :-2] + p[1:-1, 2:])[s > 0]
        assert nb.max() <= 2 and (s.sum() == 1 or (nb == 1).sum() == 2), ("spiral width", H, W)
    big = _spiral(1000, 1000)
    assert sk.label(big, connectivity=1).max() == 1 and big.sum() >= 0.45 * 1000 * 1000
    rows = np.unique(np.nonzero(T.spiral(96, 96))[0])
    assert len(rows) == 96, "the spiral reaches every row"

    for H, W in [(65, 513), (96, 600)]:
        c = T.comb(H, W)
        assert sk.label(c, connectivity=1).max() == 1, ("comb", H, W)
        assert sk.label(c[:-1], connectivity=2).max() == (W + 1) // 2, "without the spine the teeth fall apart"
        c3 = T.comb(H, W, pitch=5, width=3)
        assert sk.label(c3, connectivity=1).max() == 1 and sk.label(c3[:-1], connectivity=2).max() == (W + 4) // 5

    for H, W, blk in [(64, 64, 1), (65, 513, 1), (96, 600, 32), (70, 300, 5)]:
        ck = T.checkerboard(H, W, 3, 8, block=blk)
        squares = ((H + blk - 1) // blk) * ((W + blk - 1) // blk)
        for v in (3, 8):
            assert sk.label(ck == v, connectivity=2).max() == 1, ("checker 8-conn", H, W, blk, v)
        assert sk.label(ck == 3, connectivity=1).max() + sk.label(ck == 8, connectivity=1).max() == squares
        assert sk.label(ck, connectivity=2).max() == 2, "equal-value labelling: one component per id"
        if blk == 1:
            assert sk.label(ck == 3, connectivity=1).max() == (H * W + 1) // 2

    for anti in (False, True):
        st = T.staircase(65, 257, 6, anti)
        assert sk.label(st, connectivity=1).max() == st.sum(), "staircase pixels touch only diagonally"
        lines = len(np.unique((np.add if anti else np.subtract)(*np.nonzero(st)[::-1])))
        assert sk.label(st, connectivity=2).max() == lines

    # near their thresholds, both random masks hold components over many scales, one of them spanning most tiles
    for p, conn in ((0.41, 2), (0.59, 1)):
        m = T.percolation(256, 512, p, 3)
        lab = sk.label(m, connectivity=conn)
        sizes = np.bincount(lab.ravel())[1:]
        assert abs(m.mean() - p) < 0.01 and lab.max() > 200 and sizes.max() > 2000, (p, conn, lab.max(), sizes.max())

    for kind in T.BOUNDARIES:
        for anti in (False, True):
            (ya, xa), (yb, xb) = T.diagonal_contact(kind, 1, anti)
            assert yb == ya + 1 and abs(xb - xa) == 1
            lo, hi = min(xa, xb), max(xa, xb)
            if kind in ("word", "tilecol", "corner"):
                edge = T.TILE_W if kind != "word" else T.WORD
                assert hi % edge == 0 and lo == hi - 1, (kind, anti)
            else:
                assert lo // T.WORD == hi // T.WORD, "a tile-row contact inside one word"
            if kind in ("tilerow", "corner"):
                assert yb % T.TILE_H == 0
            else:
                assert ya // T.TILE_H == yb // T.TILE_H, "a column contact inside one tile row"
            if kind == "word":
                assert hi % T.TILE_W != 0


# --------------------------------------------------------------------------- 1. DIST markers
def _check_dist(d, what):
    """markers, raw flood and instances of ops.postproc_dist against the oracle stage by stage; -> (markers, flood)"""
    got, mk, ws = ops.postproc_dist(d, debug=True)
    di = np.clip(d, 0, 255).astype("int32")
    inv = 255 - di.astype(np.uint8)
    mask = (di > 0.5) + 0
    want_mk = sk.label(opp._find_maxima(inv, mask, literal=False))
    _diff(mk, want_mk, what + ": markers")
    _diff(ws, sk.watershed(inv, want_mk, mask=mask), what + ": raw flood")
    _diff(got, opp.dist_postprocess(None, d, literal=False)[1], what + ": instances")
    return mk, ws


@gpu
@pytest.mark.parametrize("pattern", PATTERNS)
def test_dist_markers_on_adversarial_plateaus(pattern):
    """d = 1 + P: the mask is everything and the markers are exactly the 8-connected components of P"""
    for H, W in SHAPES:
        P = _pattern(pattern, H, W)
        mk, _ = _check_dist((1 + P).astype(np.float32), "%s %dx%d" % (pattern, H, W))
        if P.min() == 0:
            assert mk.max() == sk.label(P, connectivity=2).max(), (pattern, H, W)


@gpu
@pytest.mark.parametrize("pattern", ("spiral", "perc8", "perc4", "comb"))
def test_dist_markers_full_tile(pattern):
    P = _pattern(pattern, 1000, 1000)
    mk, _ = _check_dist((1 + P).astype(np.float32), "%s 1000x1000" % pattern)
    assert mk.max() == sk.label(P, connectivity=2).max()


def _leak_site(P, y0, y1, x0, x1):
    """the first background pixel of P in rows [y0, y1) x columns [x0, x1) with an 8-neighbour on P"""
    nb = ndi.binary_dilation(P > 0, structure=np.ones((3, 3), bool)) & (P == 0)
    ys, xs = np.nonzero(nb[y0:y1, x0:x1])
    assert len(ys), "no leak site in the window"
    return y0 + ys[0], x0 + xs[0]


@gpu
@pytest.mark.parametrize("pattern", ("spiral", "comb", "comb3"))
def test_dist_plateau_flag_reaches_the_final_root(pattern):
    """a plateau spanning 3 x 3 tiles next to one higher pixel is not a maximum: only that pixel is a marker, wherever
    the flag is raised — in the tile of the plateau's first raster pixel, in the last tile (whose local root is not the
    final root), on a tile corner.  On the one-pixel spiral and comb the non-candidates around the leak cut the plateau
    into several candidate components, each of which must be dropped."""
    H, W = 96, 700
    P = T.comb(H, W, pitch=4, width=3) if pattern == "comb3" else _pattern(pattern, H, W)
    assert sk.label(P, connectivity=2).max() == 1
    sites = {"first tile": _leak_site(P, 5, T.TILE_H, 0, T.TILE_W),
             "last tile": _leak_site(P, 2 * T.TILE_H, H, 2 * T.TILE_W, W),
             "tile corner": _leak_site(P, T.TILE_H - 1, T.TILE_H + 1, T.TILE_W - 1, T.TILE_W + 1)}
    for where, (y, x) in sites.items():
        d = (1 + P).astype(np.float32)
        d[y, x] = 3
        what = "%s, leak in the %s at (%d, %d)" % (pattern, where, y, x)
        mk, _ = _check_dist(d, what)
        assert mk.max() == 1 and mk[y, x] == 1 and (mk > 0).sum() == 1, what
        if pattern != "comb3":
            # the plateau minus the leak's neighbours falls apart: several candidate components, all flagged
            cand = P.copy()
            cand[max(y - 1, 0):y + 2, max(x - 1, 0):x + 2] = 0
            assert sk.label(cand, connectivity=2).max() > 1, what


# --------------------------------------------------------------------------- 2. DIST mask blobs
def _two_blobs(kind, anti, peak_below, H=64, W=300):
    """blobs A (above) and B (below) of level 2 whose only contact is the diagonal across `kind`; a level-3 peak on the
    contact pixel of one of them.  The other blob's plateau touches that peak diagonally, so it holds no marker, and
    the 4-connected flood cannot reach it: it stays 0."""
    (ya, xa), (yb, xb) = T.diagonal_contact(kind, 1, anti)
    d = np.zeros((H, W), np.float32)
    # A extends up and away from the contact, B down and away
    ax = slice(xa - 15, xa + 1) if not anti else slice(xa, xa + 16)
    bx = slice(xb, xb + 14) if not anti else slice(xb - 13, xb + 1)
    d[ya - 11:ya + 1, ax] = 2
    d[yb:yb + 13, bx] = 2
    if peak_below:
        d[yb, xb] = 3
    else:
        d[ya, xa] = 3
    return d, (slice(ya - 11, ya + 1), ax), (slice(yb, yb + 13), bx)


@gpu
@pytest.mark.parametrize("kind", T.BOUNDARIES)
def test_dist_blobs_touching_only_diagonally(kind):
    for anti in (False, True):
        for peak_below in (False, True):
            d, A, B = _two_blobs(kind, anti, peak_below)
            what = "%s anti=%s peak %s" % (kind, anti, "below" if peak_below else "above")
            mask = d > 0.5
            assert sk.label(mask, connectivity=1).max() == 2 and sk.label(mask, connectivity=2).max() == 1
            mk, ws = _check_dist(d, what)
            flooded, left = (B, A) if peak_below else (A, B)
            assert mk.max() == 1 and (ws[flooded] > 0).all() and (ws[left] == 0).all(), what

            # two markers in the flooded blob: the multi-marker flood, with the unmarked blob still left at 0
            d2 = d.copy()
            fy, fx = flooded
            far = (fy.stop - 1 if peak_below else fy.start, fx.stop - 1 if (peak_below != anti) else fx.start)
            d2[far] = 3
            mk2, ws2 = _check_dist(d2, what + ", second marker")
            assert mk2.max() == 2 and (ws2[left] == 0).all(), what

            # one marker plateau across the contact: its 8-connected extent spans both 4-connected blobs
            d3 = d.copy()
            (ya, xa), (yb, xb) = T.diagonal_contact(kind, 1, anti)
            d3[ya, xa] = d3[yb, xb] = 3
            mk3, ws3 = _check_dist(d3, what + ", marker across the contact")
            assert mk3.max() == 1 and (ws3[A] == 1).all() and (ws3[B] == 1).all(), what


# --------------------------------------------------------------------------- 3. pair metrics
def _records(p, g):
    return (tuple(np.float64(om.pre_eval_bin_aji(p, g, literal=False))),
            tuple(np.float64(om.pre_eval_bin_pq(p, g, literal=False))))


def _check_pairs(p, g, what):
    """a batch through pair_metrics_bin with int32 and with uint16 ground truth, every entry against the oracle"""
    p, g = np.asarray(p, np.int32), np.asarray(g, np.int32)
    aji, pq = ops.pair_metrics_bin(p, g)
    aji16, pq16 = ops.pair_metrics_bin(p, g.astype(np.uint16))
    for n in range(p.shape[0]):
        want = _records(p[n], g[n])
        assert (tuple(aji[n]), tuple(pq[n])) == want, (what, n, "int32 gt", aji[n], pq[n], want)
        assert (tuple(aji16[n]), tuple(pq16[n])) == want, (what, n, "uint16 gt", aji16[n], pq16[n], want)
    return aji, pq


def _id_map(name, H, W):
    """id images from the generators: binary patterns as id 1, and the multi-id maps"""
    if name == "checker_ids":
        return T.checkerboard(H, W, 5, 9)
    if name == "blocks32":
        return T.checkerboard(H, W, 4, 1000, block=32)        # same ids meet only diagonally at word / tile corners
    if name == "blocks5":
        return T.checkerboard(H, W, 2, 7, block=5)
    if name == "noise_ids":         # equal-value components of a 3-level noise, in 48-column bands around the strip edges
        rng = np.random.default_rng(H * 31 + W)
        x = np.arange(W)
        band = (np.abs((x + 24) % T.TILE_W - 24) < 24) | (x >= W - 24)
        return (rng.integers(1, 4, (H, W)) * (rng.random((H, W)) < 0.8) * band).astype(np.int32)
    return _pattern(name, H, W).astype(np.int32)


ID_MAPS = ("spiral", "comb", "checker_ids", "blocks32", "blocks5", "stairs", "perc8", "perc4", "noise_ids")


@gpu
@pytest.mark.parametrize("H,W", SHAPES)
def test_pair_metrics_on_generator_maps(H, W):
    """each map against the next one (gt and pred of different topology), and every map against itself, where the
    PQ true positives are the 8-connected equal-value components"""
    maps = np.stack([_id_map(n, H, W) for n in ID_MAPS])
    _check_pairs(maps, np.roll(maps, 1, axis=0), "generator maps %dx%d" % (H, W))
    _, pq = _check_pairs(maps, maps, "identity %dx%d" % (H, W))
    for n, X in enumerate(maps):
        assert pq[n, 0] == sk.label(X, connectivity=2).max(), (ID_MAPS[n], H, W)


@gpu
def test_pair_metrics_full_tile_spiral_and_checkerboard():
    X = np.stack([_spiral(1000, 1000).astype(np.int32), T.checkerboard(1000, 1000, 1, 2), _id_map("perc4", 1000, 1000)])
    _, pq = _check_pairs(X, X[::-1].copy(), "1000^2 maps")
    _, pq = _check_pairs(X, X, "1000^2 identity")
    assert tuple(pq[:, 0]) == (1, 2, sk.label(X[2], connectivity=2).max())


@gpu
def test_pair_metrics_boundary_cases():
    H, W = 70, 600
    cases = []
    # the same id in two disjoint pieces: two components
    a = np.zeros((H, W), np.int32); a[5:20, 10:300] = 7; a[40:60, 250:580] = 7
    b = np.zeros((H, W), np.int32); b[5:20, 10:290] = 3; b[40:60, 260:580] = 3
    cases.append(("disjoint pieces of one id", a, b))
    # different ids adjacent across each boundary kind, and the same id touching only diagonally there
    for kind in T.BOUNDARIES:
        for anti in (False, True):
            (ya, xa), (yb, xb) = T.diagonal_contact(kind, 1, anti)
            m = np.zeros((H, W), np.int32)
            m[ya - 8:ya + 1, :] = 5                              # band above the contact row ...
            m[yb:yb + 8, :] = 6                                  # ... a different id below it
            m[:, xb if xb > xa else xa] = 0                      # cut both bands at the column edge
            m[ya, xa] = 8; m[yb, xb] = 8                         # one id across the diagonal only
            m[yb, xa] = 9                                        # and a different id on the other diagonal
            cases.append(("adjacent ids at %s anti=%s" % (kind, anti), m, np.where(m == 8, 0, m)))
    # a thick spiral against a copy eroded by one column: IoU 2/3, one match
    s3 = np.kron(_spiral(H // 3, W // 3), np.ones((3, 3), np.uint8))
    s3 = np.pad(s3, ((0, H - s3.shape[0]), (0, W - s3.shape[1])))
    er = ndi.binary_erosion(s3, structure=np.ones((1, 2), bool)).astype(np.int32)
    cases.append(("spiral vs eroded spiral", s3.astype(np.int32) * 4, er * 11))
    # entries whose gt and pred hold very different numbers of components: a leak between the gt half and the pred half
    # of the 2N labelling batch shows as wrong counts
    dots = np.zeros((H, W), np.int32); dots[::2, ::2] = 1
    one = np.zeros((H, W), np.int32); one[3:H - 3, 3:W - 3] = 2
    cases.append(("one blob vs isolated dots", one, dots))
    cases.append(("isolated dots vs one blob", dots, one))
    cases.append(("empty vs noise", np.zeros((H, W), np.int32), _id_map("noise_ids", H, W)))
    p = np.stack([c[1] for c in cases]); g = np.stack([c[2] for c in cases])
    aji, pq = _check_pairs(p, g, "boundary cases")
    for n, (name, pn, gn) in enumerate(cases):
        a1, q1 = ops.pair_metrics_bin(pn, gn)
        assert tuple(a1) == tuple(aji[n]) and tuple(q1) == tuple(pq[n]), name
    tp_fp = pq[:, 0] + pq[:, 1]
    assert tp_fp[0] == 2, "two components of one id"
    assert tuple(pq[-3, :3]) == (0.0, 1.0, (H // 2) * (W // 2)) and tuple(pq[-2, :3]) == (0.0, (H // 2) * (W // 2), 1.0)
    assert pq[-4, 0] == 1, "the eroded spiral matches"


@gpu
def test_multiclass_metrics_on_a_checkerboard():
    """k_comp_class_bits reads the same root bitmaps: classes over a two-id checkerboard and over 32-pixel blocks"""
    C = 3
    H, W = 65, 513
    for block in (1, 32):
        g = T.checkerboard(H, W, 1, 2, block=block)
        p = T.checkerboard(H, W, 3, 4, block=block)
        p[:, 300:] = np.roll(p[:, 300:], 1, axis=0)
        gs = np.where(g == 1, 1, 2).astype(np.uint8)
        ps = np.where((p == 3) ^ (np.arange(W) >= 400)[None], 1, 2).astype(np.uint8)
        r = ops.pair_metrics_multiclass(p, ps, g, gs, C)
        rp, rg = om.re_instance(p), om.re_instance(g)
        dp, dg = om.assign_sem_class_to_insts(rp, ps, C), om.assign_sem_class_to_insts(rg, gs, C)
        wa = np.stack(om.pre_eval_aji(rp, rg, dp, dg, C, reduce_zero_label=False, literal=False))
        wp = np.stack(om.pre_eval_pq(rp, rg, dp, dg, C, reduce_zero_label=False, literal=False))
        assert np.array_equal(r["aji"].astype(np.float32).T, wa), (block, r["aji"], wa)
        assert np.array_equal(r["pq"].astype(np.float32).T, wp), (block, r["pq"], wp)
        assert (tuple(r["bin_aji"]), tuple(r["bin_pq"])) == _records(p, g), block


# --------------------------------------------------------------------------- 4. batches
@gpu
def test_batches_in_any_order_match_single_calls():
    H, W = 65, 513
    names = ("spiral", "comb", "checker", "stairs", "perc8")
    P = np.stack([_pattern(n, H, W) for n in names])
    d = (1 + P).astype(np.float32)
    d[0, 40, 1] = 3                                           # a flagged plateau in one entry only
    ids = np.stack([_id_map(n, H, W) for n in ("spiral", "blocks32", "checker_ids", "noise_ids", "perc4")])
    single_d = [ops.postproc_dist(d[n], debug=True) for n in range(len(names))]
    single_p = [ops.pair_metrics_bin(ids[n], ids[(n + 1) % 5]) for n in range(5)]
    for order in ([0, 1, 2, 3, 4], [4, 2, 0, 3, 1], [3, 0]):
        o = np.array(order)
        got = ops.postproc_dist(d[o].copy(), debug=True)
        for j, n in enumerate(order):
            for out, one, what in zip(got, single_d[n], ("instances", "markers", "raw flood")):
                _diff(out[j], one, "dist %s, entry %s at %d of %r" % (what, names[n], j, order))
        aji, pq = _check_pairs(ids[o], ids[(o + 1) % 5], "pair batch %r" % order)
        for j, n in enumerate(order):
            assert tuple(aji[j]) == tuple(single_p[n][0]) and tuple(pq[j]) == tuple(single_p[n][1]), (order, n)
    for n in range(len(names)):
        _check_dist(d[n], "batch entry %s alone" % names[n])
