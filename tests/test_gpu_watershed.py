"""The ordered marker-controlled watershed (csrc/watershed.cu) at every size class and hand-over limit of its floods.

The library does not run one flood: each blob (4-connected mask component) takes one of several, chosen by its bounding
box framed by one pixel, (h + 2) (w + 2) cells, and by its area:
  uint8   one warp per blob in a big (classes 0-1) or small warp arena (classes >= WP_SMALL_CLS), one warp flooding a
          CTA-wide staging up to WP_GEN_CAP cells, one lane in global memory beyond it (flood_blob_global)
  fp64    dense ranks by k_rank_blobs<false> (area <= WR_SORT_SMALL) or <true> (<= WR_SORT_MAX); a ranked lane flood with
          up to SLOTS blobs per warp arena (cells <= ARENA), one CTA per blob up to WR_GEN_CAP cells, and the binary heap
          of k_ws_flood_f64 beyond WR_GEN_CAP cells or WR_SORT_MAX area
The limits are read from the source, so the cases move with them.  `flood_path` classifies blobs by the library's rules,
and a CPU test checks that the GPU cases of this file put flooded blobs (two or more marker labels) exactly at and just
past every limit and size class: no kernel outcome can show that.  The GPU tests then compare every output bit for bit
with the oracle's sequential (value, age, index) heap flood, sk.watershed.

NaN images are out of scope: the library makes no promise about them (the oracle's heap order is not total there)."""
import functools
import os
import re
import sys
import zlib
from collections import namedtuple

import numpy as np
import pytest
from scipy import ndimage as ndi

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import tiseg_b200  # noqa: E402,F401
from tiseg_b200 import ops  # noqa: E402
from oracle import postprocess as opp  # noqa: E402
from oracle import skimage_port as sk  # noqa: E402
import topology as T  # noqa: E402

gpu = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tissue-image-segmentation_b200", "csrc", "watershed.cu")

# evaluated in this order: an expression may only use names before it
DEFINES = ("WP_WARPS", "WP_BIG_WARPS", "WP_ARENA", "WP_SMALL_ARENA", "WP_SMALL_CLS", "WP_GEN_CAP", "WS_MAXCLS",
           "WR_SORT_SMALL", "WR_SORT_MAX", "WR_GEN_CAP")
F64_CONSTS = ("WARPS", "ARENA", "SLOTS")          # constexpr of watershed_f64_dev


def read_limits(path=SRC):
    """the flood limits of watershed.cu as ints; AssertionError naming what is missing or not understood"""
    with open(path, encoding="utf-8") as f:
        text = f.read()
    defs = {m.group(1): m.group(2).strip() for m in
            re.finditer(r"^#define[ \t]+(\w+)[ \t]+([^\n]*?)[ \t]*(?://[^\n]*)?$", text, re.M)}
    lim = {}
    for name in DEFINES:
        assert name in defs, "watershed.cu defines no %s" % name
        expr = defs[name]
        assert re.fullmatch(r"[\w\s()+*/-]+", expr), "%s = %r is not an integer expression" % (name, expr)

        def value(m):
            word = m.group(0)
            if word.isdigit():
                return word
            assert word in lim, "%s uses %s, which is not one of the limits read before it" % (name, word)
            return str(lim[word])
        lim[name] = int(eval(re.sub(r"\b\w+\b", value, expr).replace("/", "//"), {"__builtins__": {}}))
    at = text.find("int watershed_f64_dev(")
    assert at >= 0, "watershed.cu has no watershed_f64_dev"
    body = text[at:text.index("\n}\n", at)]
    for name in F64_CONSTS:
        m = re.search(r"\b%s\s*=\s*(\d+)\b" % name, body)
        assert m, "watershed_f64_dev sets no %s" % name
        lim[name] = int(m.group(1))
    # k_rank_blobs scans the sorted values in chunks of its CTA: <true> and <false> launch bounds
    m = re.search(r"__launch_bounds__\(LARGE \? (\d+) : (\d+)\)\s*k_rank_blobs\(", text)
    assert m, "watershed.cu has no k_rank_blobs with launch bounds LARGE ? n : m"
    lim["RANK_CHUNK_LARGE"], lim["RANK_CHUNK_SMALL"] = int(m.group(1)), int(m.group(2))
    return lim


LIM = read_limits()


def size_class(cells, arena, slots):
    """blob_class: -1 beyond the arena, else the most slots of arena / (c + 1) cells the box fits, capped"""
    if cells > arena:
        return -1
    return min(arena // cells - 1, slots - 1)


@functools.lru_cache(maxsize=None)
def class_top(c, arena, slots):
    """the largest cell count of size class c"""
    return max(n for n in range(1, arena + 1) if size_class(n, arena, slots) == c)


Blob = namedtuple("Blob", "path cls cells area h w y0 x0 labels rank")


def flood_path(mask, kind, markers=None):
    """The flood of csrc/watershed.cu that takes each 4-connected blob of `mask`, by the rules of blob_class,
    k_flood_scatter (uint8) and blob_is_huge / k_rank_blobs (fp64).  kind: "u8" (tiseg_watershed_u8, forest mode),
    "dist" (the DIST chain, mask mode: blobs with fewer than two marker labels are filled, not flooded) or "f64".
    -> one Blob per blob in label order; `labels` counts the distinct marker labels on it, `rank` names the ranking
    kernel (fp64; None when the blob is not ranked)."""
    lab, n = sk.label(np.asarray(mask) != 0, connectivity=1, return_num=True)
    area = np.bincount(lab.ravel(), minlength=n + 1)
    labels = np.zeros(n + 1, np.int64)
    if markers is not None:
        mk = np.asarray(markers).astype(np.int64)
        sel = (lab > 0) & (mk != 0)
        pairs = np.unique(lab[sel] * (int(mk.max()) + 1) + mk[sel])
        labels = np.bincount(pairs // (int(mk.max()) + 1), minlength=n + 1)
    out = []
    for i, (sy, sx) in enumerate(ndi.find_objects(lab), 1):
        h, w = sy.stop - sy.start, sx.stop - sx.start
        cells, a = (h + 2) * (w + 2), int(area[i])
        cls, rank = None, None
        if kind in ("u8", "dist"):
            if kind == "dist" and labels[i] < 2:
                path = "fill"
            elif cells > LIM["WP_GEN_CAP"]:
                path = "u8 global"
            elif cells > LIM["WP_ARENA"]:
                path = "u8 cta"
            else:
                cls = size_class(cells, LIM["WP_ARENA"], LIM["WS_MAXCLS"])
                path = "u8 warp small" if cls >= LIM["WP_SMALL_CLS"] else "u8 warp big"
        else:
            huge = cells > LIM["WR_GEN_CAP"] or a > LIM["WR_SORT_MAX"]
            rank = "rank small" if a <= LIM["WR_SORT_SMALL"] else None if huge else "rank large"
            if huge:
                path = "f64 heap"
            elif cells > LIM["ARENA"]:
                path = "f64 cta"
            else:
                path, cls = "f64 lane", size_class(cells, LIM["ARENA"], LIM["SLOTS"])
        out.append(Blob(path, cls, cells, a, h, w, sy.start, sx.start, int(labels[i]), rank))
    return out


# --------------------------------------------------------------------------- case construction
def _rng(name):
    return np.random.default_rng(zlib.crc32(name.encode()))


def _seeds(rng, b, k):
    """k marker pixels (labels 1..k in random order) on the host pixels (b == 1) of one blob: with k >= 2 two of them
    side by side in one row, with k >= 6 a run of them every other cell of one row (seeds of one level inside one
    32-cell window).  The islands of a "holes" blob (b == 2) get two markers, one or none, in turn."""
    mk = np.zeros(b.shape, np.int32)
    host = np.argwhere(b == 1)
    chosen = []
    if k >= 2:
        pairs = [(y, x) for y, x in host[rng.permutation(len(host))[:4000]] if x + 1 < b.shape[1] and b[y, x + 1] == 1]
        if pairs:
            y, x = pairs[0]
            chosen += [(y, x), (y, x + 1)]
    if k >= 6:
        y, x = host[rng.integers(len(host))]
        chosen += [(y, x + 2 * j) for j in range(min(k // 2, 12)) if x + 2 * j < b.shape[1] and b[y, x + 2 * j] == 1]
    chosen = list(dict.fromkeys((int(y), int(x)) for y, x in chosen))[:k]
    taken = set(chosen)
    for i in rng.permutation(len(host)):
        if len(chosen) >= min(k, len(host)):
            break
        p = (int(host[i][0]), int(host[i][1]))
        if p not in taken:
            chosen.append(p)
            taken.add(p)
    for lab, (y, x) in zip(rng.permutation(len(chosen)) + 1, chosen):
        mk[y, x] = lab
    nxt = len(chosen) + 1
    isl = sk.label(b == 2, connectivity=1)
    for j, (sy, sx) in enumerate(ndi.find_objects(isl)):
        for y, x in ((sy.start, sx.start), (sy.stop - 1, sx.stop - 1))[:(2, 1, 0)[j % 3]]:
            mk[y, x] = nxt
            nxt += 1
    return mk


def _item(rng, shape, h, w, k):
    b = T.blob(shape, h, w)
    return b, _seeds(rng, b, k)


def _pack(items, width, gap=1):
    """Shelf-pack blobs (arrays: 0 background, 1 host, 2 islands) with their local markers left to right in rows
    `gap` pixels apart and crop to the tight box: the first blob touches the top-left corner, the last shelf the
    bottom edge, the widest one the right edge.  -> (kind array 0 / 1 / 2, markers int32 numbered across the sheet)"""
    place, x, y, shelf = [], 0, 0, 0
    for b, _ in items:
        h, w = b.shape
        assert w <= width, (h, w, width)
        if x and x + w > width:
            x, y, shelf = 0, y + shelf + gap, 0
        place.append((y, x))
        x, shelf = x + w + gap, max(shelf, h)
    H = max(py + b.shape[0] for (py, _), (b, _) in zip(place, items))
    W = max(px + b.shape[1] for (_, px), (b, _) in zip(place, items))
    kindarr, mk, off = np.zeros((H, W), np.uint8), np.zeros((H, W), np.int32), 0
    for (py, px), (b, m) in zip(place, items):
        h, w = b.shape
        kindarr[py:py + h, px:px + w] = np.maximum(kindarr[py:py + h, px:px + w], b)
        mk[py:py + h, px:px + w] += np.where(m > 0, m + off, 0).astype(np.int32)
        off += int(m.max())
    return kindarr, mk


U8_PALETTES = {"two": [17, 18], "four": [0, 85, 170, 255], "full": list(range(256)), "top": [253, 254, 255]}


def _f64_palette():
    one = 1.0
    return np.array([-np.inf, -1e300, -1.0, -0.0, 0.0, 5e-324, 1e-310, np.nextafter(1e-310, 1.0), 0.5,
                     np.nextafter(one, 0.0), one, np.nextafter(one, 2.0), 2.0, np.inf])


F64_PALETTES = {"special": _f64_palette(), "ties": np.array([-0.0, 0.0, 1.0, np.nextafter(1.0, 2.0)])}


def _values(rng, mask, mk, palette):
    """image values drawn from `palette`; the seeds of each blob share one value of it, and on every other blob of an
    fp64 palette that holds 0 the seeds are -0.0 and +0.0 at random (which must tie)"""
    pal = np.asarray(palette)
    img = pal[rng.integers(len(pal), size=mask.shape)]
    lab = sk.label(mask != 0, connectivity=1)
    vb = pal[rng.integers(len(pal), size=lab.max() + 1)]
    s = (mk != 0) & (lab > 0)
    img[s] = vb[lab[s]]
    if pal.dtype.kind == "f" and (pal == 0).any():
        zero = s & (lab % 2 == 1)
        img[zero] = np.where(rng.random(int(zero.sum())) < 0.5, -0.0, 0.0)
    return img


MARKS = (2, 3, 12, 40)


def _u8_class_items(rng, lim_arena, slots, shapes_at=("box", "serpentine"), shapes_past=("frame", "stairs"), copies=None):
    """blobs exactly at the top of every size class and one framed-box size past it, in two shapes each"""
    items = []
    for c in range(slots):
        top = class_top(c, lim_arena, slots)
        at, past = T.cells_at_most(top), T.cells_above(top)
        n_at = copies(c) if copies else len(shapes_at)
        for j in range(n_at):
            shape = shapes_at[j % len(shapes_at)]
            items.append(_item(rng, shape, *T.box_for(at, "square" if shape in ("box", "frame") else "flat"), MARKS[j % 4]))
        for j, shape in enumerate(shapes_past):
            items.append(_item(rng, shape, *T.box_for(past, "square" if shape in ("box", "frame") else "flat"),
                               MARKS[(j + c) % 4]))
    return items


def _extras(rng):
    """a single-marker blob, a blob without a marker, a holes blob whose islands take two markers, one or none"""
    return [_item(rng, "box", 9, 13, 1), _item(rng, "serpentine", 7, 20, 0), _item(rng, "holes", 30, 40, 12)]


def _sheet_u8(name):
    rng = _rng(name)
    gcap = LIM["WP_GEN_CAP"]
    if name == "classes":
        items = _u8_class_items(rng, LIM["WP_ARENA"], LIM["WS_MAXCLS"]) + _extras(rng)
        return _pack(items, 800)
    if name == "cta":
        at, past = T.box_for(T.cells_at_most(gcap)), T.box_for(T.cells_above(gcap))
        items = [_item(rng, "box", *at, 40), _item(rng, "holes", *at, 30), _item(rng, "box", *past, 40),
                 _item(rng, "stairs", *past, 3), _item(rng, "frame", *T.box_for(T.cells_above(LIM["WP_ARENA"])), 12)]
        return _pack(items, max(at[1], past[1]) + 1)
    if name == "lines":           # one-row blobs: the widest staged rows (fdiv's magic division) at every u8 limit
        items = []
        for limit in (LIM["WP_SMALL_ARENA"], LIM["WP_ARENA"], gcap):
            w_at = limit // 3 - 2                               # 3 (w + 2) <= limit
            items += [_item(rng, "box", 1, w_at, 40), _item(rng, "box", 1, w_at + 1, 3)]
        return _pack(items, max(b.shape[1] for b, _ in items))
    raise ValueError(name)


U8_SHEETS = {"classes-two": ("classes", "two"), "classes-four": ("classes", "four"), "classes-full": ("classes", "full"),
             "classes-top": ("classes", "top"), "cta-four": ("cta", "four"), "cta-full": ("cta", "full"),
             "lines-two": ("lines", "two"), "lines-top": ("lines", "top"), "columns-four": ("lines", "four")}


def _unmasked_boxes():
    """whole images (one blob) at and just past every u8 limit, and one row at the CTA slice"""
    out = []
    for limit in (LIM["WP_SMALL_ARENA"], LIM["WP_ARENA"], LIM["WP_GEN_CAP"]):
        out += [T.box_for(T.cells_at_most(limit)), T.box_for(T.cells_above(limit))]
    if LIM["WP_GEN_CAP"] % 3 == 0:
        out.append((1, LIM["WP_GEN_CAP"] // 3 - 2))
    return out


U8_CASES = sorted(U8_SHEETS) + ["whole-%dx%d" % hw for hw in _unmasked_boxes()]


@functools.lru_cache(maxsize=None)
def u8_case(name):
    """-> (image uint8, markers int32, mask uint8 or None)"""
    rng = _rng("u8 " + name)
    if name.startswith("whole-"):
        H, W = map(int, name[6:].split("x"))
        mk = _seeds(rng, np.ones((H, W), np.uint8), 30)
        pal = list(U8_PALETTES)[(H * 7 + W) % len(U8_PALETTES)]
        return _values(rng, np.ones((H, W), np.uint8), mk, U8_PALETTES[pal]).astype(np.uint8), mk, None
    sheet, pal = U8_SHEETS[name]
    kindarr, mk = _sheet_u8(sheet)
    if name.startswith("columns"):
        kindarr, mk = np.ascontiguousarray(kindarr.T), np.ascontiguousarray(mk.T)
    mask = (kindarr > 0).astype(np.uint8)
    img = _values(rng, mask, mk, U8_PALETTES[pal]).astype(np.uint8)
    bg = np.argwhere(mask == 0)                  # a few markers off the mask, which the flood must drop
    if len(bg):
        for j, (y, x) in enumerate(bg[rng.permutation(len(bg))[:3]]):
            mk[y, x] = int(mk.max()) + 1 + j
    return img, mk, mask


# ---- DIST: d = 0 off the blobs, random levels >= 1 on them; the islands of a holes blob take two peaks each
def _dist_from(kindarr, rng, levels):
    lo, hi = levels
    d = np.where(kindarr > 0, rng.integers(lo, hi + 1, size=kindarr.shape), 0).astype(np.float32)
    isl = sk.label(kindarr == 2, connectivity=1)
    for sy, sx in ndi.find_objects(isl):
        d[sy, sx] = 1.0
        d[sy.start, sx.start] = d[sy.stop - 1, sx.stop - 1] = 3.0
    return d


DIST_SHEETS = {"classes-3": ("classes", (1, 3)), "classes-deep": ("classes", (1, 255)), "cta-3": ("cta", (1, 3)),
               "lines-2": ("lines", (1, 2))}
DIST_CASES = sorted(DIST_SHEETS)


@functools.lru_cache(maxsize=None)
def dist_case(name):
    """-> dist fp32 [H, W]"""
    sheet, levels = DIST_SHEETS[name]
    return _dist_from(_sheet_u8(sheet)[0], _rng("dist " + name), levels)


@functools.lru_cache(maxsize=None)
def dist_batch():
    """four tiles; blobs one framed-box size past WP_GEN_CAP (flooded in global memory) in tiles 1 and 3 only, two
    of them and a holes blob whose islands carry two peaks each in tile 3"""
    rng = _rng("dist batch")
    past = T.box_for(T.cells_above(LIM["WP_GEN_CAP"]))
    small = lambda: [_item(rng, s, *T.box_for(T.cells_at_most(class_top(c, LIM["WP_ARENA"], LIM["WS_MAXCLS"])), "flat"), 3)
                     for c, s in ((0, "box"), (3, "serpentine"), (9, "box"), (15, "frame"))]
    tiles = [small() + small(), [_item(rng, "box", *past, 3)] + small(), small(),
             [_item(rng, "serpentine", *past, 3), _item(rng, "holes", *past, 3), _item(rng, "box", *past, 3)] + small()]
    packed = [_pack(t, past[1] + 40)[0] for t in tiles]
    H, W = max(p.shape[0] for p in packed), max(p.shape[1] for p in packed)
    return np.stack([_dist_from(np.pad(p, ((0, H - p.shape[0]), (0, W - p.shape[1]))), rng, (1, 3)) for p in packed])


def dist_stages(d):
    """(mask, inverted image, markers) of DIST's flood, by the oracle"""
    di = np.clip(d, 0, 255).astype("int32")
    inv = 255 - di.astype(np.uint8)
    mask = (di > 0.5) + 0
    return mask, inv, sk.label(opp._find_maxima(inv, mask, literal=False))


# ---- fp64
def _area_item(rng, area, w, k):
    b = T.area_blob(area, w)
    return b, _seeds(rng, b, k)


def _sheet_f64(name):
    rng = _rng(name)
    if name == "classes":           # c + 1 blobs at the top of class c fill one warp's slots; two past it
        items = _u8_class_items(rng, LIM["ARENA"], LIM["SLOTS"], shapes_at=("box", "serpentine", "frame", "stairs"),
                                shapes_past=("box", "stairs"), copies=lambda c: c + 1)
        return _pack(items + _extras(rng), 900)
    if name == "limits":
        ss, sm, gc = LIM["WR_SORT_SMALL"], LIM["WR_SORT_MAX"], LIM["WR_GEN_CAP"]
        a_past = T.box_for(T.cells_above(LIM["ARENA"]))
        g_at, g_past = T.box_for(T.cells_at_most(gc)), T.box_for(T.cells_above(gc), "flat")
        side = int(round(np.sqrt(sm)))
        items = [_item(rng, "box", *a_past, 12), _item(rng, "stairs", *a_past, 3),
                 _item(rng, "serpentine", *g_at, 40), _item(rng, "frame", *g_at, 12),
                 _item(rng, "box", *g_past, 40), _item(rng, "stairs", *g_past, 3),      # area < ss, box past gc
                 _item(rng, "serpentine", *g_past, 12), _item(rng, "holes", 60, 90, 12)]
        for a in (ss, ss + 1, sm, sm + 1):
            for w in ((32, 50) if a <= ss + 1 else (side, side + 22)):
                items.append(_area_item(rng, a, w, 12))
        return _pack(items, 900)
    raise ValueError(name)


F64_SHEETS = {"classes-special": ("classes", "special"), "classes-ties": ("classes", "ties"),
              "limits-special": ("limits", "special"), "limits-ties": ("limits", "ties")}


def _unmasked_f64():
    out = []
    for limit in (LIM["ARENA"], LIM["WR_GEN_CAP"]):
        out += [T.box_for(T.cells_at_most(limit)), T.box_for(T.cells_above(limit))]
    side = int(round(np.sqrt(LIM["WR_SORT_SMALL"])))
    return out + [(side, side)]


F64_CASES = sorted(F64_SHEETS) + ["whole-%dx%d" % hw for hw in _unmasked_f64()]


@functools.lru_cache(maxsize=None)
def f64_case(name):
    """-> (image float64, markers int32, mask uint8 or None)"""
    rng = _rng("f64 " + name)
    if name.startswith("whole-"):
        H, W = map(int, name[6:].split("x"))
        mk = _seeds(rng, np.ones((H, W), np.uint8), 30)
        return _values(rng, np.ones((H, W), np.uint8), mk, F64_PALETTES["special"]), mk, None
    sheet, pal = F64_SHEETS[name]
    kindarr, mk = _sheet_f64(sheet)
    mask = (kindarr > 0).astype(np.uint8)
    return _values(rng, mask, mk, F64_PALETTES[pal]), mk, mask


# ---- batches that mix every flood across their tiles
@functools.lru_cache(maxsize=None)
def mixed_batch(kind):
    """four tiles of one shape: warp / lane floods in every tile, the CTA staging in two, the global (u8) or heap (fp64)
    flood in tiles 1, 2 and 3 -> (images, markers, masks)"""
    rng = _rng("batch " + kind)
    if kind == "u8":
        cta, big = T.box_for(T.cells_at_most(LIM["WP_GEN_CAP"])), T.box_for(T.cells_above(LIM["WP_GEN_CAP"]))
        small = lambda: [_item(rng, s, *T.box_for(T.cells_at_most(class_top(c, LIM["WP_ARENA"], LIM["WS_MAXCLS"])), "flat"), m)
                         for c, s, m in ((0, "box", 40), (1, "serpentine", 12), (2, "box", 3), (7, "frame", 2),
                                         (15, "box", 3))]
        tiles = [small(), [_item(rng, "box", *cta, 40), _item(rng, "stairs", *big, 3)] + small(),
                 [_item(rng, "box", *big, 40)] + small(),
                 [_item(rng, "serpentine", *big, 12), _item(rng, "frame", *cta, 12)] + small()]
        pal = U8_PALETTES["four"]
    else:
        cta = T.box_for(T.cells_at_most(LIM["WR_GEN_CAP"]))
        heap = T.box_for(T.cells_above(LIM["WR_GEN_CAP"]), "flat")
        small = lambda: [_item(rng, s, *T.box_for(T.cells_at_most(class_top(c, LIM["ARENA"], LIM["SLOTS"])), "flat"), m)
                         for c in (0, 3, 15) for s, m in (("box", 12), ("serpentine", 3))]
        tiles = [small(), [_item(rng, "serpentine", *cta, 40), _item(rng, "box", *heap, 12)] + small(),
                 [_area_item(rng, LIM["WR_SORT_MAX"] + 1, 200, 40)] + small(),
                 [_item(rng, "stairs", *heap, 3), _item(rng, "frame", *cta, 12)] + small()]
        pal = F64_PALETTES["special"]
    packed = [_pack(t, 760) for t in tiles]
    H, W = max(k.shape[0] for k, _ in packed), max(k.shape[1] for k, _ in packed)
    imgs, mks, masks = [], [], []
    for kindarr, mk in packed:
        pad = ((0, H - kindarr.shape[0]), (0, W - kindarr.shape[1]))
        mask, mk = (np.pad(kindarr, pad) > 0).astype(np.uint8), np.pad(mk, pad)
        masks.append(mask)
        mks.append(mk)
        imgs.append(_values(rng, mask, mk, pal))
    dt = np.uint8 if kind == "u8" else np.float64
    return np.stack(imgs).astype(dt), np.stack(mks), np.stack(masks)


def _hover_maps():
    """fp32 foreground and hv maps of one 300 x 420 tile with two confluent foreground regions cut into several nuclei
    by the hv field: a thick ring (framed box past the ranked arena, area under WR_SORT_MAX: the ranked CTA flood)
    and a solid square past WR_GEN_CAP (the heap flood)"""
    H, W = 300, 420
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
    r = np.hypot(yy - 90, xx - 100)
    ring = (r < 75) & (r >= 50)
    square = (yy >= 100) & (yy < 290) & (xx >= 220) & (xx < 410)
    fore = (ring | square).astype(np.float32)
    centers = [(90 + 62 * np.sin(t), 100 + 62 * np.cos(t)) for t in np.linspace(0, 2 * np.pi, 7)[:-1]]
    centers += [(130 + 60 * i, 250 + 60 * j) for i in range(3) for j in range(3)]
    cy, cx = np.array(centers).T
    near = np.argmin((yy[..., None] - cy) ** 2 + (xx[..., None] - cx) ** 2, axis=-1)
    hv = np.stack([np.clip((xx - cx[near]) / 25.0, -1, 1), np.clip((yy - cy[near]) / 25.0, -1, 1)], -1)
    return fore, (hv * fore[..., None]).astype(np.float32)


# --------------------------------------------------------------------------- CPU: limits, generators, coverage
def test_limits_read_from_the_source(tmp_path):
    for name in DEFINES + F64_CONSTS:
        assert isinstance(LIM[name], int) and LIM[name] > 0, name
    # what the small warp arena takes must fit it, and the classes fit the work lists' WS_MAXCLS counters
    assert class_top(LIM["WP_SMALL_CLS"], LIM["WP_ARENA"], LIM["WS_MAXCLS"]) <= LIM["WP_SMALL_ARENA"]
    assert LIM["SLOTS"] <= LIM["WS_MAXCLS"] and LIM["WR_SORT_SMALL"] < LIM["WR_SORT_MAX"]
    assert LIM["WP_ARENA"] < LIM["WP_GEN_CAP"] and LIM["ARENA"] < LIM["WR_GEN_CAP"]
    with open(SRC, encoding="utf-8") as f:
        text = f.read()
    renamed = tmp_path / "watershed.cu"
    renamed.write_text(text.replace("#define WP_GEN_CAP", "#define WP_GEN_CAP_X"), encoding="utf-8")
    with pytest.raises(AssertionError, match="WP_GEN_CAP"):
        read_limits(str(renamed))


def test_blob_generators_have_the_claimed_geometry():
    for shape in T.BLOB_SHAPES:
        for h, w in [(1, 1), (1, 17), (17, 1), (2, 9), (9, 2), (12, 12), (45, 717), (31, 42)]:
            b = T.blob(shape, h, w)
            host = b == 1
            assert b.shape == (h, w) and host.any(), (shape, h, w)
            lab, n = sk.label(host, connectivity=1, return_num=True)
            assert n == 1, (shape, h, w, "host is one 4-connected blob")
            assert host[0].any() and host[-1].any() and host[:, 0].any() and host[:, -1].any(), (shape, h, w, "box")
            if shape == "stairs":
                assert host.sum() == h + w - 1
            if shape == "holes" and h >= 9 and w >= 9:
                isl, k = sk.label(b == 2, connectivity=1, return_num=True)
                assert k >= 1 and np.bincount(isl.ravel())[1:].tolist() == [9] * k
                assert sk.label(b > 0, connectivity=1).max() == k + 1, "islands do not touch the host"
    for a, w in [(1024, 32), (1025, 32), (1024, 50), (16385, 128)]:
        b = T.area_blob(a, w)
        assert b.sum() == a and b.shape[1] == w and sk.label(b, connectivity=1).max() == 1
    for cells in (1408, 4225, 33792, 33793, 28161):
        for form in ("square", "flat"):
            h, w = T.box_for(cells, form)
            assert (h + 2) * (w + 2) == cells


def _flooded(kind, cases):
    """{case: [Blob]} of the blobs that are flooded (two or more marker labels)"""
    return {n: [b for b in flood_path(mask, kind, mk) if b.labels >= 2] for n, (mask, mk) in cases.items()}


def _at_and_past(blobs, quantity, limit, what):
    """some flooded blob sits exactly at the limit (the largest framed-box size <= it, for cells) and one just past
    it -> (blobs at, blobs past)"""
    at = T.cells_at_most(limit) if quantity == "cells" else limit
    past = T.cells_above(limit) if quantity == "cells" else limit + 1
    a = [b for b in blobs if getattr(b, quantity) == at]
    p = [b for b in blobs if getattr(b, quantity) == past]
    assert a, "%s: no flooded blob with %s == %d" % (what, quantity, at)
    assert p, "%s: no flooded blob with %s == %d" % (what, quantity, past)
    return a, p


def _check_u8_coverage(kind, per_case):
    blobs = [b for v in per_case.values() for b in v]
    A, S = LIM["WP_ARENA"], LIM["WS_MAXCLS"]
    for c in range(S):
        a, p = _at_and_past(blobs, "cells", class_top(c, A, S), "%s class %d" % (kind, c))
        assert {b.cls for b in a} == {c}
        assert {b.cls for b in p} == ({c - 1} if c else {None})
        shapes = {(b.h, b.w, b.area) for b in a}
        assert len(shapes) >= 2, "%s class %d: two shapes at the limit" % (kind, c)
    for name, here, nxt in (("WP_SMALL_ARENA", "u8 warp small", "u8 warp big"), ("WP_ARENA", "u8 warp big", "u8 cta"),
                            ("WP_GEN_CAP", "u8 cta", "u8 global")):
        a, p = _at_and_past(blobs, "cells", LIM[name], kind + " " + name)
        assert {b.path for b in a} == {here} and {b.path for b in p} == {nxt}, (name, {b.path for b in a + p})
        if name != "WP_SMALL_ARENA":
            assert len({(b.h, b.w, b.area) for b in a + p}) >= 3, (kind, name, "shapes")
    rows = [b for b in blobs if b.h == 1]
    for name in ("WP_ARENA", "WP_GEN_CAP"):
        assert any(b.cells == T.cells_at_most(LIM[name]) for b in rows), (kind, name, "one-row blob at the limit")
        assert any(b.cells > LIM[name] and b.cells <= LIM[name] + 3 for b in rows), (kind, name, "one-row past")


def test_u8_cases_reach_every_limit_on_both_sides():
    cases = {}
    for name in U8_CASES:
        img, mk, mask = u8_case(name)
        cases[name] = (np.ones(img.shape, np.uint8) if mask is None else mask, mk)
    per_case = _flooded("u8", cases)
    _check_u8_coverage("u8", per_case)
    cols = [b for b in per_case["columns-four"] if b.w == 1]
    assert any(b.cells == T.cells_at_most(LIM["WP_GEN_CAP"]) for b in cols), "a one-column blob at the CTA slice"
    # markers: 2, 3 and tens per blob; single-marker and marker-less blobs too
    counts = {b.labels for v in per_case.values() for b in v}
    assert {2, 3}.issubset(counts) and max(counts) >= 30
    every = [b for name, (mask, mk) in cases.items() for b in flood_path(mask, "u8", mk)]
    assert {0, 1}.issubset({b.labels for b in every}), "blobs without a marker and with one"
    # blobs touch every image border
    for name in ("classes-four", "cta-four"):
        mask = u8_case(name)[2]
        assert mask[0].any() and mask[-1].any() and mask[:, 0].any() and mask[:, -1].any(), name
    levels = {name: len(np.unique(u8_case(name)[0])) for name in U8_SHEETS}
    assert min(levels.values()) == 2 and max(levels.values()) == 256, levels
    assert all((u8_case(n)[0][u8_case(n)[2] > 0] == 255).any() for n in U8_SHEETS if "top" in n), "level 255 itself"


def test_dist_cases_reach_every_limit_on_both_sides():
    cases = {}
    for name in DIST_CASES:
        mask, _, mk = dist_stages(dist_case(name))
        cases[name] = (mask, mk)
    batch = dist_batch()
    for j in range(len(batch)):
        mask, _, mk = dist_stages(batch[j])
        cases["batch %d" % j] = (mask, mk)
    per_case = _flooded("dist", cases)
    _check_u8_coverage("dist", {k: v for k, v in per_case.items() if not k.startswith("batch")})
    huge = [sum(b.path == "u8 global" for b in per_case["batch %d" % j]) for j in range(len(batch))]
    assert huge[0] == 0 and huge[1] >= 1 and huge[2] == 0 and huge[3] >= 2, huge
    # a huge blob of tile 3 holds flooded (two-peak) islands inside its box
    t3 = per_case["batch 3"]
    holes = [b for b in t3 if b.path == "u8 global"]
    inside = [s for s in t3 if s.path != "u8 global" and any(
        g.y0 < s.y0 and s.y0 + s.h < g.y0 + g.h and g.x0 < s.x0 and s.x0 + s.w < g.x0 + g.w for g in holes)]
    assert len(inside) >= 4, len(inside)


def test_f64_cases_reach_every_limit_on_both_sides():
    cases = {}
    for name in F64_CASES:
        img, mk, mask = f64_case(name)
        cases[name] = (np.ones(img.shape, np.uint8) if mask is None else mask, mk)
    per_case = _flooded("f64", cases)
    blobs = [b for v in per_case.values() for b in v]
    A, S = LIM["ARENA"], LIM["SLOTS"]
    for c in range(S):
        a, p = _at_and_past(blobs, "cells", class_top(c, A, S), "f64 class %d" % c)
        assert {b.cls for b in a} == {c} and {b.cls for b in p} == ({c - 1} if c else {None})
        # one case fills a warp's c + 1 slots with blobs of class c
        assert max(sum(b.cls == c for b in v) for v in per_case.values()) >= c + 1, ("f64 class", c, "slots")
    for name, here, nxt in (("ARENA", "f64 lane", "f64 cta"), ("WR_GEN_CAP", "f64 cta", "f64 heap")):
        a, p = _at_and_past(blobs, "cells", LIM[name], "f64 " + name)
        assert here in {b.path for b in a} and {b.path for b in p} == {nxt}, (name, {b.path for b in a + p})
    for name, (r_at, r_past) in (("WR_SORT_SMALL", ("rank small", "rank large")), ("WR_SORT_MAX", ("rank large", None))):
        a, p = _at_and_past(blobs, "area", LIM[name], "f64 " + name)
        assert {b.rank for b in a} == {r_at} and {b.rank for b in p} == {r_past}, name
        assert len({(b.h, b.w) for b in a}) >= 2 and len({(b.h, b.w) for b in p}) >= 2, (name, "two shapes")
    assert any(b.rank == "rank small" and b.path == "f64 heap" for b in blobs), "ranked, then sent to the heap"
    assert any(b.rank == "rank large" and b.path == "f64 cta" for b in blobs)
    # runs of equal values (-0.0 == +0.0) longer than a chunk of the rank scan, in blobs of both ranking kernels
    longest = {"rank small": 0, "rank large": 0}
    for name in F64_CASES:
        img, mk, mask = f64_case(name)
        lab = sk.label(np.ones(img.shape, np.uint8) if mask is None else mask, connectivity=1)
        flat, ids = img.ravel() + 0.0, lab.ravel()
        order = np.lexsort((flat, ids))
        key_id, key_v = ids[order], flat[order]
        starts = np.flatnonzero(np.r_[True, (key_id[1:] != key_id[:-1]) | (key_v[1:] != key_v[:-1])])
        runs = np.diff(np.r_[starts, len(order)])
        run_of = np.zeros(lab.max() + 1, np.int64)
        np.maximum.at(run_of, key_id[starts], runs)
        for i, b in enumerate(flood_path(lab > 0, "f64", mk), 1):
            if b.rank in longest and b.labels >= 2:
                longest[b.rank] = max(longest[b.rank], int(run_of[i]))
    assert longest["rank small"] > LIM["RANK_CHUNK_SMALL"] and longest["rank large"] > LIM["RANK_CHUNK_LARGE"], longest
    for name in F64_SHEETS:         # -0.0 seeds next to +0.0 seeds, one-ulp neighbours, infinities, subnormals
        img, mk, mask = f64_case(name)
        z = img[(mk != 0) & (img == 0)]
        assert np.signbit(z).any() and (~np.signbit(z)).any(), name
        if "special" in name:
            v = set(np.unique(img).tolist())
            assert {-np.inf, np.inf, 5e-324, 1.0, np.nextafter(1.0, 2.0), np.nextafter(1.0, 0.0)} <= v, name


def test_batches_mix_every_flood():
    for kind in ("u8", "f64"):
        imgs, mks, masks = mixed_batch(kind)
        paths = [{b.path for b in flood_path(masks[j], kind, mks[j]) if b.labels >= 2} for j in range(len(imgs))]
        far = "u8 global" if kind == "u8" else "f64 heap"
        cta = "u8 cta" if kind == "u8" else "f64 cta"
        assert [far in p for p in paths] == [False, True, True, True], (kind, paths)
        assert sum(cta in p for p in paths) >= 2, (kind, paths)
        assert all(p & {"u8 warp big", "u8 warp small", "f64 lane"} for p in paths), (kind, paths)


@functools.lru_cache(maxsize=None)
def _hover_oracle():
    fore, hv = _hover_maps()
    return fore, hv, opp.hover_post_proc(fore, hv)


def test_hover_case_reaches_the_ranked_cta_and_heap_floods():
    _, _, (_, dbg) = _hover_oracle()
    paths = {b.path for b in flood_path(dbg["blb"], "f64", dbg["marker"]) if b.labels >= 2}
    assert {"f64 cta", "f64 heap"} <= paths, paths


# --------------------------------------------------------------------------- GPU: every output against the oracle
def _diff(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, "%s: shape %r vs %r" % (what, a.shape, b.shape)
    bad = np.argwhere(a != b)
    assert len(bad) == 0, "%s: %d mismatching elements, first at %r: got %r want %r" % (
        what, len(bad), tuple(bad[0]), a[tuple(bad[0])], b[tuple(bad[0])])


@gpu
@pytest.mark.parametrize("name", U8_CASES)
def test_u8_forest_mode(name):
    img, mk, mask = u8_case(name)
    _diff(ops.watershed(img, mk, mask), sk.watershed(img, mk, mask), "u8 " + name)


@gpu
@pytest.mark.parametrize("name", DIST_CASES)
def test_dist_mask_mode(name):
    d = dist_case(name)
    mask, inv, want_mk = dist_stages(d)
    got, mk, ws = ops.postproc_dist(d, debug=True)
    _diff(mk, want_mk, name + ": markers")
    _diff(ws, sk.watershed(inv, want_mk, mask=mask), name + ": raw flood")
    _diff(got, opp.dist_postprocess(None, d, literal=False)[1], name + ": instances")


@gpu
def test_dist_huge_blobs_in_later_tiles():
    """the huge-tile list, k_huge_clean and listed_geom: global floods in tiles 1 and 3 of four, two in one tile, one
    whose holes hold two-peak islands; the batch in two orders"""
    d = dist_batch()
    for order in ([0, 1, 2, 3], [3, 0, 2, 1]):
        got, mk, ws = ops.postproc_dist(np.ascontiguousarray(d[order]), debug=True)
        for j, t in enumerate(order):
            mask, inv, want_mk = dist_stages(d[t])
            what = "dist batch tile %d at %d" % (t, j)
            _diff(mk[j], want_mk, what + ": markers")
            _diff(ws[j], sk.watershed(inv, want_mk, mask=mask), what + ": raw flood")
            _diff(got[j], opp.dist_postprocess(None, d[t], literal=False)[1], what + ": instances")


@gpu
@pytest.mark.parametrize("name", F64_CASES)
def test_f64_forest_mode(name):
    img, mk, mask = f64_case(name)
    _diff(ops.watershed(img, mk, mask), sk.watershed(img, mk, mask), "f64 " + name)


@gpu
@pytest.mark.parametrize("kind", ["u8", "f64"])
def test_mixed_batch_equals_single_tiles(kind):
    """a batch whose tiles take every flood (global / heap floods in three tiles: per-tile arena slices) equals the
    single-tile calls and the oracle, in two orders, from host arrays and from CUDA tensors"""
    import torch
    imgs, mks, masks = mixed_batch(kind)
    want = [sk.watershed(imgs[j], mks[j], masks[j]) for j in range(len(imgs))]
    for j in range(len(imgs)):
        _diff(ops.watershed(imgs[j], mks[j], masks[j]), want[j], "%s single tile %d" % (kind, j))
    for order in ([0, 1, 2, 3], [2, 3, 1, 0]):
        args = [np.ascontiguousarray(a[order]) for a in (imgs, mks, masks)]
        got = ops.watershed(*args)
        dev = ops.watershed(*[torch.from_numpy(a).cuda() for a in args])
        assert dev.is_cuda
        for j, t in enumerate(order):
            _diff(got[j], want[t], "%s batch tile %d at %d" % (kind, t, j))
            _diff(dev[j].cpu().numpy(), want[t], "%s CUDA batch tile %d at %d" % (kind, t, j))


@gpu
def test_hover_ranked_cta_and_heap():
    fore, hv, (want, dbg) = _hover_oracle()
    inst, blb, dist, mk = ops.postproc_hover(fore, hv, debug=True)
    _diff(blb, dbg["blb"], "hover blb")
    _diff(mk, dbg["marker"], "hover markers")
    _diff(np.asarray(dist).view(np.uint64), dbg["dist"].view(np.uint64), "hover flooded image")
    _diff(inst, want, "hover inst")
