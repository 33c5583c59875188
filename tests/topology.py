"""numpy generators of adversarial topologies for the connected-component labellers: long union chains that cross many
tiles, diagonal-only contacts, and contacts placed exactly on the word, tile-column and tile-row edges of the bit-plane
labeller (csrc/bitccl.cuh: tiles of 32 rows x 8 words of 32 pixels).  tests/test_gpu_bitccl.py checks each generator's
claimed topology on the CPU.  TEST INFRASTRUCTURE ONLY."""
import numpy as np

WORD = 32            # pixels per bit-plane word
TILE_W = 256         # tile width in pixels (BT_TWW words)
TILE_H = 32          # tile height in rows (BT_TH)


def spiral(H, W):
    """One-pixel-wide rectangular spiral with one-pixel gaps between its turns, walking inwards clockwise from (0, 0):
    a single 4-connected simple path over about half the pixels.  A step is taken only into a pixel none of whose
    other 4-neighbours is already on the path, which keeps the path one pixel wide and the gaps open."""
    s = np.zeros((H, W), np.uint8)
    dirs = ((0, 1), (1, 0), (0, -1), (-1, 0))
    y = x = d = 0
    s[0, 0] = 1
    turned = False

    def free(ny, nx, fy, fx):
        if not (0 <= ny < H and 0 <= nx < W) or s[ny, nx]:
            return False
        for qy, qx in ((ny - 1, nx), (ny + 1, nx), (ny, nx - 1), (ny, nx + 1)):
            if (qy, qx) != (fy, fx) and 0 <= qy < H and 0 <= qx < W and s[qy, qx]:
                return False
        return True

    while True:
        dy, dx = dirs[d]
        if free(y + dy, x + dx, y, x):
            y, x = y + dy, x + dx
            s[y, x] = 1
            turned = False
        elif turned:
            return s
        else:
            d, turned = (d + 1) % 4, True


def comb(H, W, pitch=2, width=1):
    """Vertical teeth `width` pixels wide every `pitch` columns, over every row, joined by ONE spine along the last row:
    one 4-connected component whose teeth meet only at the bottom, so every tooth's union chain crosses every tile row
    and the teeth of different tile columns meet only through the spine."""
    c = np.zeros((H, W), np.uint8)
    for k in range(width):
        c[:, k::pitch] = 1
    c[H - 1, :] = 1
    return c


def checkerboard(H, W, a=1, b=2, block=1):
    """Two ids in a checkerboard of `block` x `block` squares: squares of one id touch only at their corners, so each id
    is ONE 8-connected component (H, W > block) and one 4-connected component per square."""
    yy, xx = np.indices((H, W))
    return np.where(((yy // block) + (xx // block)) % 2 == 0, a, b).astype(np.int32)


def staircase(H, W, pitch=4, anti=False):
    """Diagonal lines every `pitch` pixels: x - y = const (down-right, the above-left contacts), or x + y = const with
    ``anti`` (down-left, the above-right contacts).  Every pixel is its own 4-connected component; each line is one
    8-connected component."""
    yy, xx = np.indices((H, W))
    return (((xx + yy) if anti else (xx - yy)) % pitch == 0).astype(np.uint8)


def percolation(H, W, p, seed):
    """Random mask with density p: p = 0.41 sits near the 8-connected percolation threshold (0.407), 0.59 near the
    4-connected one (0.593), where component sizes are spread over every scale."""
    return (np.random.default_rng(seed).random((H, W)) < p).astype(np.uint8)


BOUNDARIES = ("word", "tilecol", "tilerow", "corner")


def boundary_point(kind, k=1):
    """(y, x) of the pixel just past the k-th boundary of `kind`: a contact between (y - 1, x - 1) and (y, x), or
    between (y - 1, x) and (y, x - 1), crosses
      word     x = 32k - 1 | 32k        (inside a tile, between two words; y inside a tile row)
      tilecol  x = 256k - 1 | 256k      (between two tile columns; y inside a tile row)
      tilerow  y = 32k - 1 | 32k        (between two tile rows; x inside a word)
      corner   both tile edges at once  (y = 32k, x = 256k)."""
    if kind == "word":
        assert k % (TILE_W // WORD), "word edge %d is a tile-column edge" % k
        return 20, WORD * k
    if kind == "tilecol":
        return 20, TILE_W * k
    if kind == "tilerow":
        return TILE_H * k, 100
    if kind == "corner":
        return TILE_H * k, TILE_W * k
    raise ValueError(kind)


def diagonal_contact(kind, k=1, anti=False):
    """The two pixels of a diagonal-only contact across the named boundary: ((upper y, x), (lower y, x)).  Down-right
    ((y - 1, x - 1), (y, x)) by default, down-left ((y - 1, x), (y, x - 1)) with ``anti``."""
    y, x = boundary_point(kind, k)
    return ((y - 1, x), (y, x - 1)) if anti else ((y - 1, x - 1), (y, x))


# --------------------------------------------------------------------------- single blobs with an exact bounding box
# for the size limits of the watershed's floods (csrc/watershed.cu), which pick a flood by the blob's bounding box framed
# by one pixel, (h + 2) (w + 2) cells, and by its area.  tests/test_gpu_watershed.py checks their claims on the CPU.
BLOB_SHAPES = ("box", "frame", "serpentine", "stairs", "holes")


def framed_boxes(cells):
    """every (h, w) whose framed box (h + 2) (w + 2) holds exactly `cells` cells, from one row to one column"""
    return [(d - 2, cells // d - 2) for d in range(3, cells // 3 + 1) if cells % d == 0]


def cells_at_most(limit):
    """the largest framed-box size <= limit (a prime has no box)"""
    c = limit
    while not framed_boxes(c):
        c -= 1
    return c


def cells_above(limit):
    """the smallest framed-box size > limit"""
    c = limit + 1
    while not framed_boxes(c):
        c += 1
    return c


def box_for(cells, form="square"):
    """(h, w) with (h + 2) (w + 2) == cells: "square" (closest to square), "flat" (closest to h : w = 1 : 8), "row"
    (h = 1) or "col" (w = 1)"""
    boxes = framed_boxes(cells)
    assert boxes, "no framed box holds %d cells" % cells
    if form in ("row", "col"):
        hw = [b for b in boxes if (b[0] if form == "row" else b[1]) == 1]
        assert hw, "%d cells: no %s of them" % (cells, form)
        return hw[0]
    ratio = 1.0 if form == "square" else 0.125
    return min(boxes, key=lambda b: (abs(np.log(b[0] / b[1] / ratio)), b[0]))


def blob(shape, h, w):
    """One 4-connected blob whose bounding box is exactly h x w (uint8, 1 on the blob):
      box         solid
      frame       a one-pixel frame (solid when h or w <= 2)
      serpentine  full rows every other row, joined at alternate ends: about half the box
      stairs      a 4-connected monotone staircase from corner to corner: h + w - 1 pixels
      holes       solid with 5 x 5 holes every 8 pixels, each holding a 3 x 3 island (marked 2: a blob of its own,
                  one pixel clear of the host all round)"""
    s = np.zeros((h, w), np.uint8)
    if shape == "box":
        s[:] = 1
    elif shape == "frame":
        s[:] = 1
        if h > 2 and w > 2:
            s[1:-1, 1:-1] = 0
    elif shape == "serpentine":
        s[0::2, :] = 1
        for y in range(1, h, 2):
            s[y, w - 1 if (y // 2) % 2 == 0 else 0] = 1
    elif shape == "stairs":
        y = x = 0
        s[0, 0] = 1
        while (y, x) != (h - 1, w - 1):
            if x < w - 1 and (y == h - 1 or (x + 1) * h <= (y + 1) * w):
                x += 1
            else:
                y += 1
            s[y, x] = 1
    elif shape == "holes":
        s[:] = 1
        for y0 in range(2, h - 6, 8):
            for x0 in range(2, w - 6, 8):
                s[y0:y0 + 5, x0:x0 + 5] = 0
                s[y0 + 1:y0 + 4, x0 + 1:x0 + 4] = 2
    else:
        raise ValueError(shape)
    return s


def area_blob(area, w):
    """`area` pixels filled in raster order over rows of width w: full rows and one partial row (bounding box
    ceil(area / w) x w for area >= w)"""
    s = np.zeros(((area + w - 1) // w, w), np.uint8)
    s.ravel()[:area] = 1
    return s
