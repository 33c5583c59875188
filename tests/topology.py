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
