"""The arithmetic the HoVer-Net Sobel kernels (csrc/hover.cu, k_sobel_row / k_sobel_col) implement for every kernel size
hover_post_proc's fx can give, restated in numpy and checked against cv2.Sobel bit for bit.  No GPU needed.

Recipe of cv2.Sobel(x32, CV_64F, dx, dy, ksize) with the kernels of cv2.getDerivKernels:
  row pass     sequential taps in fp64, k[0] * x[-r] + k[1] * x[-r + 1] + ...
  column pass  centre tap (0 for the derivative), then k[r + t] * (R[+t] +/- R[-t]) for t = 1..r, multiply and add
               rounded separately (no FMA)
  border       BORDER_REFLECT_101, reflected again until the index is inside (images smaller than the radius)
ksize 1 is the derivative [-1, 0, 1] with the smoothing [1]; every other ksize has radius ksize // 2 in both passes."""
import math

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

KSIZES = list(range(1, 32, 2))
SHAPES = [(1, 37), (37, 1), (5, 7), (12, 9), (33, 64), (64, 33), (128, 96), (97, 131)]


def _binomial(n):
    b = np.array([1.0])
    for _ in range(n):
        b = np.convolve(b, [1.0, 1.0])
    return b


def kernels(ksize):
    """-> (derivative, smoothing) taps, applied as correlation: k[t] multiplies x[i + t - r]"""
    if ksize == 1:
        return np.array([-1.0, 0.0, 1.0]), np.array([1.0])
    return np.convolve(_binomial(ksize - 2), [-1.0, 1.0]), _binomial(ksize - 1)


def _reflect101(i, n):
    if n == 1:
        return 0
    while i < 0 or i >= n:
        i = -i if i < 0 else 2 * n - 2 - i
    return i


def _taps(n, r):
    """[n, 2r+1] source indices of every output along an axis of length n"""
    return np.array([[_reflect101(j + t - r, n) for t in range(2 * r + 1)] for j in range(n)], dtype=np.int64)


def sobel(x32, dx, dy, ksize):
    """cv2.Sobel(x32, CV_64F, dx, dy, ksize) for (dx, dy) in {(1, 0), (0, 1)}"""
    d, sm = kernels(ksize)
    kx, ky = (d, sm) if dx == 1 else (sm, d)
    H, W = x32.shape
    x = x32.astype(np.float64)
    rx, ry = len(kx) // 2, len(ky) // 2
    ix = _taps(W, rx)
    row = kx[0] * x[:, ix[:, 0]]
    for t in range(1, 2 * rx + 1):
        row = row + kx[t] * x[:, ix[:, t]]
    iy = _taps(H, ry)
    acc = np.zeros_like(row) if dy == 1 else ky[ry] * row[iy[:, ry]]
    for t in range(1, ry + 1):
        a, b = row[iy[:, ry + t]], row[iy[:, ry - t]]
        acc = acc + ky[ry + t] * ((a - b) if dy == 1 else (a + b))
    return acc


def _same_bits(got, want, what):
    assert got.dtype == want.dtype == np.float64 and got.shape == want.shape, what
    bad = np.argwhere(got.view(np.uint64) != want.view(np.uint64))
    assert len(bad) == 0, "%s: %d of %d differ, first at %r: %r vs %r" % (
        what, len(bad), got.size, tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])])


@pytest.mark.parametrize("ksize", KSIZES)
def test_kernels_are_cv2_deriv_kernels(ksize):
    d, sm = kernels(ksize)
    kd, ks = cv2.getDerivKernels(1, 0, ksize, ktype=cv2.CV_64F)
    assert np.array_equal(d, kd.ravel()) and np.array_equal(sm, ks.ravel())
    assert sm.max() < 2 ** 28                         # row products of fp32 sources are exact in fp64


@pytest.mark.parametrize("ksize", KSIZES)
def test_recipe_equals_cv2_sobel_random(ksize):
    rng = np.random.default_rng(ksize)
    for H, W in SHAPES:
        x = rng.random((H, W)).astype(np.float32)
        for dx, dy in ((1, 0), (0, 1)):
            _same_bits(sobel(x, dx, dy, ksize), cv2.Sobel(x, cv2.CV_64F, dx, dy, ksize=ksize),
                       "ksize %d %dx%d d=(%d,%d)" % (ksize, H, W, dx, dy))


@pytest.mark.parametrize("ksize", KSIZES)
def test_recipe_equals_cv2_sobel_on_normalised_hv_maps(ksize):
    """the inputs hover_post_proc gives cv2.Sobel: cv2.normalize'd channels of synthetic HV maps"""
    from tiseg_b200 import synth
    for j, (H, W) in enumerate(((256, 256), (200, 333))):
        hv = synth.tile_hover(3, 70 + j, H=H, W=W)["hv_map"]
        for ch, (dx, dy) in enumerate(((1, 0), (0, 1))):
            n = cv2.normalize(hv[:, :, ch], None, alpha=0, beta=1, norm_type=cv2.NORM_MINMAX, dtype=cv2.CV_32F)
            _same_bits(sobel(n, dx, dy, ksize), cv2.Sobel(n, cv2.CV_64F, dx, dy, ksize=ksize),
                       "hv ksize %d %dx%d channel %d" % (ksize, H, W, ch))


@pytest.mark.parametrize("ksize", [2, 6, 16, 33])
def test_cv2_refuses_even_and_oversized_ksize(ksize):
    x = np.zeros((40, 40), np.float32)
    with pytest.raises(cv2.error):
        cv2.Sobel(x, cv2.CV_64F, 1, 0, ksize=ksize)


# fx -> (ksize, obj_size) of the reference's hover_post_proc
FX_TABLE = {0.02: (1, 1), 0.1: (3, 1), 0.2: (5, 1), 0.3: (7, 1), 0.4: (9, 2), 0.5: (11, 3), 0.6: (13, 4), 0.7: (15, 5),
            0.8: (17, 7), 0.9: (19, 9), 1.0: (21, 10), 1.1: (23, 13), 1.2: (25, 15), 1.3: (27, 17), 1.4: (29, 20),
            1.5: (31, 23), 0: (1, 0)}


def test_fx_table_matches_reference_expressions():
    for fx, want in FX_TABLE.items():
        assert (int((20 * fx) + 1), math.ceil(10 * (fx ** 2))) == want, fx
    # the fx values whose ksize cv2.Sobel refuses
    for fx in (0.05, 0.15, 0.25, 0.75):
        assert int((20 * fx) + 1) % 2 == 0, fx
    assert int((20 * 1.6) + 1) == 33
