"""HoVer-Net post-process at every fx of the reference's hover_post_proc(fore_map, hv_map, fx, scale_factor): Sobel
ksize int(20 * fx + 1) from 1 to 31 and marker obj_size ceil(10 * fx^2), compared bit for bit with the CPU oracle, which
calls cv2 and scipy as the reference does."""
import functools
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import tiseg_b200  # noqa: E402,F401
from tiseg_b200 import _lib, ops, segmentors, synth  # noqa: E402
from oracle import postprocess as opp  # noqa: E402
from test_gpu_half_inputs import HALF, _rounded, _same  # noqa: E402

FXS = [0, 0.02, 0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9, 1.1, 1.2, 1.3, 1.4, 1.5]
SHAPES = [(64, 100), (250, 131), (7, 9), (1, 40), (33, 1), (500, 517)]


@functools.lru_cache(maxsize=None)
def _maps(H, W, idx):
    """(fore [H,W], hv [H,W,2]) fp32, cropped from a tile of at least 40 x 40"""
    t = synth.tile_hover(3, idx, H=max(H, 40), W=max(W, 40))
    return np.ascontiguousarray(t["fore_map"][:H, :W]), np.ascontiguousarray(t["hv_map"][:H, :W])


def _bits(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, "%s: shape %r vs %r" % (what, a.shape, b.shape)
    if a.dtype.kind == "f":
        assert a.dtype == b.dtype, what
        a, b = a.view("u%d" % a.itemsize), b.view("u%d" % b.itemsize)
    bad = np.argwhere(a != b)
    assert len(bad) == 0, "%s: %d of %d elements differ, first at %r" % (what, len(bad), a.size, tuple(bad[0]))


def _check_oracle(fore, hv, fx, sf, what):
    want, dbg = opp.hover_post_proc(fore, hv, fx=fx, scale_factor=sf)
    inst, blb, dist, mk = ops.postproc_hover(fore, hv, scale_factor=sf, debug=True, fx=fx)
    _bits(blb, dbg["blb"], what + " blb")
    _bits(mk, dbg["marker"], what + " markers")
    _bits(dist, dbg["dist"], what + " flooded image (fp64)")
    _bits(inst, want, what + " inst")
    return inst


@pytest.mark.parametrize("fx", FXS)
def test_every_kernel_size_equals_oracle(fx):
    """ksize 1 (fx 0, 0.02: derivative [-1, 0, 1] without smoothing; fx 0 also drops no marker) to 31 (fx 1.5), at
    scale 1 and 2; 7 x 9, 1 x 40 and 33 x 1 are smaller than the kernel radius, so the border reflects repeatedly"""
    for i, (H, W) in enumerate(SHAPES):
        fore, hv = _maps(H, W, i)
        for sf in (1, 2):
            _check_oracle(fore, hv, fx, sf, "fx %g scale %d %dx%d" % (fx, sf, H, W))


@pytest.mark.parametrize("fx", [0.5, 1.5])
def test_full_tiles_batched(fx):
    tiles = [synth.tile_hover(3, 20 + j) for j in range(2)]
    fore, hv = np.stack([t["fore_map"] for t in tiles]), np.stack([t["hv_map"] for t in tiles])
    got = ops.postproc_hover(fore, hv, debug=True, fx=fx)
    for j in range(2):
        want, dbg = opp.hover_post_proc(tiles[j]["fore_map"], tiles[j]["hv_map"], fx=fx)
        for g, w, name in zip(got, (want, dbg["blb"], dbg["dist"], dbg["marker"]), ("inst", "blb", "dist", "markers")):
            _bits(g[j], w, "fx %g 1000^2 tile %d %s" % (fx, j, name))
        assert got[0][j].max() > 3


@pytest.mark.parametrize("fx", [0.3, 0.5, 1.3])
def test_batch_equals_single_calls_and_host_equals_device(fx):
    import torch
    maps = [_maps(250, 131, 30 + j) for j in range(3)]
    fore, hv = np.stack([m[0] for m in maps]), np.stack([m[1] for m in maps])
    for sf in (1, 2):
        batch = ops.postproc_hover(fore, hv, scale_factor=sf, debug=True, fx=fx)
        for j in range(3):
            single = ops.postproc_hover(fore[j], hv[j], scale_factor=sf, debug=True, fx=fx)
            for b, s in zip(batch, single):
                _bits(b[j], s, "fx %g scale %d batch entry %d" % (fx, sf, j))
        dev = ops.postproc_hover(torch.from_numpy(fore).cuda(), torch.from_numpy(hv).cuda(), scale_factor=sf, debug=True, fx=fx)
        _same(tuple(x.cpu().numpy() for x in dev), batch, "fx %g scale %d CUDA tensors vs numpy" % (fx, sf))


@pytest.mark.parametrize("dtype", HALF)
def test_half_inputs_equal_upcast(dtype):
    """the resize or the normalise step reads the half inputs; the Sobel kernels see fp32 either way"""
    for H, W, n in ((256, 256, 2), (200, 333, 1)):
        ts = [synth.tile_hover(3, 50 + i, H=H, W=W) for i in range(n)]
        fh, fr = _rounded(np.stack([t["fore_map"] for t in ts]), dtype)
        hh, hr = _rounded(np.stack([t["hv_map"] for t in ts]), dtype)
        for fx in (0.02, 0.5, 1.5):
            for sf in (1, 2):
                _same(ops.postproc_hover(fh, hh, scale_factor=sf, debug=True, fx=fx),
                      ops.postproc_hover(fr, hr, scale_factor=sf, debug=True, fx=fx),
                      "postproc_hover %s %dx%d fx %g scale %d" % (dtype, H, W, fx, sf))


def _call(name, fore, hv, sf, *extra):
    N, H, W = fore.shape
    inst = np.empty((N, H, W), np.int32)
    blb = np.empty((N, H * sf, W * sf), np.uint8)
    dist = np.empty((N, H * sf, W * sf), np.float64)
    mk = np.empty((N, H * sf, W * sf), np.int32)
    p = _lib.ptr
    _lib.get_ctx().call(name, _lib.DTYPE_F32, p(fore), p(hv), N, H, W, sf, *extra, p(inst), p(blb), p(dist), p(mk))
    return inst, blb, dist, mk


def test_fx_1_is_the_typed_entry():
    maps = [_maps(250, 131, 40 + j) for j in range(2)]
    fore, hv = np.stack([m[0] for m in maps]), np.stack([m[1] for m in maps])
    for sf in (1, 2):
        typed = _call("tiseg_postproc_hover_typed", fore, hv, sf)
        _same(_call("tiseg_postproc_hover_ex", fore, hv, sf, 21, 10), typed, "ex(21, 10) scale %d" % sf)
        _same(ops.postproc_hover(fore, hv, scale_factor=sf, debug=True, fx=1), typed, "fx=1 scale %d" % sf)
        _same(ops.postproc_hover(fore, hv, scale_factor=sf, debug=True), typed, "default fx scale %d" % sf)


def test_reference_api_hover_post_proc():
    fore, hv = _maps(500, 517, 5)
    want, _ = opp.hover_post_proc(fore, hv, fx=0.5)
    _bits(segmentors.HoverNet(3).hover_post_proc(fore, hv, fx=0.5), want, "HoverNet.hover_post_proc fx 0.5")
    want, _ = opp.hover_post_proc(fore, hv, fx=1.2, scale_factor=2)
    _bits(segmentors.HoverNet(3).hover_post_proc(fore, hv, fx=1.2, scale_factor=2), want, "fx 1.2 scale 2")


@pytest.mark.parametrize("fx,ksize", [(0.25, 6), (0.75, 16), (1.6, 33), (-0.5, -9), (-0.02, 0)])
def test_refused_fx(fx, ksize):
    fore, hv = _maps(64, 100, 6)
    with pytest.raises(_lib.TisegError, match=r"status 2\).*ksize.*got %d\b" % ksize):
        ops.postproc_hover(fore, hv, fx=fx)
    with pytest.raises(_lib.TisegError, match=r"status 2\)"):
        segmentors.HoverNet(3).hover_post_proc(fore, hv, fx=fx)


def test_refused_c_arguments():
    fore, hv = [a[None] for a in _maps(64, 100, 6)]
    for sf, ksize, obj_size, what in ((1, 2, 3, "ksize.*got 2"), (1, -1, 3, "ksize.*got -1"), (1, 33, 3, "ksize.*got 33"),
                                      (1, 11, -1, "obj_size.*got -1"), (3, 11, 3, "scale_factor.*got 3")):
        with pytest.raises(_lib.TisegError, match=r"status 2\).*" + what):
            _call("tiseg_postproc_hover_ex", fore, hv, sf, ksize, obj_size)


@pytest.mark.parametrize("fx,rd,rs", [(0, 1, 0), (0.5, 5, 5), (1, 10, 10), (1.5, 15, 15)])
def test_sobel_kernels_of_each_radius_run(fx, rd, rs):
    """the host dispatch launches the kernels of the ksize's tap radii, under names bench.py maps by prefix"""
    fore, hv = _maps(64, 100, 7)
    ctx = _lib.get_ctx()
    ops.postproc_hover(fore, hv, fx=fx)                       # modules loaded
    ctx.timing(True)
    try:
        ops.postproc_hover(fore, hv, fx=fx)
        ctx.synchronize()
        names = {k for k in ctx.timing_report() if k.startswith("k_sobel")}
    finally:
        ctx.timing(False)
    assert names == {"k_sobel_row<true, %d>" % rd, "k_sobel_col<false, %d>" % rs, "k_sobel_row<false, %d>" % rs,
                     "k_sobel_col<true, %d>" % rd}, names
