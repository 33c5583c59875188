"""ctypes loader of ``libtiseg_b200.so`` (the C-ABI CUDA library, ``include/tiseg_b200.h``).

There is no CPU fallback: ``get_ctx()`` raises if the library is missing or no CUDA device is
present, and every op goes through it.
"""
import ctypes
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libtiseg_b200.so")

_vp, _i, _ll = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong

# name -> argtypes (every function returns int unless listed in _RESTYPE)
SIGNATURES = {
    "tiseg_create": [ctypes.POINTER(_vp), _i],
    "tiseg_destroy": [_vp],
    "tiseg_set_stream": [_vp, _vp],
    "tiseg_synchronize": [_vp],
    "tiseg_last_error": [],
    "tiseg_launch_count": [_vp],
    "tiseg_version": [],
    "tiseg_build_hash": [],
    "tiseg_timing_enable": [_vp, _i],
    "tiseg_timing_report": [_vp, ctypes.c_char_p, _i],
    "tiseg_softmax_argmax_typed": [_vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp],
    "tiseg_tta_input_elems": [_i, _i, _i, _i, _vp, _i, _i],
    "tiseg_softmax_argmax_tta_typed": [_vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp],
    "tiseg_tta_mean_typed": [_vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp],
    "tiseg_ddm_enhance": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i],
    "tiseg_mtcdnet_refine_typed": [_vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "tiseg_pair_metrics_bin_iou": [_vp, _vp, _vp, _i, _i, _i, ctypes.c_double, _vp, _vp],
    "tiseg_pair_metrics_bin_u16gt": [_vp, _vp, _vp, _i, _i, _i, ctypes.c_double, _vp, _vp],
    "tiseg_label": [_vp, _vp, _i, _i, _i, ctypes.c_int32, _i, _vp, _vp],
    "tiseg_label_u8": [_vp, _vp, _i, _i, _i, ctypes.c_int32, _i, _vp, _vp],
    "tiseg_re_instance": [_vp, _vp, _i, _i, _i, _vp, _vp],
    "tiseg_fill_holes": [_vp, _vp, _i, _i, _i, _vp],
    "tiseg_remove_small_objects": [_vp, _vp, _i, _i, _i, _i, _i, _vp],
    "tiseg_remove_small_labels": [_vp, _vp, _i, _i, _i, _i, _vp],
    "tiseg_dilate_labels": [_vp, _vp, _i, _i, _i, _i, _i, _vp],
    "tiseg_erode_labels": [_vp, _vp, _i, _i, _i, _i, _i, _vp],
    "tiseg_postproc_unet": [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp],
    "tiseg_watershed_u8": [_vp, _vp, _vp, _vp, _i, _i, _i, _vp],
    "tiseg_watershed_f64": [_vp, _vp, _vp, _vp, _i, _i, _i, _vp],
    "tiseg_postproc_dist_lambda_typed": [_vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp],
    "tiseg_reconstruction_erosion_u8": [_vp, _vp, _vp, _i, _i, _i, _vp],
    "tiseg_postproc_hover_ex": [_vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp],
    "tiseg_ddm": [_vp, _vp, _i, _i, _i, _vp],
    "tiseg_cdnet_refine_typed": [_vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp],
    "tiseg_align_foreground": [_vp, _vp, _vp, _i, _i, _i, _i],
    "tiseg_postproc_multitask": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp],
    "tiseg_pair_metrics_multiclass": [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp],
    "tiseg_sem_counts": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp],
    "tiseg_assign_sem_class": [_vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "tiseg_mudslide_watershed": [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp],
    "tiseg_gen_hv_map": [_vp, _vp, _i, _i, _i, _vp],
    "tiseg_instance_distance_map": [_vp, _vp, _i, _i, _i, _i, _vp],
    "tiseg_fix_inst": [_vp, _vp, _i, _i, _i, _vp],
    "tiseg_unet_weight_map": [_vp, _vp, _i, _i, _i, ctypes.c_double, ctypes.c_double, _vp, _vp],
    "tiseg_direction_labels": [_vp, _vp, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp],
    "tiseg_bound_label": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp],
    "tiseg_distance_transform_edt": [_vp, _vp, _i, _i, _i, _vp],
    "tiseg_distance_transform_cdt": [_vp, _vp, _i, _i, _i, _vp],
}
_RESTYPE = {"tiseg_last_error": ctypes.c_char_p, "tiseg_build_hash": ctypes.c_char_p, "tiseg_launch_count": _ll, "tiseg_tta_input_elems": _ll}

_lib = None
_lock = threading.Lock()
_ctxs = {}


class TisegError(RuntimeError):
    pass


def _check_fresh(lib):
    """The .so is git-ignored but travels with repo snapshots: refuse one that was not built from the sources beside it."""
    if not os.path.isdir(os.path.join(_HERE, "csrc")) or os.environ.get("TISEG_ALLOW_STALE"):
        return
    import importlib.util
    spec = importlib.util.spec_from_file_location("_tiseg_build", os.path.join(_HERE, "build.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    have, want = (lib.tiseg_build_hash() or b"").decode(), b.source_hash()
    if have != want:
        raise TisegError("libtiseg_b200.so is stale (built from %s, sources are %s): run "
                         "`python tissue-image-segmentation_b200/build.py`" % (have, want))


def load():
    """dlopen the library and bind every declared symbol (no CUDA call is made)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(SO_PATH):
                raise TisegError(
                    "libtiseg_b200.so is not built (run `python tissue-image-segmentation_b200/build.py`); "
                    "tiseg_b200 has no CPU fallback")
            lib = ctypes.CDLL(SO_PATH)
            for name, argtypes in SIGNATURES.items():
                fn = getattr(lib, name)           # AttributeError if a declared symbol is missing
                fn.argtypes = argtypes
                fn.restype = _RESTYPE.get(name, _i)
            _check_fresh(lib)
            _lib = lib
    return _lib


def last_error():
    return (load().tiseg_last_error() or b"").decode("utf-8", "replace")


def check(status, what):
    if status != 0:
        raise TisegError("%s failed (status %d): %s" % (what, status, last_error()))


class Context:
    """One per (process, device): owns the workspace arena and the stream binding."""

    def __init__(self, device=0):
        lib = load()
        h = _vp()
        check(lib.tiseg_create(ctypes.byref(h), int(device)), "tiseg_create")
        self.handle = h
        self.device = int(device)
        self.lib = lib

    def set_stream(self, stream_ptr):
        check(self.lib.tiseg_set_stream(self.handle, _vp(stream_ptr or 0)), "tiseg_set_stream")

    def synchronize(self):
        check(self.lib.tiseg_synchronize(self.handle), "tiseg_synchronize")

    def launch_count(self):
        return int(self.lib.tiseg_launch_count(self.handle))

    def timing(self, on):
        check(self.lib.tiseg_timing_enable(self.handle, 1 if on else 0), "tiseg_timing_enable")

    def timing_report(self):
        """-> {kernel_name: (launches, total_ms)} since timing was enabled / last report."""
        buf = ctypes.create_string_buffer(1 << 16)
        check(self.lib.tiseg_timing_report(self.handle, buf, len(buf)), "tiseg_timing_report")
        out = {}
        for line in buf.value.decode().splitlines():
            name, n, ms = line.rsplit(" ", 2)
            out[name] = (int(n), float(ms))
        return out

    def call(self, name, *args):
        check(getattr(self.lib, name)(self.handle, *args), name)


_slot = threading.local()


def get_ctx(device=None):
    """Context for ``device`` (default: torch's current CUDA device), bound to torch's current
    stream so that zero-copy calls on CUDA tensors are ordered with the producer kernels.
    Inside ``with lane(k):`` the context of lane k is returned instead: every lane owns its own
    workspace arena, so calls issued on different streams never share scratch memory."""
    import torch
    if not torch.cuda.is_available():
        # still go through tiseg_create so the error is the library's own
        load()
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    device = int(device)
    key = (device, getattr(_slot, "k", 0))
    ctx = _ctxs.get(key)
    if ctx is None:
        ctx = Context(device)
        _ctxs[key] = ctx
    if torch.cuda.is_available():
        s = torch.cuda.current_stream(device).cuda_stream
        if getattr(ctx, "_bound", None) != s:
            ctx.set_stream(s)
            ctx._bound = s
    return ctx


class lane:
    """``with lane(k, stream):`` — operator calls inside use the k-th context of the device (own arena) and,
    if given, run on ``stream`` (a ``torch.cuda.Stream``).  Lanes are how a caller overlaps the host-to-device
    staging of one chunk of tiles with the kernels of the previous one (see ``parallel.HostFeed``)."""

    def __init__(self, k, stream=None):
        self.k, self.stream, self._sc = int(k), stream, None

    def __enter__(self):
        import torch
        self.prev = getattr(_slot, "k", 0)
        _slot.k = self.k
        if self.stream is not None:
            self._sc = torch.cuda.stream(self.stream)
            self._sc.__enter__()
        return self

    def __exit__(self, *exc):
        if self._sc is not None:
            self._sc.__exit__(*exc)
        _slot.k = self.prev
        return False


# --------------------------------------------------------------------------- array plumbing
def is_torch(a):
    return type(a).__module__.startswith("torch")


def ptr(a):
    if a is None:
        return _vp(0)
    if is_torch(a):
        return _vp(a.data_ptr())
    return _vp(a.ctypes.data)


_NP2T = None


def _torch_dtype(np_dtype):
    global _NP2T
    import torch
    if _NP2T is None:
        _NP2T = {np.dtype(np.uint8): torch.uint8, np.dtype(np.uint16): torch.uint16, np.dtype(np.int32): torch.int32,
                 np.dtype(np.int64): torch.int64,
                 np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64}
    return _NP2T[np.dtype(np_dtype)]


def as_input(a, dtype):
    """C-contiguous array of ``dtype``: numpy stays on the host (the library stages it), a CUDA
    tensor stays on the device (zero-copy)."""
    if is_torch(a):
        import torch
        td = _torch_dtype(dtype)
        if a.dtype == torch.bool and np.dtype(dtype) == np.uint8:
            a = a.to(torch.uint8)
        if a.dtype != td:
            a = a.to(td)
        return a.contiguous()
    a = np.asarray(a)
    if a.dtype == np.bool_ and np.dtype(dtype) == np.uint8:
        a = a.view(np.uint8)
    return np.ascontiguousarray(a, dtype=dtype)


# element type codes of the network outputs an entry with a dtype argument reads (TISEG_DTYPE_* in tiseg_b200.h)
DTYPE_F32, DTYPE_F16, DTYPE_BF16 = 0, 1, 2


def _half_code(a):
    if is_torch(a):
        import torch
        return {torch.float16: DTYPE_F16, torch.bfloat16: DTYPE_BF16}.get(a.dtype, DTYPE_F32)
    return DTYPE_F16 if isinstance(a, np.ndarray) and a.dtype == np.float16 else DTYPE_F32


def net_inputs(*arrays):
    """Network outputs of one call -> (arrays, dtype code).  fp16 / bf16 tensors (CUDA or CPU) and numpy float16 arrays are
    kept in their dtype, made C-contiguous, when every array of the call shares it: the library converts them to fp32 as
    it loads them (half the bytes read and staged, the same results as their fp32 upcast).  Anything else, mixed dtypes
    included, is converted to fp32 like ``as_input`` does (code DTYPE_F32)."""
    codes = {_half_code(a) for a in arrays}
    if len(codes) == 1 and DTYPE_F32 not in codes:
        return tuple(a.contiguous() if is_torch(a) else np.ascontiguousarray(a) for a in arrays), codes.pop()
    return tuple(as_input(a, np.float32) for a in arrays), DTYPE_F32


_device_out = threading.local()


class device_outputs:
    """``with device_outputs():`` — operators return CUDA tensors even for host (numpy) inputs, so a chain
    of calls keeps its intermediates in HBM and only the inputs cross PCIe."""

    def __enter__(self):
        self.prev = getattr(_device_out, "on", False)
        _device_out.on = True
        return self

    def __exit__(self, *exc):
        _device_out.on = self.prev
        return False


def empty_like_kind(ref, shape, dtype):
    """Output buffer of the same kind (numpy / CUDA tensor) as ``ref``."""
    import torch
    if is_torch(ref) and ref.is_cuda:
        return torch.empty(tuple(shape), dtype=_torch_dtype(dtype), device=ref.device)
    if getattr(_device_out, "on", False):
        return torch.empty(tuple(shape), dtype=_torch_dtype(dtype), device="cuda")
    return np.empty(tuple(shape), dtype=dtype)


def batched(a):
    """-> (array viewed as [N,H,W], was_2d)."""
    if a.ndim == 2:
        return a[None], True
    if a.ndim == 3:
        return a, False
    raise ValueError("expected a [H,W] or [N,H,W] array, got shape %r" % (tuple(a.shape),))
