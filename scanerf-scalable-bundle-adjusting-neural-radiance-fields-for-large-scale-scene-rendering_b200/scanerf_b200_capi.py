"""ctypes loader for libscanerf_b200.so -- the C-ABI boundary (include/scanerf_b200.h).

There is NO CPU fallback and no alternative backend: if the shared library is
missing, or a tensor is not on a CUDA device, the call raises.  PyTorch is used
only for device memory and streams; every op takes raw device pointers, sizes
and the current CUDA stream.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libscanerf_b200.so")
_lib = None

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_float = ctypes.c_float


# --- instrumentation used by bench.py: launch counter and per-entry-point CUDA-event timing
launch_count = 0            # C-ABI calls that launched a kernel since last reset
_timed_name = None          # entry point being timed (None = off)
_timed_events = []          # [(start_event, end_event, units)]
_UNITS_ARG = {"snrf_hash_fwd": 7, "snrf_hash_bwd": 8, "snrf_field_encode_fwd": 13, "snrf_field_encode_bwd": 16,
              "snrf_field_encode_bwd_adam": 27, "snrf_field_encode_bwd_ert": 16, "snrf_field_encode_bwd_adam_ert": 27}
_HOST_ONLY = {"snrf_last_error", "snrf_version", "snrf_device_sm_count", "snrf_l2_fetch_granularity", "snrf_hash_set_levels_per_block",
              "snrf_decoder_set_precision", "snrf_composite_set_fwd_packed", "snrf_infer_set_chunk_log2", "snrf_infer_release_scratch", "snrf_field_set_passes_log2", "snrf_field_set_aggregate_levels", "snrf_field_set_run_length", "snrf_field_set_bwd_impl", "snrf_field_set_fwd_pairing", "snrf_field_set_fwd_l2_policy", "snrf_field_set_fwd_pair_loads", "snrf_field_set_fwd_split_levels", "snrf_field_set_levels_per_group", "snrf_field_set_profile", "snrf_field_last_profile", "snrf_field_last_launch_count", "snrf_field_set_overlap", "snrf_field_set_coarse_concurrent", "snrf_field_set_l2_hints", "snrf_field_set_pdl", "snrf_field_set_persist_mib", "snrf_field_set_occupancy_smem", "snrf_field_set_slice_log2",
              "snrf_voxelize_mesh_host"}


class _Lib:
    """Thin proxy over the CDLL: counts kernel-launching calls and, when asked, brackets one
    entry point with CUDA events on the current stream."""

    def __init__(self, cdll):
        self._cdll = cdll
        self._cache = {}

    def __getattr__(self, name):
        fn = self._cache.get(name)
        if fn is None:
            raw = getattr(self._cdll, name)
            if name in _HOST_ONLY:
                fn = raw
            else:
                def fn(*args, _raw=raw, _name=name):
                    global launch_count
                    launch_count += 1
                    if _timed_name is not None and _name in _timed_name:
                        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        a.record()
                        rc = _raw(*args)
                        b.record()
                        u = args[_UNITS_ARG[_name]] if _name in _UNITS_ARG else 0
                        _timed_events.append((a, b, int(getattr(u, "value", u)), _name))
                        return rc
                    return _raw(*args)
            self._cache[name] = fn
        return fn


def time_calls(name):
    """Start (a name, or a tuple of names) or stop (None) CUDA-event timing of C-ABI entry points."""
    global _timed_name
    _timed_name = (name,) if isinstance(name, str) else (tuple(name) if name else None)
    if name is not None:
        _timed_events.clear()


def timed_results():
    """([ms per launch], [units per launch]) of the calls timed since time_calls(name); synchronises."""
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b, _, _ in _timed_events], [u for _, _, u, _ in _timed_events]


def timed_by_name():
    """{entry point: [ms per call]} of the calls timed since time_calls(names); synchronises."""
    torch.cuda.synchronize()
    out = {}
    for a, b, _, name in _timed_events:
        out.setdefault(name, []).append(a.elapsed_time(b))
    return out


def lib():
    """Load (once) and return the library.  Raises loudly when the build is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"scanerf_b200: native library not found at {LIB_PATH}. "
                "Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C <package>/csrc`). There is no CPU / PyTorch fallback.")
        cdll = ctypes.CDLL(LIB_PATH)
        cdll.snrf_last_error.restype = ctypes.c_char_p
        _lib = _Lib(cdll)
    return _lib


def stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def check(rc, name):
    if rc != 0:
        msg = lib().snrf_last_error()
        raise RuntimeError(f"scanerf_b200::{name} failed (code {rc}): {msg.decode() if msg else ''}")


def _require_cuda(t, name):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t)}")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor (scanerf_b200 has no CPU fallback)")
    if t.device.index != torch.cuda.current_device():
        # kernels are launched on the CURRENT device's current stream (one process per GPU, as the reference: cuda:0 of
        # its CUDA_VISIBLE_DEVICES, admm_trainer.py:202); a tensor of another device would be dereferenced there
        raise RuntimeError(f"{name} lives on {t.device} but the current CUDA device is cuda:{torch.cuda.current_device()}; "
                           "call torch.cuda.set_device(...) first")


def inp(t, dtype, name):
    """Input tensor -> contiguous tensor of `dtype` on the GPU (the reference calls
    .contiguous() on every input too).  Returns the tensor; keep it alive during the call."""
    _require_cuda(t, name)
    if t.dtype != dtype:
        raise RuntimeError(f"{name} must have dtype {dtype}, got {t.dtype}")
    return t.contiguous()


class Out:
    """Output tensor written in place.  A non-contiguous output is staged through a
    contiguous copy and copied back (the reference silently wrote to a temporary)."""

    def __init__(self, t, dtype, name):
        _require_cuda(t, name)
        if t.dtype != dtype:
            raise RuntimeError(f"{name} must have dtype {dtype}, got {t.dtype}")
        self.orig = t
        self.t = t if t.is_contiguous() else t.contiguous()

    @property
    def ptr(self):
        return c_void_p(self.t.data_ptr())

    def done(self):
        if self.t is not self.orig:
            self.orig.copy_(self.t)


def ptr(t):
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(0)
