"""ctypes binding of the C-ABI shared library ``matrix0_b200/_lib/libmatrix0_b200.so``.

The library is the product: there is no CPU or PyTorch fallback behind these entry points.  If
the library is missing, was not built for sm_100a, or no CUDA device is visible, every compute
call raises ``NativeLibraryError`` loudly instead of degrading to another implementation.
Symbols are declared in ``include/matrix0_b200.h``.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint64, c_void_p
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libmatrix0_b200.so")


class NativeLibraryError(RuntimeError):
    pass


M0_ERR_ARG = -2   # include/matrix0_b200.h: invalid argument


_lib: Optional[ctypes.CDLL] = None

# name -> (restype, argtypes); kept in one table so tests can check every header symbol is exported
SIGNATURES = {
    "m0_last_error": (c_char_p, []),
    "m0_version": (c_int, []),
    "m0_device_count": (c_int, []),
    "m0_device_sm_count": (c_int, [c_int]),
    "m0_launch_count": (c_uint64, []),
    "m0_positions_pack": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "m0_random_playouts": (c_int, [c_void_p, c_int, c_uint64, c_int, c_void_p]),
    "m0_encode_positions": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "m0_encode_planes": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "m0_legal_mask": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "m0_ssl_targets": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "m0_legal_moves": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "m0_engine_create": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_void_p)]),
    "m0_engine_destroy": (c_int, [c_void_p]),
    "m0_engine_bytes": (c_int64, [c_void_p]),
    "m0_engine_configure": (c_int, [c_void_p, c_void_p, c_void_p]),
    "m0_games_reset": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "m0_games_set_positions": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "m0_games_get_positions": (c_int, [c_void_p, c_void_p, c_void_p]),
    "m0_search_begin": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "m0_search_select": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "m0_search_expand_backup": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "m0_search_add_dirichlet": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "m0_search_pending": (c_int, [c_void_p, c_void_p, c_void_p]),
    "m0_search_pending_counts": (c_int, [c_void_p, c_void_p, c_void_p]),
    "m0_search_result": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "m0_search_multi_enable": (c_int, [c_void_p, c_int, c_int]),
    "m0_search_set_streams": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p]),
    "m0_search_select_multi": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "m0_search_multi_encode": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p]),
    "m0_search_expand_backup_multi": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p]),
    "m0_search_reuse_enable": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "m0_search_reuse_clear": (c_int, [c_void_p, c_void_p]),
    "m0_gumbel_configure": (c_int, [c_void_p, c_int, c_int, c_double, c_double]),
    "m0_gumbel_set_draws": (c_int, [c_void_p, c_void_p]),
    "m0_gumbel_select": (c_int, [c_void_p, c_void_p, c_void_p]),
    "m0_gumbel_expand_backup": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "m0_gumbel_result": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "m0_selfplay_advance_gumbel": (c_int, [c_void_p, c_void_p, c_void_p]),
    "m0_engine_counters": (c_int, [c_void_p, c_void_p]),
    "m0_engine_status": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "m0_search_select_var": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "m0_selfplay_plies": (c_int, [c_void_p, c_void_p, c_void_p]),
    "m0_selfplay_configure": (c_int, [c_void_p, c_void_p, c_void_p]),
    "m0_selfplay_start": (c_int, [c_void_p, c_void_p]),
    "m0_selfplay_advance": (c_int, [c_void_p, c_void_p, c_void_p]),
    "m0_selfplay_set_start_budget": (c_int, [c_void_p, c_int64, c_void_p]),
    "m0_selfplay_active_games": (c_int, [c_void_p, ctypes.POINTER(c_int), c_void_p]),
    "m0_selfplay_set_uniforms": (c_int, [c_void_p, c_void_p]),
    "m0_trees_clear": (c_int, [c_void_p, c_void_p]),
    "m0_selfplay_finished": (c_int, [c_void_p, c_void_p, c_int, ctypes.POINTER(c_int), c_void_p]),
    "m0_net_create": (c_int, [c_int, c_void_p, c_void_p, ctypes.POINTER(c_void_p)]),
    "m0_net_destroy": (c_int, [c_void_p]),
    "m0_net_forward": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p]),
    "m0_tc_conv": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "m0_tc_conv_fp8": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "m0_profile_enable": (c_int, [c_int]),
    "m0_profile_get": (c_int, [c_char_p, ctypes.POINTER(c_double), ctypes.POINTER(ctypes.c_longlong)]),
    "m0_net_forward_ssl": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
}


class SearchConfigStruct(ctypes.Structure):
    """struct m0_search_config (include/matrix0_b200.h)."""
    _fields_ = [
        ("fpu_reduction", c_double), ("draw_penalty", c_double), ("selection_jitter", c_double),
        ("dirichlet_alpha", c_double), ("dirichlet_frac", c_double),
        ("deterministic", c_int), ("no_instant_backtrack", c_int), ("legal_softmax", c_int),
        ("enable_entropy_noise", c_int), ("value_from_white", c_int), ("cpuct_len", c_int),
        ("seed", c_uint64), ("cpuct_by_depth", ctypes.POINTER(c_double)),
        ("max_children", c_int), ("raw_logit_priors", c_int), ("min_child_prior", c_double),
        ("virtual_loss", c_double), ("virtual_loss_on", c_int), ("reserved", c_int),
    ]


def load_library() -> ctypes.CDLL:
    """Load the shared library (no GPU needed for loading) and bind the declared signatures."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise NativeLibraryError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). matrix0_b200 has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def lib() -> ctypes.CDLL:
    """Library handle for compute calls: additionally requires a visible CUDA device."""
    l = load_library()
    if l.m0_device_count() <= 0:
        raise NativeLibraryError("no CUDA device visible: matrix0_b200 runs only on a GPU (sm_100a), no CPU path exists")
    return l


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load_library().m0_last_error()
        raise NativeLibraryError(f"{what or 'native call'} failed (rc={rc}): {msg.decode() if msg else '?'}")


def ptr(t) -> int:
    """Device pointer of a torch tensor (or 0 for None)."""
    return 0 if t is None else t.data_ptr()


def current_stream() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


def on_own_device(cls):
    """Class decorator: every plain method defined by ``cls`` (no generators, properties or static / class methods) runs with
    ``self.device`` as the current CUDA device.  The library launches on the caller's current device and stream, so an object that
    lives on cuda:1 must not depend on the caller having selected cuda:1 -- the reference's workers pick their device by process
    index (internal.py:120-130) and an orchestrator process may hold objects on several devices."""
    import functools
    import inspect

    def wrap(fn):
        @functools.wraps(fn)
        def run(self, *a, **kw):
            dev = getattr(self, "device", None)
            if dev is None:                              # still inside __init__, before the device is known
                return fn(self, *a, **kw)
            import torch
            with torch.cuda.device(dev):
                return fn(self, *a, **kw)
        return run

    for name, fn in list(vars(cls).items()):
        if name in ("__init__", "__del__", "close") or (name.startswith("__") and name.endswith("__")):
            continue
        if inspect.isfunction(fn) and not inspect.isgeneratorfunction(fn):
            setattr(cls, name, wrap(fn))
    return cls
