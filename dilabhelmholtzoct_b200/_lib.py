"""ctypes binding of libtopoloss.so (include/topoloss.h).  No fallback: if the library is missing
or was built for another ABI this module raises, and every compute entry point needs a CUDA device."""
from __future__ import annotations

import ctypes
import os

from . import build as _build

_LIB = None

c_fp = ctypes.c_void_p  # device pointers travel as integers
TL_OK = 0
ABI_VERSION = 5
OPT_FORCE_GLOBAL_KERNEL, OPT_PROFILE, OPT_NO_BINARY_PATH, OPT_WORST_CASE_WORKSPACE, OPT_NO_FUSED_MATCH, OPT_NO_FUSED_GRAD = 0, 1, 2, 3, 4, 5
OPT_LIST_MODE = 6
STATUS_BITS = {1: "pair arena exhausted (pass a larger state buffer: TL_ARENA_FACTOR / set_arena_factor)",
               2: "basin tables exhausted (set TL_OPT_WORST_CASE_WORKSPACE)", 4: "a map holds a NaN"}

SIGNATURES = {
    "tl_version": (ctypes.c_int, []),
    "tl_last_error": (ctypes.c_char_p, []),
    "tl_max_pairs": (ctypes.c_int, [ctypes.c_int] * 3),
    "tl_set_option": (ctypes.c_int, [ctypes.c_int, ctypes.c_int]),
    "tl_get_option": (ctypes.c_int, [ctypes.c_int]),
    "tl_status": (ctypes.c_int, [c_fp, ctypes.POINTER(ctypes.c_int), c_fp]),
    "tl_workspace_bytes": (ctypes.c_int, [ctypes.c_int] * 5 + [ctypes.POINTER(ctypes.c_size_t)] * 2),
    "tl_pairs_workspace_bytes": (ctypes.c_int, [ctypes.c_int] * 4 + [ctypes.POINTER(ctypes.c_size_t)]),
    "tl_forward": (ctypes.c_int, [c_fp, c_fp] + [ctypes.c_int] * 5 + [ctypes.c_float, ctypes.c_float,
                                  ctypes.c_int, ctypes.c_int, c_fp, ctypes.c_size_t, c_fp, ctypes.c_size_t, c_fp, c_fp]),
    "tl_forward_backward": (ctypes.c_int, [c_fp, c_fp] + [ctypes.c_int] * 5 + [ctypes.c_float, ctypes.c_float,
                                           ctypes.c_int, ctypes.c_int, c_fp, ctypes.c_size_t, c_fp, ctypes.c_size_t, c_fp, c_fp, c_fp]),
    "tl_unpack_mask_bits": (ctypes.c_int, [c_fp, c_fp, ctypes.c_longlong, c_fp]),
    "tl_scale_gradient": (ctypes.c_int, [c_fp, c_fp, ctypes.c_longlong, c_fp]),
    "tl_backward": (ctypes.c_int, [c_fp, c_fp, ctypes.c_size_t] + [ctypes.c_int] * 5 +
                    [ctypes.c_float, ctypes.c_float, ctypes.c_int, ctypes.c_int, c_fp, c_fp]),
    "tl_persistence_pairs": (ctypes.c_int, [c_fp] + [ctypes.c_int] * 4 + [c_fp, ctypes.c_size_t, c_fp,
                                            ctypes.c_int, c_fp, c_fp]),
    "tl_wasserstein": (ctypes.c_int, [c_fp] * 4 + [ctypes.c_int] * 3 + [ctypes.c_float, c_fp,
                                      ctypes.c_size_t, c_fp, c_fp, c_fp]),
    "tl_timing_enable": (ctypes.c_int, [ctypes.c_int]),
    "tl_timing_read": (ctypes.c_int, [ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int)]),
    "tl_debug_profile": (ctypes.c_int, [c_fp, ctypes.POINTER(ctypes.c_ulonglong)]),
    "tl_debug_tail_profile": (ctypes.c_int, [c_fp] + [ctypes.c_int] * 3 + [ctypes.POINTER(ctypes.c_ulonglong), ctypes.c_int]),
    "tl_resample_forward": (ctypes.c_int, [c_fp] + [ctypes.c_int] * 5 + [c_fp, c_fp]),
    "tl_resample_backward": (ctypes.c_int, [c_fp, c_fp] + [ctypes.c_int] * 5 + [c_fp, c_fp]),
    "tl_postprocess_forward": (ctypes.c_int, [c_fp] + [ctypes.c_int] * 8 + [c_fp, c_fp]),
    "tl_postprocess_backward": (ctypes.c_int, [c_fp] + [ctypes.c_int] * 8 + [c_fp, c_fp]),
    "tl_dice_ce_workspace_bytes": (ctypes.c_int, [ctypes.c_int] * 2 + [ctypes.POINTER(ctypes.c_size_t)]),
    "tl_dice_ce_forward": (ctypes.c_int, [c_fp, c_fp] + [ctypes.c_int] * 3 + [c_fp, c_fp, c_fp]),
    "tl_dice_ce_backward": (ctypes.c_int, [c_fp, c_fp, c_fp] + [ctypes.c_int] * 3 + [c_fp, c_fp, c_fp]),
    "tl_wasserstein_workspace_bytes": (ctypes.c_int, [ctypes.c_int] * 3 + [ctypes.POINTER(ctypes.c_size_t)]),
    "tl_diagrams_workspace_bytes": (ctypes.c_int, [ctypes.c_int] * 4 + [ctypes.POINTER(ctypes.c_size_t)]),
    "tl_diagrams_compute": (ctypes.c_int, [c_fp] + [ctypes.c_int] * 4 + [c_fp, ctypes.c_size_t, c_fp, c_fp, c_fp]),
    "tl_diagrams_gather": (ctypes.c_int, [c_fp] + [ctypes.c_int] * 4 + [c_fp, ctypes.c_size_t, c_fp, c_fp,
                                          ctypes.c_longlong, c_fp, c_fp, c_fp]),
    "tl_diagrams_backward": (ctypes.c_int, [c_fp] * 3 + [ctypes.c_longlong] + [ctypes.c_int] * 3 + [c_fp, c_fp]),
    "tl_wasserstein_backward": (ctypes.c_int, [c_fp] * 4 + [ctypes.c_int, ctypes.c_float] + [c_fp] * 5),
    "tl_betti_workspace_bytes": (ctypes.c_int, [ctypes.c_int] * 4 + [ctypes.POINTER(ctypes.c_size_t)]),
    "tl_betti_compute": (ctypes.c_int, [c_fp, c_fp] + [ctypes.c_int] * 4 + [c_fp, ctypes.c_size_t, c_fp, c_fp, c_fp, c_fp]),
    "tl_betti_gather": (ctypes.c_int, [ctypes.c_int] * 4 + [c_fp, ctypes.c_size_t, c_fp, c_fp] + [ctypes.c_longlong] * 3 +
                        [c_fp] * 4),
    "tl_betti_backward": (ctypes.c_int, [c_fp, c_fp] + [ctypes.c_int] * 3 + [c_fp, c_fp, ctypes.c_longlong, c_fp,
                          ctypes.c_longlong, c_fp, ctypes.c_longlong] + [c_fp] * 4),
    "tl_prior_workspace_bytes": (ctypes.c_int, [ctypes.c_int] * 4 + [ctypes.POINTER(ctypes.c_size_t)] * 2),
    "tl_prior_forward": (ctypes.c_int, [c_fp] + [ctypes.c_int] * 4 + [c_fp, c_fp, ctypes.c_size_t, c_fp, ctypes.c_size_t,
                                        c_fp, c_fp]),
    "tl_prior_backward": (ctypes.c_int, [c_fp] + [ctypes.c_int] * 4 + [c_fp, ctypes.c_size_t, c_fp, c_fp, c_fp]),
    "tl_edt_workspace_bytes": (ctypes.c_int, [ctypes.c_int] * 3 + [ctypes.POINTER(ctypes.c_size_t)]),
    "tl_edt": (ctypes.c_int, [c_fp] + [ctypes.c_int] * 3 + [c_fp, c_fp, ctypes.c_size_t, c_fp, c_fp]),
    "tl_hausdorff_dt_workspace_bytes": (ctypes.c_int, [ctypes.c_int] * 3 + [ctypes.POINTER(ctypes.c_size_t)] * 2),
    "tl_hausdorff_dt_forward": (ctypes.c_int, [c_fp, c_fp] + [ctypes.c_int] * 3 + [ctypes.c_double, c_fp, c_fp,
                                               ctypes.c_size_t, c_fp, ctypes.c_size_t, c_fp, c_fp]),
    "tl_hausdorff_dt_backward": (ctypes.c_int, [c_fp, c_fp] + [ctypes.c_int] * 3 + [c_fp, ctypes.c_size_t, c_fp, c_fp, c_fp]),
    "tl_surface_workspace_bytes": (ctypes.c_int, [ctypes.c_int] * 3 + [ctypes.POINTER(ctypes.c_size_t)]),
    "tl_surface_distances": (ctypes.c_int, [c_fp, c_fp] + [ctypes.c_int] * 3 + [c_fp, ctypes.c_double, ctypes.c_double,
                                            c_fp, ctypes.c_size_t, c_fp, c_fp]),
    "tl_boundary_workspace_bytes": (ctypes.c_int, [ctypes.c_int] * 3 + [ctypes.POINTER(ctypes.c_size_t)] * 2),
    "tl_boundary_forward": (ctypes.c_int, [c_fp, c_fp] + [ctypes.c_int] * 3 + [c_fp, c_fp, ctypes.c_size_t, c_fp,
                                           ctypes.c_size_t, c_fp, c_fp]),
    "tl_boundary_backward": (ctypes.c_int, [c_fp] + [ctypes.c_int] * 3 + [c_fp, ctypes.c_size_t, c_fp, c_fp, c_fp]),
    "tl_signed_distance": (ctypes.c_int, [c_fp] + [ctypes.c_int] * 3 + [c_fp, c_fp, ctypes.c_size_t, c_fp, c_fp]),
}


def lib() -> ctypes.CDLL:
    global _LIB
    if _LIB is None:
        path = os.environ.get("TL_LIB_PATH") or _build.LIB_PATH  # TL_LIB_PATH: a debug build of the same library
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} is missing: build it with `python -m dilabhelmholtzoct_b200.build` "
                "(nvcc, sm_100a).  There is no CPU or PyTorch fallback for the topological loss.")
        L = ctypes.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        if L.tl_version() != ABI_VERSION:
            raise RuntimeError(f"libtopoloss.so ABI {L.tl_version()} != expected {ABI_VERSION}; rebuild")
        _LIB = L
    return _LIB


def check(rc: int, what: str) -> None:
    if rc != TL_OK:
        msg = lib().tl_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError(f"{what}: {msg}")
        raise RuntimeError(f"{what} failed ({rc}): {msg}")
