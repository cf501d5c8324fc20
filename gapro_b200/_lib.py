"""ctypes binding of libgapro_b200.so (the C ABI declared in include/gapro_b200.h).

There is no fallback: if the shared library is missing or a call fails, the
caller gets an exception.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int32, c_int64, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgapro_b200.so")

EV_NEST_B1, EV_NEST_B2, EV_GP = 0, 1, 2
GP_NOT_PSD, GP_NAN, GP_RETRY_SHIFT = 1, 2, 8

_lib = None

P = c_void_p
_SIGNATURES = {
    "gapro_version": (ctypes.c_int, []),
    "gapro_last_error": (c_char_p, []),
    "gapro_densify_workspace_bytes": (c_size_t, [c_int64, c_int32]),
    "gapro_densify_spp": (ctypes.c_int, [P, P, c_int32, P, P, P, P, P, c_size_t, P]),
    "gapro_floor_boxes": (ctypes.c_int, [P, P, P, c_int32, c_int64, c_double, P, P, P, P]),
    "gapro_occupancy": (ctypes.c_int, [P, P, P, P, P, P, c_int32, c_int32, c_int32, c_int32, c_double, c_float,
                                       P, P, P, P, P, P]),
    "gapro_occupancy_points_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "gapro_occupancy_points": (ctypes.c_int, [P, P, P, P, P, P, P, P, c_int32, c_int64, c_int32, c_int32, c_int32,
                                              c_double, c_float, P, P, P, P, P, P, c_size_t, P]),
    "gapro_heuristic_labels": (ctypes.c_int, [P, P, P, P, P, P, P, P, c_int32, c_int32, c_int32, c_int32, c_int32,
                                              c_float, P, P, P]),
    "gapro_multibox_workspace_bytes": (c_size_t, [c_int64]),
    "gapro_multibox_sources": (ctypes.c_int, [P, P, P, P, c_int32, c_int64, P, P, c_size_t, P]),
    "gapro_heuristic_finalize": (ctypes.c_int, [P, P, P, P, P, P, c_int32, c_int32, c_int32, c_int64, c_int32, P, P,
                                                P, P]),
    "gapro_pool_feats": (ctypes.c_int, [P, P, P, c_int32, c_int32, P, P]),
    "gapro_enumerate_events": (ctypes.c_int, [P, c_int32, P, P, c_int32, P, P, P, c_int32]),
    "gapro_box_iou": (ctypes.c_int, [P, c_int32, P]),
    "gapro_compact_lists": (ctypes.c_int, [P, P, P, c_int32, P, P, P, P, c_int32, P, P]),
    "gapro_gp_workspace_bytes": (c_size_t, [c_int32, P, P, c_int32]),
    "gapro_gp_min_workspace_bytes": (c_size_t, [c_int32, P, P, c_int32]),
    "gapro_gp_fit_batch": (ctypes.c_int, [P, c_int32, c_int32, P, P, P, P, P, P, c_int32, c_double, c_double,
                                          c_double, P, P, P, P, P, P, P, P, P, c_size_t, P]),
    "gapro_gp_last_launch_count": (c_int64, []),
    "gapro_gp_debug_aux_slack": (c_int64, [c_int32, P, P, c_int32]),
    "gapro_gp_set_profiling": (ctypes.c_int, [ctypes.c_int]),
    "gapro_gp_phase_names": (c_char_p, []),
    "gapro_gp_get_profile": (ctypes.c_int, [P, P, P, c_int32]),
    "gapro_fp64_peak": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, P, P, P]),
    "gapro_gather_peak": (ctypes.c_int, [P, P, c_int64, P, P]),
    "gapro_gp_debug_run": (ctypes.c_int, [P, c_int32, c_int32, c_int32, c_int32, P, P, P, c_int32, c_int32,
                                          c_double, c_double, c_double, P, c_size_t, P, c_int32, P]),
    "gapro_gp_debug_layout_names": (c_char_p, []),
    "gapro_resolve_spp": (ctypes.c_int, [P, P, c_int32, P, P, P, P, P, c_int32, c_int32, P, P, P, P, P, P, P, P,
                                         P, P, P, P, P, P, P, P, P, P, P]),
    "gapro_broadcast_labels": (ctypes.c_int, [P, c_int64, P, P, P, P, P]),
    "gapro_ozaki_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32, c_int32]),
    "gapro_ozaki_gemm": (ctypes.c_int, [P, c_int32, c_int32, P, P, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32,
                                        P, c_int32, P, c_size_t, c_int32, P, P, P]),
    "gapro_instance_info_workspace_bytes": (c_size_t, [c_int32]),
    "gapro_instance_info": (ctypes.c_int, [P, P, P, c_int64, c_int32, c_int32, P, P, P, P, P, c_size_t, P]),
    "gapro_eval_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "gapro_eval_miou_scene": (ctypes.c_int, [P, P, P, P, c_int64, c_int32, c_int32, P, P, P, c_size_t, P]),
    "gapro_eval_sem_conf": (ctypes.c_int, [P, P, c_int64, c_int32, P, P]),
}
EXPORTS = tuple(_SIGNATURES)


class GaproError(RuntimeError):
    pass


class GaproSceneError(GaproError):
    """A GP region of one or more scenes could not be fitted (gpytorch would raise NotPSDError / NanError and
    kill the run, gen_ps_utils.py:434-437).  `.scenes` maps the batch index of every failed scene to a message;
    the other scenes of the batch were labelled and are in `.results` (None at the failed positions)."""

    def __init__(self, scenes, results):
        self.scenes, self.results = dict(scenes), results
        super().__init__("; ".join(f"scene {i}: {m}" for i, m in sorted(self.scenes.items())))


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GaproError(
            f"{LIB_PATH} is missing: build it with `python -m gapro_b200.build` "
            "(nvcc, sm_100a).  gapro_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc < 0:
        msg = load().gapro_last_error().decode("utf-8", "replace")
        raise GaproError(f"{what} failed ({rc}): {msg}")
    return rc
