"""ctypes binding of libperfb200.so (the C-ABI declared in include/perfb200.h).

The library is the product; there is NO fallback.  If it is missing and cannot be built, or a
call fails, this module raises.  Nothing here imports ``oracle``.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

u32, u64, f32, i32, vp = C.c_uint32, C.c_uint64, C.c_float, C.c_int, C.c_void_p

PERF_FLAG_TRAINING = 1
PERF_FLAG_SIMT_MLP = 2
PERF_FLAG_SCAN_KERNEL = 4
PERF_FLAG_GENERIC_ADDR = 8
PERF_FLAG_L0_SMEM = 16


class GridCfg(C.Structure):
    _fields_ = [("n_levels", u32), ("n_features_per_level", u32), ("log2_hashmap_size", u32),
                ("base_resolution", u32), ("per_level_scale", f32), ("interpolation", u32)]


class Level(C.Structure):
    _fields_ = [("scale", f32), ("resolution", u32), ("size", u32), ("offset", u32), ("hashed", u32)]


class MlpCfg(C.Structure):
    _fields_ = [("n_in", u32), ("n_out", u32), ("n_neurons", u32), ("n_hidden_layers", u32),
                ("output_activation", u32)]


class RenderArgs(C.Structure):
    _fields_ = [("grid", GridCfg), ("d_packed_table", vp), ("d_geo_mlp_half", vp), ("d_app_mlp_half", vp),
                ("aabb", f32 * 6), ("n_samples", u32), ("near", f32), ("far", f32), ("flags", u32),
                ("d_jitter", vp), ("d_bg_noise", vp), ("d_rgb", vp), ("d_distance", vp), ("d_opacity", vp), ("image_width", u32)]


class OccRenderArgs(C.Structure):
    _fields_ = [("d_binaries", vp), ("res", i32 * 3), ("aabb", f32 * 6), ("near", f32), ("far", f32), ("step", f32),
                ("early_stop_eps", f32), ("d_n_samples", vp)]


P_u32 = C.POINTER(u32)
PERF_MAX_SEGMENTS = 64


class TrainBuffers(C.Structure):
    _fields_ = [("d_sigma", vp), ("d_weights", vp), ("d_trans", vp), ("d_rgb", vp), ("d_feat", vp), ("d_h1", vp),
                ("d_h2", vp), ("d_dist_acc", vp), ("d_distloss", vp), ("d_seg_trans", vp), ("h_segments_out", P_u32)]


PERF_PHASE_GEO, PERF_PHASE_APP = 1, 2

P = C.POINTER
# name -> (restype, argtypes); must list every symbol include/perfb200.h declares
SIGNATURES = {
    "perf_abi_version": (i32, []),
    "perf_last_error": (C.c_char_p, []),
    "perf_device_arch": (i32, []),
    "perf_grid_describe": (i32, [P(GridCfg), P(Level), P(u64)]),
    "perf_network_param_count": (i32, [P(GridCfg), P(MlpCfg), P(u64)]),
    "perf_params_to_half": (i32, [vp, vp, u64, vp]),
    "perf_packed_table_entries": (i32, [P(GridCfg), P(u64)]),
    "perf_pack_tables": (i32, [P(GridCfg), P(MlpCfg), P(MlpCfg), vp, vp, vp, vp]),
    "perf_raygen_pano": (i32, [P(f32), i32, i32, i32, i32, vp, vp, vp]),
    "perf_raygen_pers": (i32, [P(f32), f32, i32, i32, vp, vp, vp]),
    "perf_hashgrid_fwd": (i32, [P(GridCfg), vp, vp, u64, vp, vp]),
    "perf_hashgrid_bwd": (i32, [P(GridCfg), vp, vp, u64, vp, vp]),
    "perf_hashgrid_bwd_input": (i32, [P(GridCfg), vp, vp, vp, u64, vp, vp]),
    "perf_hashgrid_bwd_bwd_input": (i32, [P(GridCfg), vp, vp, vp, vp, u64, vp, vp, vp, vp]),
    "perf_network_fwd": (i32, [P(GridCfg), P(MlpCfg), vp, vp, u64, vp, vp, vp, vp, u32, vp]),
    "perf_mlp_fwd": (i32, [P(MlpCfg), vp, vp, u64, vp, vp, vp, u32, vp]),
    "perf_weights_from_density": (i32, [vp, vp, vp, vp, u64, u64, vp, vp, vp, vp]),
    "perf_weights_from_density_bwd": (i32, [vp, vp, vp, vp, u64, u64, vp, vp, vp, vp, vp, vp]),
    "perf_accumulate_along_rays": (i32, [vp, vp, i32, vp, u64, u64, vp, vp]),
    "perf_render_rays": (i32, [P(RenderArgs), vp, vp, u64, vp]),
    "perf_render_packed": (i32, [P(RenderArgs), vp, vp, u64, vp, vp, vp, vp]),
    "perf_render_pano": (i32, [P(RenderArgs), P(f32), i32, i32, i32, i32, vp]),
    "perf_render_rays_occ": (i32, [P(RenderArgs), P(OccRenderArgs), vp, vp, u64, vp]),
    "perf_render_pano_occ": (i32, [P(RenderArgs), P(OccRenderArgs), P(f32), i32, i32, i32, i32, vp]),
    "perf_train_forward": (i32, [P(RenderArgs), vp, vp, u64, i32, P(TrainBuffers), vp]),
    "perf_train_backward_composite": (i32, [i32, u32, u32, f32, f32, u64, vp, vp, P(TrainBuffers), vp, vp, vp, vp, vp, vp, vp, vp]),
    "perf_hashgrid_bwd_rays": (i32, [P(GridCfg), P(f32), vp, vp, vp, u64, u32, f32, f32, vp, vp, vp]),
    "perf_occ_count": (i32, [vp, P(i32), P(f32), vp, vp, vp, u64, f32, f32, f32, u32, vp, vp, vp]),
    "perf_occ_write": (i32, [vp, P(i32), P(f32), vp, vp, vp, u64, f32, f32, f32, u32, vp, u64, vp, vp, vp, vp, vp]),
    "perf_mlp_bwd": (i32, [P(MlpCfg), vp, vp, vp, vp, vp, u64, vp, vp, vp, u32, vp]),
    "perf_mlp_bwd_scatter": (i32, [P(MlpCfg), vp, vp, vp, vp, vp, u64, vp, vp, P(GridCfg), P(f32), vp, vp, vp, u64, u32, f32, f32, vp, vp]),
    "perf_hashgrid_bwd_rays_coarse": (i32, [P(GridCfg), P(f32), vp, vp, vp, u64, u32, f32, f32, vp, vp, vp]),
    "perf_fields_packed": (i32, [P(RenderArgs), vp, vp, vp, vp, vp, u64, vp, i32, vp, vp, vp, vp, vp, vp, vp]),
    "perf_composite_packed_fwd": (i32, [vp, vp, vp, vp, vp, u64, f32, u32, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "perf_composite_packed_bwd": (i32, [i32, vp, vp, vp, vp, vp, u64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "perf_hashgrid_bwd_merged": (i32, [P(GridCfg), vp, vp, u64, vp, vp, u32, vp]),
    "perf_gather_rows": (i32, [vp, u64, i32, vp, vp, vp, vp]),
    "perf_draw_gather_rows": (i32, [vp, u64, u64, vp, i32, vp, vp, vp, vp]),
    "perf_train_loss": (i32, [vp, vp, u64, u64, f32, f32, vp, vp, vp, f32, vp, vp, vp, vp]),
    "perf_debug_atomic_rate": (i32, [vp, u64, u64, i32, vp]),
    "perf_occ_points": (i32, [vp, u64, P(i32), P(f32), u64, vp, vp]),
    "perf_occ_update": (i32, [vp, u64, vp, vp, u64, f32, f32, vp, vp, vp]),
    "perf_mlp_bwd_out": (i32, [vp, i32, vp, vp, vp, u64, vp]),
    "perf_relu_mask": (i32, [vp, vp, u64, vp]),
    "perf_adam_step": (i32, [vp, vp, vp, vp, vp, u64, f32, f32, f32, f32, u32, f32, vp]),
    "perf_set_scalars": (i32, [vp, P(f32), i32, vp]),
    "perf_adam_step_dev": (i32, [vp, vp, vp, vp, vp, u64, vp, f32, f32, f32, f32, vp]),
}

_LIB = None


def lib_path() -> str:
    return _build.LIB


def load(rebuild_if_stale: bool = True) -> C.CDLL:
    """Load (building first when nvcc is available and sources are newer) libperfb200.so."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    override = os.environ.get("PERF_B200_LIB")           # A/B of kernel variants (tools/ab_lib.py): load this build as it is
    if override:
        path, rebuild_if_stale = override, False
    if rebuild_if_stale and (not os.path.exists(path) or _build.is_stale()):
        try:
            _build.build()
        except _build.NvccMissing as e:             # no compiler on this box: the shipped .so is all there is
            if not os.path.exists(path):
                raise ImportError(f"libperfb200.so is missing and could not be built: {e}") from e
            import warnings
            warnings.warn("libperfb200.so is older than its sources and nvcc is not available: using the shipped binary")
        # any other failure (an nvcc compile error after a kernel edit) propagates: never run a stale binary silently
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)                     # AttributeError if the symbol is not exported
        fn.restype, fn.argtypes = res, args
    if lib.perf_abi_version() != 1:
        raise ImportError(f"libperfb200.so ABI {lib.perf_abi_version()} != 1")
    _LIB = lib
    return lib


class PerfError(RuntimeError):
    pass


def check(rc: int) -> None:
    if rc != 0:
        msg = load().perf_last_error()
        raise PerfError(f"libperfb200 error {rc}: {msg.decode() if msg else '?'}")
