"""ctypes binding of the C ABI declared in include/gecco_b200.h.

The shared library is built in-tree by gecco_b200.build; there is no CPU fallback: if the
library is missing or the device is not sm_100 every op raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_LIB_PATH = Path(__file__).resolve().parent / "lib" / "libgecco_b200.so"
_lib = None
_inited_devices: set[int] = set()


class GeccoError(RuntimeError):
    pass


# activation codes (GECCO_ACT_*)
ACT_NONE, ACT_GAUSSIAN, ACT_GAUSSIAN_RAW, ACT_RELU = 0, 1, 2, 3


class ANorm(C.Structure):
    _fields_ = [
        ("stats", C.c_void_p), ("stat_gs", C.c_int32), ("groups", C.c_int32), ("eps", C.c_float),
        ("t", C.c_void_p), ("t_stride", C.c_int32),
        ("scale_w", C.c_void_p), ("scale_b", C.c_void_p), ("bias_w", C.c_void_p), ("bias_b", C.c_void_p),
    ]


class GemmArgs(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("lda", C.c_int64),
        ("w", C.c_void_p), ("ldw", C.c_int64),
        ("m", C.c_int32), ("n_out", C.c_int32), ("k", C.c_int32),
        ("rows_per_cloud", C.c_int32), ("valid_rows", C.c_int32), ("w_rows_per_cloud", C.c_int32),
        ("bias", C.c_void_p), ("bias_stride", C.c_int32),
        ("act", C.c_int32), ("act_alpha", C.c_float),
        ("res", C.c_void_p), ("ldr", C.c_int64),
        ("out_f32", C.c_void_p), ("ldo32", C.c_int64),
        ("out_bf16", C.c_void_p), ("ldo16", C.c_int64),
        ("stats", C.c_void_p),
        ("geom", C.c_void_p),
        ("sigma", C.c_void_p), ("sigma_stride", C.c_int32), ("sigma_data", C.c_float),
        ("wx", C.c_void_p),
        ("anorm", ANorm),
        ("stat_gs", C.c_int32),
    ]


class MlpArgs(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("lda", C.c_int64),
        ("w1", C.c_void_p), ("ldw1", C.c_int64), ("w1_rows_per_cloud", C.c_int32),
        ("b1", C.c_void_p), ("b1_stride", C.c_int32),
        ("act_alpha", C.c_float),
        ("w2", C.c_void_p), ("ldw2", C.c_int64),
        ("b2", C.c_void_p),
        ("m", C.c_int32), ("c", C.c_int32), ("hidden", C.c_int32),
        ("rows_per_cloud", C.c_int32), ("valid_rows", C.c_int32),
        ("res", C.c_void_p), ("ldr", C.c_int64),
        ("out_f32", C.c_void_p), ("ldo32", C.c_int64),
        ("out_bf16", C.c_void_p), ("ldo16", C.c_int64),
        ("stats", C.c_void_p),
        ("anorm", ANorm),
        ("scratch", C.c_void_p),
        ("stat_gs", C.c_int32),
        ("act", C.c_int32),
    ]


class AdaGNArgs(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("ldx", C.c_int64),
        ("stats", C.c_void_p), ("stat_gs", C.c_int32),
        ("t", C.c_void_p), ("t_stride", C.c_int32), ("ctx_dim", C.c_int32),
        ("scale_w", C.c_void_p), ("scale_b", C.c_void_p), ("bias_w", C.c_void_p), ("bias_b", C.c_void_p),
        ("clouds", C.c_int32), ("rows_per_cloud", C.c_int32), ("valid_rows", C.c_int32), ("c", C.c_int32),
        ("groups", C.c_int32),
        ("eps", C.c_float),
        ("out_bf16", C.c_void_p), ("ldo16", C.c_int64),
        ("out_f32", C.c_void_p), ("ldo32", C.c_int64),
    ]


class LiftArgs(C.Structure):
    _fields_ = [
        ("xin", C.c_void_p),
        ("sigma", C.c_void_p), ("sigma_stride", C.c_int32), ("sigma_data", C.c_float),
        ("w", C.c_void_p), ("b", C.c_void_p),
        ("clouds", C.c_int32), ("rows_per_cloud", C.c_int32), ("valid_rows", C.c_int32), ("c", C.c_int32),
        ("x", C.c_void_p), ("ldx", C.c_int64),
        ("x_bf16", C.c_void_p), ("ldxb", C.c_int64),
        ("stats", C.c_void_p), ("stat_gs", C.c_int32),
    ]


class FoldAdaGNArgs(C.Structure):
    _fields_ = [
        ("w", C.c_void_p), ("ldw", C.c_int64),
        ("bias", C.c_void_p),
        ("n_out", C.c_int32), ("c", C.c_int32),
        ("stats", C.c_void_p), ("stat_gs", C.c_int32), ("groups", C.c_int32), ("valid_rows", C.c_int32), ("eps", C.c_float),
        ("t", C.c_void_p), ("t_stride", C.c_int32), ("ctx_dim", C.c_int32),
        ("scale_w", C.c_void_p), ("scale_b", C.c_void_p), ("bias_w", C.c_void_p), ("bias_b", C.c_void_p),
        ("clouds", C.c_int32),
        ("w_folded_bf16", C.c_void_p), ("ldwf", C.c_int64), ("wf_cloud_stride", C.c_int64),
        ("bias_folded", C.c_void_p), ("bias_stride", C.c_int32),
    ]


class HeadArgs(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("ldx", C.c_int64),
        ("clouds", C.c_int32), ("rows_per_cloud", C.c_int32), ("valid_rows", C.c_int32), ("c", C.c_int32),
        ("norm", C.c_int32), ("groups", C.c_int32), ("stats", C.c_void_p), ("stat_gs", C.c_int32), ("eps", C.c_float),
        ("w_out", C.c_void_p), ("b_out", C.c_void_p),
        ("xin", C.c_void_p),
        ("sigma", C.c_void_p), ("sigma_stride", C.c_int32), ("sigma_data", C.c_float),
        ("mode", C.c_int32),
        ("out_f32", C.c_void_p),
        ("x_hat", C.c_void_p), ("x_next", C.c_void_p), ("d_cur", C.c_void_p), ("xin_next", C.c_void_p),
        ("noise_next", C.c_void_p),
        ("t_hat", C.c_double), ("t_next", C.c_double), ("churn_next", C.c_double),
    ]


MAX_LEVELS = 4


class LookupArgs(C.Structure):
    _fields_ = [
        ("xin", C.c_void_p),
        ("sigma", C.c_void_p), ("sigma_stride", C.c_int32), ("sigma_data", C.c_float),
        ("reparam", C.c_int32),
        ("mean", C.c_float * 3), ("sigma_r", C.c_float * 3), ("logit_scale", C.c_float),
        ("K", C.c_void_p),
        ("n_levels", C.c_int32),
        ("level_ptr", C.c_void_p * MAX_LEVELS),
        ("level_h", C.c_int32 * MAX_LEVELS), ("level_w", C.c_int32 * MAX_LEVELS), ("level_c", C.c_int32 * MAX_LEVELS),
        ("clouds", C.c_int32), ("points", C.c_int32), ("rows_per_cloud", C.c_int32),
        ("out_bf16", C.c_void_p), ("ldo16", C.c_int64),
        ("out_f32", C.c_void_p), ("ldo32", C.c_int64),
        ("stats", C.c_void_p), ("stat_groups", C.c_int32),
    ]


class PoolArgs(C.Structure):
    _fields_ = [
        ("kv", C.c_void_p), ("ld", C.c_int64), ("k_off", C.c_int32), ("v_off", C.c_int32),
        ("clouds", C.c_int32), ("rows_per_cloud", C.c_int32), ("valid_rows", C.c_int32),
        ("heads", C.c_int32), ("head_dim", C.c_int32), ("inducers", C.c_int32),
        ("q_inducers", C.c_void_p),
        ("splits", C.c_int32), ("partial", C.c_void_p),
        ("out_bf16", C.c_void_p), ("ldo", C.c_int64),
    ]


class UnpoolArgs(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("ldq", C.c_int64),
        ("kv", C.c_void_p), ("ldkv", C.c_int64), ("v_off", C.c_int32),
        ("clouds", C.c_int32), ("rows_per_cloud", C.c_int32),
        ("heads", C.c_int32), ("head_dim", C.c_int32), ("inducers", C.c_int32),
        ("out_bf16", C.c_void_p), ("ldo", C.c_int64),
        ("vt_scratch", C.c_void_p),
        ("vt_ready", C.c_int32),
    ]


MAX_LAYERS = 32
NW_COUNT = 6
LW_COUNT = 33


class ChainArgs(C.Structure):
    _fields_ = [
        ("clouds", C.c_int32), ("inducers", C.c_int32), ("c", C.c_int32), ("hidden", C.c_int32), ("heads", C.c_int32),
        ("groups", C.c_int32),
        ("first_stage", C.c_int32),
        ("partial", C.c_void_p), ("splits", C.c_int32),
        ("pooled", C.c_void_p),
        ("w_pool_out", C.c_void_p), ("w_mlp0", C.c_void_p), ("w_mlp2", C.c_void_p), ("w_kv", C.c_void_p),
        ("b_mlp0", C.c_void_p), ("b_mlp2", C.c_void_p), ("b_kv", C.c_void_p),
        ("act_alpha", C.c_float),
        ("norm", (C.c_void_p * 4) * 2),
        ("t", C.c_void_p), ("t_stride", C.c_int32), ("eps", C.c_float),
        ("hn", C.c_void_p), ("hh", C.c_void_p), ("h3", C.c_void_p), ("khv", C.c_void_p), ("vt", C.c_void_p),
        ("cache_out", C.c_void_p),
        ("act", C.c_int32),
    ]


class ModelDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("n_layers", C.c_int32), ("feature_dim", C.c_int32), ("num_heads", C.c_int32), ("num_inducers", C.c_int32),
        ("mlp_hidden", C.c_int32),
        ("adagn_groups", C.c_int32),
        ("head_norm", C.c_int32),
        ("head_groups", C.c_int32),
        ("img_groups", C.c_int32),
        ("n_levels", C.c_int32), ("level_c", C.c_int32 * MAX_LEVELS),
        ("reparam", C.c_int32),
        ("mean", C.c_float * 3), ("sigma", C.c_float * 3), ("logit_scale", C.c_float),
        ("sigma_data", C.c_float),
        ("mlp_act", C.c_int32),
    ]


class Context(C.Structure):
    _fields_ = [
        ("level_ptr", C.c_void_p * MAX_LEVELS),
        ("level_h", C.c_int32 * MAX_LEVELS), ("level_w", C.c_int32 * MAX_LEVELS),
        ("K", C.c_void_p),
    ]


class DenoiseArgs(C.Structure):
    _fields_ = [
        ("x", C.c_void_p),
        ("sigma", C.c_void_p), ("sigma_stride", C.c_int32), ("sigma_imm", C.c_float),
        ("t_embed", C.c_void_p), ("t_stride", C.c_int32),
        ("clouds", C.c_int32), ("points", C.c_int32),
        ("ctx", Context),
        ("cache_in", C.c_void_p), ("cache_out", C.c_void_p),
        ("mode", C.c_int32),
        ("out", C.c_void_p),
        ("x_hat", C.c_void_p), ("x_next", C.c_void_p), ("d_cur", C.c_void_p), ("xin_next", C.c_void_p),
        ("noise_next", C.c_void_p),
        ("t_hat", C.c_double), ("t_next", C.c_double), ("churn_next", C.c_double),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64),
    ]


class SampleArgs(C.Structure):
    _fields_ = [
        ("clouds", C.c_int32), ("points", C.c_int32), ("num_steps", C.c_int32),
        ("host_t_steps", C.POINTER(C.c_double)), ("host_gamma", C.POINTER(C.c_double)), ("s_noise", C.c_double),
        ("latents", C.c_void_p), ("noise", C.c_void_p),
        ("ctx", Context),
        ("x_out", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64),
    ]


class UpsampleStepArgs(C.Structure):
    _fields_ = [
        ("clouds", C.c_int32), ("seed_points", C.c_int32), ("new_points", C.c_int32), ("num_substeps", C.c_int32),
        ("last_step", C.c_int32),
        ("t_cur", C.c_double), ("t_next", C.c_double), ("gamma", C.c_double), ("s_noise", C.c_double),
        ("seed_data", C.c_void_p), ("seed_noise", C.c_void_p), ("noise", C.c_void_p),
        ("x", C.c_void_p),
        ("ctx", Context),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64),
    ]


CHAMFER_ALL, CHAMFER_PAIRED, CHAMFER_SELF = 0, 1, 2


class ChamferArgs(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("ma", C.c_int32), ("na", C.c_int32),
        ("b", C.c_void_p), ("mb", C.c_int32), ("nb", C.c_int32),
        ("mode", C.c_int32),
        ("out", C.c_void_p),
    ]


class NearestArgs(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("y", C.c_void_p),
        ("clouds", C.c_int32), ("nx", C.c_int32), ("ny", C.c_int32),
        ("dist_xy", C.c_void_p), ("idx_xy", C.c_void_p),
        ("dist_yx", C.c_void_p), ("idx_yx", C.c_void_p),
        ("scratch", C.c_void_p), ("scratch_bytes", C.c_int64),
    ]


class EmdExactArgs(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("ma", C.c_int32), ("na", C.c_int32),
        ("b", C.c_void_p), ("mb", C.c_int32), ("nb", C.c_int32),
        ("mode", C.c_int32),
        ("out", C.c_void_p),
        ("lower", C.c_void_p),
        ("match", C.c_void_p),
    ]


class ProfileEntry(C.Structure):
    _fields_ = [("name", C.c_char * 32), ("launches", C.c_int64), ("ms", C.c_double), ("flops", C.c_double),
                ("bytes", C.c_double)]


def lib_path() -> Path:
    return _LIB_PATH


def load() -> C.CDLL:
    """Loads libgecco_b200.so (building it first if GECCO_B200_AUTOBUILD=1 and it is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        if os.environ.get("GECCO_B200_AUTOBUILD", "0") == "1":
            from . import build as _build

            _build.build()
        else:
            raise GeccoError(
                f"{_LIB_PATH} is missing: build it with `python -m gecco_b200.build` "
                "(gecco_b200 has no CPU or PyTorch fallback)"
            )
    lib = C.CDLL(str(_LIB_PATH))
    lib.gecco_last_error.restype = C.c_char_p
    lib.gecco_abi_version.restype = C.c_int
    lib.gecco_workspace_bytes.restype = C.c_int64
    lib.gecco_workspace_bytes.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    lib.gecco_launch_count.restype = C.c_int64
    lib.gecco_create.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gecco_destroy.argtypes = [C.c_void_p]
    lib.gecco_denoise.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gecco_sample.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gecco_upsample_workspace_bytes.restype = C.c_int64
    lib.gecco_upsample_workspace_bytes.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32]
    lib.gecco_upsample_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gecco_graph_status.argtypes = [C.c_void_p]
    lib.gecco_adam_ema_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_double,
                                        C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_void_p]
    lib.gecco_train_gauss_act_fwd.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]
    lib.gecco_train_gauss_act_bwd.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]
    lib.gecco_train_affine.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                       C.c_int32, C.c_void_p]
    lib.gecco_train_gauss_act_bwd_parts.argtypes = [C.c_int64]
    lib.gecco_train_gauss_act_bwd_parts.restype = C.c_int64
    lib.gecco_train_colsum2_parts.argtypes = [C.c_int32, C.c_int32]
    lib.gecco_train_colsum2_parts.restype = C.c_int32
    lib.gecco_train_colsum2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    lib.gecco_graph_status.restype = C.c_int
    lib.gecco_chamfer.argtypes = [C.c_void_p, C.c_void_p]
    lib.gecco_emd.argtypes = [C.c_void_p, C.c_void_p]
    lib.gecco_emd_exact.argtypes = [C.c_void_p, C.c_void_p]
    lib.gecco_nearest.argtypes = [C.c_void_p, C.c_void_p]
    lib.gecco_nearest_scratch_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int32]
    lib.gecco_nearest_scratch_bytes.restype = C.c_int64
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().gecco_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError(f"gecco_b200: {msg}")
        raise GeccoError(f"gecco_b200 (code {rc}): {msg}")


def init(device_index: int) -> C.CDLL:
    lib = load()
    if device_index not in _inited_devices:
        check(lib.gecco_init(C.c_int(device_index)))
        _inited_devices.add(device_index)
    return lib
