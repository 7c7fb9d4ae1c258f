"""ctypes binding of libmbe.so (C ABI declared in include/mbe.h).

There is no CPU fallback: if the CUDA library is missing or cannot be loaded this module
raises, and so does every product entry point that needs it."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MBE_LIB_PATH") or os.path.join(HERE, "csrc", "libmbe.so")

MBE_ABI_VERSION = 2
MODE_FORK, MODE_GYM = 0, 1
HANDLER_CENTRAL, HANDLER_MA = 0, 1
SCHED_RESOURCE_FAIR, SCHED_PROPORTIONAL_FAIR, SCHED_RATE_FAIR = 0, 1, 2
BS_SHARED, BS_PER_ENV = 0, 1
MAX_CLASSES = 16
MAX_UE_CLASSES = 8
FLAG_GENERIC_KERNEL = 1
FLAG_SHARED_TRAJECTORY = 2
PHASE_MOVE, PHASE_PRE, PHASE_CLOCK, PHASE_POST, PHASE_ALL = 1, 2, 4, 8, 15
RENDER_PALETTE = 262


class BsClass(C.Structure):
    _fields_ = [
        ("l0", C.c_double),
        ("k", C.c_double),
        ("l_zero", C.c_double),
        ("d2max", C.c_int32),
        ("log2snr_len", C.c_int32),
        ("rate_lut", C.POINTER(C.c_double)),
        ("log2snr_lut", C.POINTER(C.c_float)),
    ]


class UeClass(C.Structure):
    _fields_ = [("velocity", C.c_double), ("move_d2max", C.c_int32), ("reserved", C.c_int32)]


class Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("device", C.c_int32),
        ("num_envs", C.c_int32),
        ("num_ues", C.c_int32),
        ("num_bs", C.c_int32),
        ("mode", C.c_int32),
        ("handler", C.c_int32),
        ("scheduler", C.c_int32),
        ("bs_layout", C.c_int32),
        ("bs_random_min", C.c_int32),
        ("bs_random_max", C.c_int32),
        ("autoreset", C.c_int32),
        ("reset_rng_episode", C.c_int32),
        ("ep_time", C.c_int32),
        ("move_d2max", C.c_int32),
        ("env_offset", C.c_int64),
        ("seed", C.c_uint64),
        ("width", C.c_double),
        ("height", C.c_double),
        ("velocity", C.c_double),
        ("util_lower", C.c_double),
        ("util_upper", C.c_double),
        ("util_w1", C.c_double),
        ("util_w2", C.c_double),
        ("util_w3", C.c_double),
        ("num_classes", C.c_int32),
        ("flags", C.c_int32),
        ("classes", BsClass * MAX_CLASSES),
        ("bs_class", C.POINTER(C.c_uint8)),
        ("num_ue_classes", C.c_int32),
        ("num_trajectories", C.c_int32),
        ("ue_class", C.POINTER(C.c_uint8)),
        ("ue_classes", UeClass * MAX_UE_CLASSES),
    ]


class Buffers(C.Structure):
    _fields_ = [
        ("pos", C.c_void_p),
        ("wp", C.c_void_p),
        ("t", C.c_void_p),
        ("episode", C.c_void_p),
        ("bs_xy", C.c_void_p),
        ("nbs", C.c_void_p),
        ("conn", C.c_void_p),
        ("assoc", C.c_void_p),
        ("actions", C.c_void_p),
        ("rate", C.c_void_p),
        ("utility", C.c_void_p),
        ("obs", C.c_void_p),
        ("reward", C.c_void_p),
        ("done", C.c_void_p),
        ("metrics", C.c_void_p),
        ("dbg_snr", C.c_void_p),
        ("inj_wp", C.c_void_p),
        ("wp_cnt", C.c_void_p),
        ("inj_k", C.c_int32),
        ("reserved", C.c_int32),
    ]


class RolloutOut(C.Structure):
    """mbe_rollout_out: per-step series [T,E,U] of a fused episode (device pointers, may be NULL)."""

    _fields_ = [("pos", C.c_void_p), ("wp", C.c_void_p), ("assoc", C.c_void_p), ("rate", C.c_void_p),
                ("utility", C.c_void_p)]


class RenderStyle(C.Structure):
    """mbe_render_style: frame size, entity sizes in pixels and the palette (rows: see render.py)."""

    _fields_ = [("height", C.c_int32), ("width", C.c_int32), ("ue_radius", C.c_int32), ("bs_half", C.c_int32),
                ("line_width", C.c_int32), ("palette", (C.c_uint8 * 3) * RENDER_PALETTE)]


class EvolveParams(C.Structure):
    """mbe_evolve_params: Philox seed and generation, tournament size, move step, operator probabilities."""

    _fields_ = [("seed", C.c_uint64), ("generation", C.c_uint32), ("tournament", C.c_int32), ("step", C.c_int32),
                ("reserved", C.c_int32), ("p_cross", C.c_double), ("p_move", C.c_double), ("p_add", C.c_double),
                ("p_del", C.c_double)]


class MapParams(C.Structure):
    """mbe_map_params: grid stride, the map UE's class, UEs sharing the serving BS, low-QoE threshold."""

    _fields_ = [("stride", C.c_int32), ("ue_class", C.c_int32), ("load", C.c_int32), ("reserved", C.c_int32),
                ("threshold", C.c_float)]


# every symbol include/mbe.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("mbe_abi_version", C.c_int, []),
    ("mbe_build_info", C.c_char_p, []),
    ("mbe_last_error", C.c_char_p, []),
    ("mbe_struct_size", C.c_int, [C.c_int]),
    ("mbe_create", C.c_int, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    ("mbe_destroy", None, [C.c_void_p]),
    ("mbe_bind", C.c_int, [C.c_void_p, C.POINTER(Buffers)]),
    ("mbe_reset", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    ("mbe_step", C.c_int, [C.c_void_p, C.c_void_p]),
    ("mbe_step_window", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    ("mbe_stage", C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    ("mbe_channel", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("mbe_observe", C.c_int, [C.c_void_p, C.c_void_p]),
    ("mbe_accumulate_qoe", C.c_int, [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p]),
    ("mbe_rollout", C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_float, C.POINTER(RolloutOut), C.c_void_p]),
    ("mbe_render", C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(RolloutOut), C.c_int,
                             C.POINTER(RenderStyle), C.c_void_p, C.c_void_p]),
    ("mbe_evolve_layouts", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                     C.POINTER(EvolveParams), C.c_void_p, C.c_void_p, C.c_void_p]),
    ("mbe_layout_map", C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(MapParams), C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("mbe_launch_count", C.c_int64, [C.c_void_p]),
    ("mbe_step_kernel_name", C.c_char_p, [C.c_void_p]),
    ("mbe_step_host", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
]

_lib = None


class MbeError(RuntimeError):
    pass


def load():
    """Loads libmbe.so (once). Raises if it is not built -- never falls back to the CPU."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MbeError(
            f"{LIB_PATH} is missing: build it with `python -m mobile_env_gan_b200.csrc.build` "
            "(nvcc, sm_100a). There is no CPU fallback for the step path."
        )
    lib = C.CDLL(LIB_PATH)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)  # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    if lib.mbe_abi_version() != MBE_ABI_VERSION:
        raise MbeError(f"libmbe ABI {lib.mbe_abi_version()} != binding {MBE_ABI_VERSION}")
    for which, struct in enumerate((Config, Buffers, BsClass, UeClass, RolloutOut, RenderStyle, EvolveParams,
                                          MapParams)):
        if lib.mbe_struct_size(which) != C.sizeof(struct):
            raise MbeError(f"struct layout mismatch: {struct.__name__} is {C.sizeof(struct)} bytes here, "
                           f"{lib.mbe_struct_size(which)} in {LIB_PATH}")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise MbeError(load().mbe_last_error().decode())
