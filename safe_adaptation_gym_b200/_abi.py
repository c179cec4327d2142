"""ctypes binding of the C ABI declared in ``include/sag_b200.h``.

The product loads exactly one library: ``csrc/libsag_b200.so`` (built in-tree by ``_build.build()`` /
``__graft_entry__.build()`` with nvcc for sm_100a).  There is no CPU fallback: if the library is missing
or no CUDA device is present, importing the env raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SAG_B200_LIB: build-variant override for tuning experiments (must still be a CUDA build of csrc/sag_kernels.cu)
LIB_PATH = os.environ.get("SAG_B200_LIB") or os.path.join(_HERE, "csrc", "libsag_b200.so")

NUM_TASKS = 14
MAX_SLOTS = 32
MAX_GREMLINS = 4
F_ROBOT, F_OBJECTS, F_TASK_F64, F_TASK_I32, F_FLAGS, F_ROBOT_EXT, F_GREMLINS, F_NEXT_TASK = range(8)
FLAG_PHYSICS_ERROR, FLAG_RESAMPLE_FAILED, FLAG_NEEDS_RESET, ERR_BAD_TASK_ID, ERR_BAD_ENV_INDEX = 1, 2, 4, 8, 16


class SagConfig(C.Structure):
    _fields_ = [
        ("n_envs", C.c_int32), ("robot", C.c_int32), ("seed", C.c_uint64), ("env_id_base", C.c_uint32),
        ("max_episode_steps", C.c_int32), ("max_layout_draws", C.c_int32), ("random_bound", C.c_int32),
        ("placements_margin", C.c_double), ("robot_keepout", C.c_double),
        ("hazards_size", C.c_double), ("vases_size", C.c_double), ("pillars_size", C.c_double), ("gremlins_size", C.c_double),
        ("hazards_keepout", C.c_double), ("gremlins_keepout", C.c_double), ("vases_keepout", C.c_double),
        ("pillars_keepout", C.c_double),
        ("gremlins_travel", C.c_double), ("robot_ctrl_range_scale", C.c_double), ("action_noise", C.c_double),
        ("max_bound", C.c_double),
        ("num_gremlins", C.c_int32), ("reserved_", C.c_int32),
    ]


class SagError(RuntimeError):
    pass


class SagLib:
    """Prototype-checked view of one shared library exporting the sag_* symbols."""

    SYMBOLS = [
        "sag_last_error", "sag_abi_version", "sag_default_config", "sag_create", "sag_destroy", "sag_stride",
        "sag_obs_dim", "sag_field_bytes", "sag_launch_count", "sag_debug_read", "sag_set_tasks", "sag_set_tasks_host", "sag_bound_host",
        "sag_set_next_tasks", "sag_set_next_tasks_host", "sag_bound", "sag_copy_envs", "sag_copy_envs_host",
        "sag_error_flags", "sag_reset_obs", "sag_reset_host", "sag_seed", "sag_reset", "sag_step", "sag_observe",
        "sag_step_host", "sag_observe_host", "sag_host_alloc", "sag_host_alloc_outputs", "sag_probe_d2h", "sag_host_free", "sag_rollout", "sag_read_field",
        "sag_write_field", "sag_task_stats", "sag_lidar", "sag_cost", "sag_export_outputs",
    ]

    def __init__(self, path, host_api=True):
        if not os.path.exists(path):
            raise SagError(
                f"{path} not found: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()'). "
                "There is no CPU fallback.")
        self.path = path
        L = self.L = C.CDLL(path)
        vp, i32, u8p, fp, dp = C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p
        L.sag_last_error.restype = C.c_char_p
        L.sag_abi_version.restype = C.c_int
        L.sag_default_config.argtypes = [C.POINTER(SagConfig)]
        L.sag_create.argtypes = [C.POINTER(SagConfig), i32, C.POINTER(vp)]
        L.sag_destroy.argtypes = [vp]
        L.sag_stride.argtypes = [vp]
        L.sag_obs_dim.argtypes = [vp]
        L.sag_debug_read.argtypes = [vp, vp]
        L.sag_launch_count.restype = C.c_ulonglong
        L.sag_launch_count.argtypes = [vp]
        L.sag_field_bytes.restype = C.c_size_t
        L.sag_field_bytes.argtypes = [vp, i32]
        L.sag_set_tasks.argtypes = [vp, vp, vp]
        # (entry points added after the host emulation of the CPU suite was written: set where the library has them;
        # build() and tests/test_api.py require every SYMBOLS entry of the product library)
        if hasattr(L, "sag_set_next_tasks"):
            L.sag_set_next_tasks.argtypes = [vp, vp, vp]
            L.sag_bound.argtypes = [vp, dp, vp]
        if hasattr(L, "sag_copy_envs"):
            L.sag_copy_envs.argtypes = [vp, vp, vp, vp]
            L.sag_copy_envs_host.argtypes = [vp, vp, vp]
        L.sag_seed.argtypes = [vp, C.c_uint64]
        L.sag_error_flags.argtypes = [vp, i32]
        L.sag_reset_obs.argtypes = [vp, u8p, i32, i32, fp, u8p, vp]
        L.sag_reset.argtypes = [vp, u8p, i32, i32, vp]
        L.sag_step.argtypes = [vp, fp, fp, dp, dp, u8p, u8p, vp]
        L.sag_observe.argtypes = [vp, fp, vp]
        L.sag_rollout.argtypes = [vp, i32, fp, dp, u8p, u8p, vp]
        L.sag_export_outputs.argtypes = [vp, fp, dp, i32, u8p, u8p, dp, fp, dp, fp, u8p, dp, vp]
        L.sag_read_field.argtypes = [vp, i32, vp, vp]
        L.sag_write_field.argtypes = [vp, i32, vp, vp]
        L.sag_task_stats.argtypes = [vp, dp, i32, vp]
        L.sag_lidar.argtypes = [dp, dp, u8p, i32, i32, fp, vp]
        L.sag_cost.argtypes = [dp, fp, u8p, i32, i32, C.c_double, u8p, vp]
        if host_api:
            L.sag_step_host.argtypes = [vp, fp, fp, dp, u8p, u8p]
            L.sag_observe_host.argtypes = [vp, fp]
            L.sag_set_tasks_host.argtypes = [vp, vp]
            L.sag_set_next_tasks_host.argtypes = [vp, vp]
            L.sag_bound_host.argtypes = [vp, dp]
            L.sag_reset_host.argtypes = [vp, u8p, i32, i32, fp]
            L.sag_host_alloc.restype = vp
            L.sag_host_alloc.argtypes = [C.c_size_t]
            L.sag_host_free.argtypes = [vp]
            L.sag_probe_d2h.argtypes = [vp, C.c_size_t, i32, C.POINTER(C.c_double)]
            L.sag_host_alloc_outputs.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]

    def check(self, rc):
        if rc != 0:
            raise SagError(self.L.sag_last_error().decode())

    def default_config(self):
        cfg = SagConfig()
        self.L.sag_default_config(C.byref(cfg))
        return cfg


_lib = None


def load():
    """The product library (CUDA).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        _lib = SagLib(LIB_PATH)
    return _lib
