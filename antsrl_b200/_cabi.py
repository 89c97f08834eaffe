"""ctypes binding of libantsrl_b200.so (include/antsrl_b200.h).  There is no CPU fallback: if the library is
missing or no CUDA device is present, the product path raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ANTS_LIB") or os.path.join(_HERE, "lib", "libantsrl_b200.so")   # ANTS_LIB: experiment builds

ABI_VERSION = 1
MAX_PHERO, MAX_CHANNELS, MAX_RADIUS, MAX_SAMPLES, MAX_ROCKS, MAX_ANTS = 4, 16, 7, 225, 64, 65535
CH_ANTS, CH_PHERO, CH_ANTHILL, CH_WALLS, CH_FOOD, CH_ROCKS = range(6)
REWARD_ALL, REWARD_EXPLORE, REWARD_FOOD = range(3)
EVAP_DENSE, EVAP_ACTIVE_TILES, EVAP_LAZY = 0, 1, 2
REC_F64, REC_COMPACT, REC_COMPACT8 = 0, 1, 2

EXPORTED_SYMBOLS = [
    "ants_abi_version", "ants_last_error", "ants_create", "ants_destroy", "ants_set_stream", "ants_synchronize",
    "ants_import_state", "ants_export_state", "ants_activate_all_pheromones", "ants_observe", "ants_step",
    "ants_update", "ants_rollout", "ants_host_alloc", "ants_host_free", "ants_observe_host", "ants_step_host",
    "ants_update_host", "ants_get_stats", "ants_set_profiling", "ants_get_kernel_ms", "ants_reset_kernel_ms",
    "ants_sample_actions", "ants_export_env_state", "ants_packed_layout", "ants_step_host_packed", "ants_unpack_obs",
    "ants_import_env_state", "ants_generate_env_maps", "ants_generate_env_maps_ex", "ants_perlin_noise",
]


class AntsConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("device", C.c_int32),
        ("n_envs", C.c_int32), ("n_ants", C.c_int32), ("w", C.c_int32), ("h", C.c_int32),
        ("n_phero", C.c_int32), ("n_rocks", C.c_int32), ("max_time", C.c_int32),
        ("radius", C.c_int32), ("has_mask", C.c_int32), ("mask", C.c_uint8 * MAX_SAMPLES),
        ("n_channels", C.c_int32), ("channel_kind", C.c_int32 * MAX_CHANNELS),
        ("channel_arg", C.c_int32 * MAX_CHANNELS),
        ("delta", C.c_double), ("fwd_delta", C.c_double),
        ("reward_threshold", C.c_double), ("max_speed", C.c_double), ("max_rot_speed", C.c_double),
        ("carry_speed_reduction", C.c_double), ("backward_speed_reduction", C.c_double),
        ("reward_kind", C.c_int32), ("reward_factors", C.c_double * 5),
        ("diffuse_factor", C.c_double), ("evap_factor", C.c_double),
        ("has_max_val", C.c_int32), ("phero_max_val", C.c_double), ("max_hold", C.c_double),
        ("rng_seed", C.c_uint64), ("env_id_base", C.c_int64),
        ("evap_mode", C.c_int32), ("record_format", C.c_int32), ("reserved", C.c_int32 * 6),
    ]


_PD, _PU8, _PI32 = C.POINTER(C.c_double), C.POINTER(C.c_uint8), C.POINTER(C.c_int32)


class AntsHostState(C.Structure):
    _fields_ = [
        ("x", _PD), ("y", _PD), ("theta", _PD), ("prev_x", _PD), ("prev_y", _PD), ("prev_theta", _PD),
        ("holding", _PD), ("seed", _PD), ("activation", _PD),
        ("mandibles", _PU8), ("reward_state", _PU8),
        ("rw_holding_prev", _PD), ("rw_prev_dist", _PD), ("rewards", _PD),
        ("explored", _PU8), ("walls", _PU8), ("phero", _PD), ("food", _PD),
        ("anthill_xyr", _PI32), ("anthill_food", _PD),
        ("rock_centers", _PD), ("rock_radii", _PD), ("rock_weights", _PD),
        ("timestep", C.c_int64), ("rw_alias", C.c_int32), ("act_bool", C.c_int32),
    ]


class AntsStats(C.Structure):
    _fields_ = [("steps", C.c_int64), ("updates", C.c_int64), ("observations", C.c_int64),
                ("kernel_launches", C.c_int64), ("active_tiles", C.c_int64), ("total_tiles", C.c_int64),
                ("food_commits", C.c_int64), ("absorb_events", C.c_int64), ("device_bytes", C.c_int64),
                ("e2e_dense_permille", C.c_int64)]


class AntsPackedLayout(C.Structure):
    _fields_ = [("supported", C.c_int32), ("n_samples", C.c_int32), ("n_channels", C.c_int32), ("n_visible", C.c_int32),
                ("sample_bytes", C.c_int32), ("bytes_per_ant", C.c_int64), ("flag_channel", C.c_int32 * 8),
                ("value_channel", C.c_int32 * 2), ("food_channel", C.c_int32), ("visible_index", C.c_uint8 * 228)]


class AntsPerlinLayer(C.Structure):
    _fields_ = [("offsets", C.POINTER(C.c_int32)), ("scale", C.c_double), ("density", C.c_double),
                ("octaves", C.c_int32), ("reserved", C.c_int32), ("persistence", C.c_double),
                ("lacunarity", C.c_double)]


class AntsError(RuntimeError):
    pass


_lib = None


def load_library(path=None):
    """dlopen the CUDA library.  Raises AntsError if it has not been built (run __graft_entry__.build())."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise AntsError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`; "
                        "antsrl_b200 has no CPU fallback" % path)
    lib = C.CDLL(path)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    lib.ants_abi_version.restype = C.c_int
    lib.ants_last_error.restype = C.c_char_p
    lib.ants_create.argtypes = [C.POINTER(AntsConfig), C.POINTER(vp)]
    lib.ants_destroy.argtypes = [vp]
    lib.ants_set_stream.argtypes = [vp, vp]
    lib.ants_synchronize.argtypes = [vp]
    lib.ants_import_state.argtypes = [vp, C.POINTER(AntsHostState)]
    lib.ants_export_state.argtypes = [vp, C.POINTER(AntsHostState)]
    lib.ants_export_env_state.argtypes = [vp, i32, i32, C.POINTER(AntsHostState)]
    lib.ants_import_env_state.argtypes = [vp, i32, i32, C.POINTER(AntsHostState)]
    lib.ants_generate_env_maps_ex.argtypes = [vp, i32, i32, vp, i32, vp, C.POINTER(AntsPerlinLayer), i32, vp,
                                              C.POINTER(AntsPerlinLayer)]
    lib.ants_perlin_noise.argtypes = [i32, C.POINTER(AntsPerlinLayer), i32, i32, i32, vp, vp]
    lib.ants_activate_all_pheromones.argtypes = [vp, vp, i32]
    lib.ants_observe.argtypes = [vp, vp, vp, vp, vp]
    lib.ants_step.argtypes = [vp, vp, vp, vp, vp, vp, C.POINTER(i32)]
    lib.ants_update.argtypes = [vp, vp]
    lib.ants_rollout.argtypes = [vp, vp, vp, i32, vp, vp, vp]
    lib.ants_sample_actions.argtypes = [vp, C.c_uint64, i32, i32, vp, vp]
    lib.ants_host_alloc.argtypes = [C.c_uint64]
    lib.ants_host_alloc.restype = vp
    lib.ants_host_free.argtypes = [vp]
    lib.ants_observe_host.argtypes = [vp, vp, vp, vp, vp]
    lib.ants_step_host.argtypes = [vp, vp, vp, vp, vp, vp, C.POINTER(i32)]
    lib.ants_update_host.argtypes = [vp, vp]
    lib.ants_packed_layout.argtypes = [C.POINTER(AntsConfig), C.POINTER(AntsPackedLayout)]
    lib.ants_step_host_packed.argtypes = [vp, vp, vp, vp, vp, vp, C.POINTER(i32)]
    lib.ants_unpack_obs.argtypes = [C.POINTER(AntsPackedLayout), vp, i64, vp, i32]
    lib.ants_get_stats.argtypes = [vp, C.POINTER(AntsStats)]
    lib.ants_set_profiling.argtypes = [vp, i32]
    lib.ants_get_kernel_ms.argtypes = [vp, C.c_char_p, C.POINTER(C.c_double), C.POINTER(i64)]
    lib.ants_reset_kernel_ms.argtypes = [vp]
    for name in EXPORTED_SYMBOLS:
        fn = getattr(lib, name)
        if name not in ("ants_last_error", "ants_host_alloc", "ants_abi_version"):
            fn.restype = C.c_int
    if lib.ants_abi_version() != ABI_VERSION:
        raise AntsError("ABI mismatch: library %d, binding %d" % (lib.ants_abi_version(), ABI_VERSION))
    if path == LIB_PATH:
        _lib = lib
    return lib


def check(lib, rc):
    if rc != 0:
        raise AntsError("libantsrl_b200: %s (code %d)" % (lib.ants_last_error().decode("utf-8", "replace"), rc))
