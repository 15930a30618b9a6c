"""ctypes binding of libcube_b200.so (the C ABI declared in include/cube_b200.h).

There is no CPU fallback: if the CUDA library is missing and cannot be built,
or no CUDA device is usable, every entry point raises.
"""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libcube_b200.so")

SYMBOLS = (
    "cube_abi_version", "cube_last_error", "cube_sm_count", "cube_set_reserved_sms", "cube_moves_from_seeds", "cube_scramble", "cube_scramble_step", "cube_scramble_prefixes", "cube_scramble_prefixes_max_depth", "cube_step", "cube_walk",
    "cube_solved", "cube_encode", "cube_expand", "cube_expand_codes", "cube_adi_targets", "cube_mcts_traverse", "cube_mcts_update", "cube_decode", "cube_validate_actions",
    "cube_peer_buffer_bytes", "cube_peer_allreduce_i64",
    "cube_pipeline_create", "cube_pipeline_destroy", "cube_pipeline_scramble_host", "cube_pipeline_reset_host", "cube_host_alloc", "cube_host_free",
    "cube_env_host_create", "cube_env_host_destroy", "cube_env_host_step", "cube_env_host_scramble", "cube_env_host_encode",
    "cube_distance_table_entries", "cube_distance_table_build", "cube_distance", "cube_solve_optimal",
)

ABI_VERSION = 2
CUBE_ERR_SIZE, CUBE_ERR_ARG, CUBE_ERR_ALIGN, CUBE_ERR_ACTION = -1, -2, -3, -4
DTYPE_BF16, DTYPE_F32, DTYPE_U8 = 0, 1, 2
ENCODING_REFERENCE, ENCODING_EXACT = 0, 1
DISTANCE_UNREACHABLE, DISTANCE_MAX_2 = 255, 14

_lib = None


class CubeLibraryError(RuntimeError):
    pass


def build_library(force=False):
    """Compile the library with nvcc (in-tree).  Used by __graft_entry__.build()."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("_cube_b200_build", os.path.join(_PKG, "csrc", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build(force=force)


def load():
    """Load (building first if the .so is absent and nvcc exists) and type the C ABI."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        try:
            build_library()
        except Exception as exc:  # noqa: BLE001 - reported below, never swallowed
            raise CubeLibraryError(
                "libcube_b200.so is missing and could not be built (%s); run "
                "`python -c 'import __graft_entry__ as g; g.build()'` -- there is no CPU fallback" % (exc,))
    lib = ctypes.CDLL(LIB_PATH)
    vp, i64, ci = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
    lib.cube_abi_version.restype = ci
    lib.cube_last_error.restype = ctypes.c_char_p
    lib.cube_sm_count.restype = ci
    lib.cube_set_reserved_sms.argtypes = [ci]
    lib.cube_moves_from_seeds.argtypes = [ci, vp, i64, ci, vp, vp, vp]
    lib.cube_scramble.argtypes = [ci, vp, i64, ci, vp, vp, vp, vp, vp]
    lib.cube_scramble_step.argtypes = [ci, vp, vp, i64, ci, vp, vp, vp, vp, vp]
    lib.cube_scramble_prefixes.argtypes = [ci, vp, i64, ci, vp, vp, vp, vp]
    lib.cube_scramble_prefixes_max_depth.argtypes = [ci]
    lib.cube_step.argtypes = [ci, vp, vp, i64, vp, vp, vp, vp]
    lib.cube_walk.argtypes = [ci, vp, vp, i64, ci, vp, vp, vp, vp, vp]
    lib.cube_solved.argtypes = [ci, vp, i64, vp, vp, vp, vp]
    lib.cube_encode.argtypes = [ci, vp, i64, vp, ci, ci, vp]
    lib.cube_expand.argtypes = [ci, vp, i64, vp, vp, vp, ci, ci, vp, vp, vp, vp]
    lib.cube_expand_codes.argtypes = [ci, vp, i64, vp, vp, vp, vp, ci, ci, vp, vp, vp, vp]
    lib.cube_adi_targets.argtypes = [ci, vp, vp, vp, vp, vp, ci, i64, vp, vp, vp, vp]
    lib.cube_mcts_traverse.argtypes = [ci, vp, ctypes.c_float, ci, vp]
    lib.cube_mcts_update.argtypes = [ci, vp, vp, vp, vp, vp, vp, ctypes.c_float, ci, vp, vp, vp, vp, vp]
    lib.cube_decode.argtypes = [ci, vp, ci, ci, i64, vp, vp]
    lib.cube_validate_actions.argtypes = [ci, vp, i64, vp, vp]
    lib.cube_peer_buffer_bytes.argtypes = [ci]
    lib.cube_peer_buffer_bytes.restype = i64
    lib.cube_peer_allreduce_i64.argtypes = [ci, ci, vp, vp, ci, ci, ctypes.c_uint32, vp]
    lib.cube_pipeline_create.argtypes = [ci, ci, i64, ci, ctypes.POINTER(vp)]
    lib.cube_pipeline_destroy.argtypes = [vp]
    lib.cube_pipeline_scramble_host.argtypes = [vp, vp, i64, vp, vp, vp, ctypes.POINTER(i64)]
    lib.cube_pipeline_reset_host.argtypes = [vp, vp, i64, vp, vp, vp, ctypes.POINTER(i64)]
    lib.cube_host_alloc.argtypes = [i64, ctypes.POINTER(vp)]
    lib.cube_host_free.argtypes = [vp]
    lib.cube_env_host_create.argtypes = [ci, ci, ctypes.POINTER(vp)]
    lib.cube_env_host_destroy.argtypes = [vp]
    lib.cube_env_host_step.argtypes = [vp, vp, ci, vp, vp, ctypes.POINTER(ci), vp]
    lib.cube_env_host_scramble.argtypes = [vp, vp, ci, vp, vp, ctypes.POINTER(ci), vp]
    lib.cube_env_host_encode.argtypes = [vp, vp, vp, vp]
    lib.cube_distance_table_entries.argtypes = [ci]
    lib.cube_distance_table_build.argtypes = [ci, vp, vp]
    lib.cube_distance.argtypes = [ci, vp, vp, i64, vp, vp]
    lib.cube_solve_optimal.argtypes = [ci, vp, vp, i64, vp, vp, vp]
    for name in SYMBOLS:
        if name not in ("cube_last_error",):
            getattr(lib, name).restype = ci
    lib.cube_distance_table_entries.restype = i64
    if lib.cube_abi_version() != ABI_VERSION:
        raise CubeLibraryError("libcube_b200.so has ABI version %d, expected %d" % (lib.cube_abi_version(), ABI_VERSION))
    _lib = lib
    return lib


def check(rc, what):
    """Map a C-ABI return code to the exception the reference would raise."""
    if rc == 0:
        return
    msg = load().cube_last_error().decode("utf-8", "replace") or what
    if rc == CUBE_ERR_SIZE:
        raise NotImplementedError(msg)                       # cube_env.py:43-44
    if rc == CUBE_ERR_ACTION:
        raise IndexError(msg)                                # cube_env.py:86,96
    if rc in (CUBE_ERR_ARG, CUBE_ERR_ALIGN):
        raise ValueError(msg)
    raise CubeLibraryError(msg)
