"""ctypes binding of libtinycarlo_b200.so (include/tinycarlo_b200.h). Raw device pointers and a cudaStream_t go
across the boundary; torch only owns the memory and the stream. There is no fallback: if the library is missing or a
call fails, an exception is raised."""
import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.environ.get("TC_LIB") or os.path.join(LIB_DIR, "libtinycarlo_b200.so")   # TC_LIB: A/B test another build
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-fmad=false",
              "-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared"]

TC_SF_N, TC_SI_N, TC_CP_N, TC_CAM_N, TC_RNG_N = 8, 16, 8, 20, 5
TC_OBS_CLASSES, TC_OBS_RGB, TC_OBS_CLASSES_BITS, TC_OBS_CLASSES_BF16 = 0, 1, 2, 3


class TinyCarloError(RuntimeError):
    pass


class TcMapDesc(C.Structure):
    _fields_ = [("n_classes", C.c_int32), ("ll_node_off", C.c_void_p), ("ll_edge_off", C.c_void_p), ("ll_nodes", C.c_void_p),
                ("ll_edges", C.c_void_p), ("ll_colors", C.c_void_p), ("lp_n_nodes", C.c_int32), ("lp_n_edges", C.c_int32),
                ("lp_nodes", C.c_void_p), ("lp_edges", C.c_void_p), ("lp_orient", C.c_void_p), ("lp_orient_rev", C.c_void_p)]


class TcSimDesc(C.Structure):
    _fields_ = [("height", C.c_int32), ("width", C.c_int32), ("obs_format", C.c_int32)]


class TcBevDesc(C.Structure):
    _fields_ = [("height", C.c_int32), ("width", C.c_int32), ("pixel_per_meter", C.c_double), ("car_col", C.c_double),
                ("car_row", C.c_double), ("line_thickness", C.c_int32), ("route", C.c_int32), ("format", C.c_int32)]


OUTPUT_FIELDS = ["obs", "cte", "heading_error", "velocity", "reward", "position", "orientation", "laneline_distances",
                 "nearest_edge", "local_path", "local_path_nodes", "path_len", "terminated", "truncated", "info_f64", "seg_count",
                 "seg_i32"]


class TcOutputs(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in OUTPUT_FIELDS]


def sources():
    """Every file the library is compiled from (csrc/* and the public header)."""
    files = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h")))
    return files + [os.path.join(ROOT, "include", "tinycarlo_b200.h")]


def source_hash():
    """sha256 over the sources and the compiler flags (16 hex digits): compiled into the library (tc_build_info) so that
    a stale prebuilt .so is detected whatever the file times say."""
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for f in sources():
        h.update(os.path.basename(f).encode())
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def built_hash(path=None):
    """The source hash the library at `path` was compiled from (None: no library / an old one without tc_build_info)."""
    path = path or LIB_PATH
    if not os.path.exists(path):
        return None
    try:
        L = C.CDLL(path)
        L.tc_build_info.restype = C.c_char_p
        return L.tc_build_info().decode()
    except (OSError, AttributeError):
        return None


def build(force=False, verbose=False):
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> tinycarlo_b200/lib/libtinycarlo_b200.so (in-tree). Rebuilds when
    the library is missing or was compiled from other sources (hash check); safe when several ranks call it at once
    (file lock, atomic rename)."""
    want = source_hash()
    if not force and built_hash() == want:
        return LIB_PATH
    import fcntl
    os.makedirs(LIB_DIR, exist_ok=True)
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not force and built_hash() == want:   # another rank built it while we waited
            return LIB_PATH
        tmp = LIB_PATH + f".tmp{os.getpid()}"
        cmd = ["nvcc"] + NVCC_FLAGS + [f'-DTC_SRC_HASH="{want}"', "-o", tmp, os.path.join(CSRC, "tc_api.cu")]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
        os.replace(tmp, LIB_PATH)
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if os.environ.get("TC_LIB"):
        pass   # an explicitly chosen build is loaded as it is
    else:
        try:
            build()   # no-op when the prebuilt library matches the sources
        except Exception as e:  # no silent fallback
            raise TinyCarloError(f"libtinycarlo_b200.so is missing or stale and could not be built with nvcc: {e}") from e
    L = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.tc_abi_version.restype = C.c_int
    L.tc_last_error.restype = C.c_char_p
    L.tc_build_info.restype = C.c_char_p
    L.tc_create.argtypes = [C.POINTER(TcMapDesc), C.POINTER(TcSimDesc), i32, i32, C.POINTER(vp)]
    L.tc_create_rig.argtypes = [C.POINTER(TcMapDesc), C.POINTER(TcSimDesc), i32, i32, i32, C.POINTER(vp)]
    L.tc_destroy.argtypes = [vp]
    L.tc_set_car_params.argtypes = [vp, vp, vp]
    L.tc_set_camera_params.argtypes = [vp, vp, vp, vp]
    L.tc_set_camera_params_host.argtypes = [vp, vp, vp, vp, vp]
    L.tc_debug_cull_stats.argtypes = [vp, C.POINTER(C.c_double)]
    L.tc_set_wrapped.argtypes = [vp, i32]
    L.tc_set_autoreset.argtypes = [vp, vp]
    L.tc_set_reset_mask.argtypes = [vp, vp]
    L.tc_set_bev.argtypes = [vp, C.POINTER(TcBevDesc), vp]
    L.tc_render_bev.argtypes = [vp, vp, vp]
    L.tc_set_spawn_rng.argtypes = [vp, vp, vp, i32, vp]
    L.tc_debug_set_timeline.argtypes = [vp, vp]
    L.tc_debug_cull_info.argtypes = [vp, C.POINTER(C.c_double)]
    L.tc_debug_render_info.argtypes = [vp, C.POINTER(i32)]
    L.tc_episode_stats.argtypes = [vp, vp, vp, i32, vp, vp]
    L.tc_noise_blobs.argtypes = [vp, vp, C.c_uint64, C.c_uint32, i32, i32, i32, vp, vp]
    L.tc_reset.argtypes = [vp, vp, vp, C.POINTER(TcOutputs), vp]
    L.tc_step.argtypes = [vp, vp, vp, C.POINTER(TcOutputs), vp]
    L.tc_step_f64.argtypes = [vp, vp, vp, C.POINTER(TcOutputs), vp]
    L.tc_render.argtypes = [vp, vp, vp, i32, vp, vp, vp]
    L.tc_get_state.argtypes = [vp, vp, vp, vp]
    L.tc_set_state.argtypes = [vp, vp, vp, vp]
    L.tc_step_host.argtypes = [vp, vp, vp, C.POINTER(TcOutputs), vp, vp, vp, vp, vp, vp]
    L.tc_step_host_obs.argtypes = [vp, vp, vp, C.POINTER(TcOutputs), vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
    L.tc_launch_count.argtypes = [vp]
    L.tc_launch_count.restype = i64
    L.tc_profile_begin.argtypes = [vp, i32]
    L.tc_profile_end.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(i32)]
    L.tc_debug_layer_query.argtypes = [vp, i32, C.c_double, C.c_double, C.c_double, i32, i32, vp, vp, vp]
    for name in ("tc_episode_stats", "tc_set_camera_params_host", "tc_debug_cull_stats", "tc_debug_render_info", "tc_step_host_obs", "tc_set_reset_mask", "tc_debug_cull_info", "tc_set_spawn_rng", "tc_noise_blobs", "tc_step_f64", "tc_debug_set_timeline", "tc_set_autoreset", "tc_set_bev", "tc_render_bev", "tc_create", "tc_create_rig", "tc_destroy", "tc_set_car_params", "tc_set_camera_params", "tc_set_wrapped", "tc_reset", "tc_step",
                 "tc_render", "tc_get_state", "tc_set_state", "tc_step_host", "tc_debug_layer_query", "tc_profile_begin", "tc_profile_end"):
        getattr(L, name).restype = C.c_int
    if L.tc_abi_version() != 1:
        raise TinyCarloError("libtinycarlo_b200.so ABI version mismatch")
    _lib = L
    return L


def build_info() -> str:
    """Source hash the loaded library was compiled from (bench.py prints it next to its numbers)."""
    return lib().tc_build_info().decode()


def check(rc, what):
    if rc != 0:
        msg = lib().tc_last_error()
        raise TinyCarloError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")
