"""Build and load ``libcosk.so`` (the C ABI of include/cosk.h) and bind it with ctypes.

The product path has no fallback: if the library is missing and cannot be built, or no CUDA
device is present when a model is stepped, a ``CoskError`` is raised.
"""
import ctypes
import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
ROOT = os.path.dirname(PKG_DIR)
MAX_BLOCKS = 16
ABI_VERSION = 3

NVCC_FLAGS = [
    "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3",
    "-std=c++17",
]


class CoskError(RuntimeError):
    pass


class BlockCfg(ctypes.Structure):
    _fields_ = [("cin", ctypes.c_int32), ("cout", ctypes.c_int32), ("stride", ctypes.c_int32), ("res_kind", ctypes.c_int32),
                ("gconv", ctypes.c_int32)]


class Config(ctypes.Structure):
    _fields_ = [
        ("abi_version", ctypes.c_int32), ("vertices", ctypes.c_int32), ("persons", ctypes.c_int32),
        ("c_in", ctypes.c_int32), ("n_blocks", ctypes.c_int32), ("padding", ctypes.c_int32),
        ("classes", ctypes.c_int32), ("pool_size", ctypes.c_int32), ("pool_padding", ctypes.c_int32),
        ("data_bn", ctypes.c_int32), ("device", ctypes.c_int32), ("path", ctypes.c_int32),
        ("blocks", BlockCfg * MAX_BLOCKS),
    ]


class StreamMeta(ctypes.Structure):
    """cosk_stream_meta: what an exported stream payload was taken from."""
    _fields_ = [("abi_version", ctypes.c_int32), ("geometry", ctypes.c_uint64), ("frame", ctypes.c_int64)]


def library_path():
    return os.path.join(CSRC, "libcosk.so")


def _sources():
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh"))] + [
        os.path.join(ROOT, "include", "cosk.h")
    ]


def _fresh(out):
    return os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in _sources())


def build_library(force=False, verbose=False):
    """nvcc cross-compiles for sm_100a; no GPU needed.  Rebuilds when a source is newer.

    Safe under concurrency (N ranks of one job importing the package at once): the build runs under an exclusive file
    lock, a rank that waited re-checks freshness instead of building again, the compiler writes to a per-process
    temporary and the result is moved into place atomically -- no rank can ever dlopen a half-written library."""
    import fcntl

    out = library_path()
    if not force and _fresh(out):
        return out
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise CoskError("nvcc not found: cannot build libcosk.so")
    with open(os.path.join(CSRC, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and _fresh(out):  # another process built it while this one waited
                return out
            tmp = f"{out}.{os.getpid()}.tmp"
            cmd = [nvcc] + NVCC_FLAGS + ["-o", tmp, os.path.join(CSRC, "cosk.cu")]
            if os.environ.get("COSK_WITH_AGCNT") == "1":  # the unverified channel-major dense mix (csrc/tc_agcnt.cuh), +2 min
                cmd.insert(1, "-DCOSK_WITH_AGCNT")
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                if os.path.exists(tmp):
                    os.remove(tmp)
                raise CoskError("nvcc failed:\n" + r.stdout + r.stderr)
            os.replace(tmp, out)
            if verbose:
                print(r.stderr)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return out


# name -> (restype, argtypes); every symbol include/cosk.h declares
_P = ctypes.c_void_p
SYMBOLS = {
    "cosk_create": (ctypes.c_int, [ctypes.POINTER(Config), ctypes.POINTER(_P)]),
    "cosk_destroy": (None, [_P]),
    "cosk_load_weights": (ctypes.c_int, [_P, ctypes.c_char_p, _P, ctypes.c_size_t]),
    "cosk_set_batch": (ctypes.c_int, [_P, ctypes.c_int64]),
    "cosk_set_batch_ex": (ctypes.c_int, [_P, ctypes.c_int64, ctypes.c_int32]),
    "cosk_reset": (ctypes.c_int, [_P]),
    "cosk_step": (ctypes.c_int, [_P, _P, ctypes.c_int64, _P, ctypes.POINTER(ctypes.c_int32), _P]),
    "cosk_steps": (ctypes.c_int, [_P, _P, ctypes.c_int32, _P, ctypes.c_int64, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32), _P]),
    "cosk_steps_ex": (ctypes.c_int, [_P, _P, ctypes.c_int32, _P, ctypes.c_int64, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32), _P,
                                     ctypes.c_int32]),
    "cosk_state_bytes": (ctypes.c_int64, [_P]),
    "cosk_last_schedule": (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_int32), ctypes.c_int32]),
    "cosk_simulate_schedule": (ctypes.c_int, [ctypes.POINTER(Config), ctypes.c_int32, ctypes.POINTER(ctypes.c_int32)]),
    "cosk_schedule_compatible": (ctypes.c_int, [ctypes.POINTER(Config), ctypes.c_int64, ctypes.c_int64]),
    "cosk_frame_count": (ctypes.c_int64, [_P]),
    "cosk_stream_bytes": (ctypes.c_int64, [_P]),
    "cosk_reset_streams": (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_int64), ctypes.c_int64, _P]),
    "cosk_export_streams": (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_int64), ctypes.c_int64, _P, ctypes.POINTER(StreamMeta), _P]),
    "cosk_import_streams": (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_int64), ctypes.c_int64, _P, ctypes.POINTER(StreamMeta), _P]),
    "cosk_resize_batch": (ctypes.c_int, [_P, ctypes.c_int64, ctypes.POINTER(ctypes.c_int64)]),
    "cosk_prime_streams": (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_int64), ctypes.c_int64, _P, ctypes.c_int32, ctypes.c_int32, _P]),
    "cosk_read_block": (ctypes.c_int, [_P, ctypes.c_int32, _P, _P]),
    "cosk_launch_count": (ctypes.c_int64, [_P]),
    "cosk_block_uses_tensor_cores": (ctypes.c_int, [_P, ctypes.c_int32]),
    "cosk_profile_enable": (ctypes.c_int, [_P, ctypes.c_int32]),
    "cosk_profile_read": (ctypes.c_int, [_P, ctypes.c_int32, ctypes.c_int32, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64)]),
    "cosk_trace_read": (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_uint64), ctypes.c_int32]),
    "cosk_device_error": (ctypes.c_int, [_P, ctypes.POINTER(ctypes.c_uint32)]),
    "cosk_describe": (ctypes.c_int, [_P, ctypes.c_char_p, ctypes.c_size_t]),
    "cosk_last_error": (ctypes.c_char_p, [_P]),
    "cosk_version": (ctypes.c_char_p, []),
}

_LIB = None


def load_library(build=True):
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if build:
        try:
            path = build_library()
        except CoskError:
            if not os.path.exists(path):
                raise
    if not os.path.exists(path):
        raise CoskError(f"{path} is missing; run __graft_entry__.build()")
    lib = ctypes.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _LIB = lib
    return lib
