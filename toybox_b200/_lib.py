"""Loader for the C-ABI library (include/toybox_b200.h).  The library is built in-tree by `build()`
(nvcc, sm_100a only).  There is no CPU fallback: if the library is missing or no CUDA device is present the
callers raise."""
import ctypes as C
import os
import re
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.environ.get("TBX_LIB_PATH") or os.path.join(_HERE, "libtoybox_b200.so")   # TBX_LIB_PATH: tuning builds
_CSRC = os.path.join(_HERE, "csrc")
_LIB = None

NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-fmad=false",
              "-Xcompiler", "-fPIC,-ffp-contract=off"]
SOURCES = ["tbx_pool.cu", "tbx_direct.cu", "tbx_host.cpp"]
_OBJ = os.path.join(_HERE, "build")
_INC = re.compile(r'^\s*#\s*include\s+"([^"]+)"', re.M)


def _deps(path, seen=None):
    """`path` and every local header it includes, transitively (quoted includes only)."""
    seen = set() if seen is None else seen
    path = os.path.normpath(path)
    if path in seen or not os.path.exists(path):
        return seen
    seen.add(path)
    for inc in _INC.findall(open(path).read()):
        _deps(os.path.join(os.path.dirname(path), inc), seen)
    return seen


def _newer(target, deps):
    return not os.path.exists(target) or any(os.path.getmtime(d) > os.path.getmtime(target) for d in deps)


def build(force=False, verbose=False):
    """Compile toybox_b200/libtoybox_b200.so for sm_100a (cross-compiles without a GPU): one object per translation unit
    under toybox_b200/build/, rebuilt only when the unit or a header it includes changed, compiled in parallel."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = os.environ.get("TBX_NVCC_EXTRA", "").split()          # tuning experiments, e.g. -DTBX_AREA_MIN_CTAS=2
    os.makedirs(_OBJ, exist_ok=True)
    jobs, objs = [], []
    for src in SOURCES:
        path = os.path.join(_CSRC, src)
        obj = os.path.join(_OBJ, os.path.splitext(src)[0] + (".tuned.o" if extra else ".o"))
        objs.append(obj)
        if force or extra or _newer(obj, _deps(path)):
            cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj]
            jobs.append(subprocess.Popen(cmd))
    for j in jobs:
        if j.wait() != 0:
            raise subprocess.CalledProcessError(j.returncode, j.args)
    if jobs or _newer(_SO, objs):
        subprocess.check_call([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", _SO] + objs)
    return _SO


# restype and argtypes of every symbol include/toybox_b200.h declares
vp, i32, u64, sz, cp = C.c_void_p, C.c_int, C.c_uint64, C.c_size_t, C.c_char_p
SIGNATURES = {
    "tbx_last_error": (cp, []),
    "tbx_version": (i32, []),
    "tbx_pool_create": (i32, [cp, i32, i32, cp, C.POINTER(vp)]),
    "tbx_pool_destroy": (i32, [vp]),
    "tbx_frame_width": (i32, [vp]),
    "tbx_frame_height": (i32, [vp]),
    "tbx_n_envs": (i32, [vp]),
    "tbx_device": (i32, [vp]),
    "tbx_legal_actions": (i32, [vp, vp, i32]),
    "tbx_obs_bytes": (sz, [vp, i32, i32, i32]),
    "tbx_seed": (i32, [vp, vp, vp, i32]),
    "tbx_new_game": (i32, [vp, vp, vp]),
    "tbx_step": (i32, [vp, vp, i32, vp, vp, vp, vp, vp]),
    "tbx_step_inputs": (i32, [vp, vp, i32, vp, vp, vp, vp, vp]),
    "tbx_step_random": (i32, [vp, u64, u64, u64, i32, vp, vp, vp, vp, vp]),
    "tbx_check": (i32, [vp, vp]),
    "tbx_render": (i32, [vp, vp, i32, i32, i32, vp]),
    "tbx_read_scalars": (i32, [vp, vp, vp, vp, vp]),
    "tbx_step_host": (i32, [vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp]),
    "tbx_state_to_json": (i32, [vp, vp, i32, C.POINTER(vp)]),
    "tbx_state_from_json": (i32, [vp, vp, i32, C.POINTER(cp)]),
    "tbx_config_to_json": (i32, [vp, C.POINTER(vp)]),
    "tbx_config_from_json": (i32, [vp, cp]),
    "tbx_schema_for_state": (i32, [cp, C.POINTER(vp)]),
    "tbx_schema_for_config": (i32, [cp, C.POINTER(vp)]),
    "tbx_query_json": (i32, [vp, i32, cp, cp, C.POINTER(vp)]),
    "tbx_free_str": (None, [vp]),
    "tbx_stats_read": (i32, [vp, vp, i32, vp]),
    "tbx_stats_read_device": (i32, [vp, vp, vp]),
    "tbx_breakout_columns": (i32, [vp, i32, i32, vp, vp, vp]),
    "tbx_fill_actions": (i32, [vp, vp, u64, u64, u64, vp]),
    "tbx_fill_actions_at": (i32, [vp, vp, u64, u64, vp, vp]),
    "tbx_fill_actions_policy": (i32, [vp, vp, i32, u64, vp]),
    "tbx_field_lookup": (i32, [cp, cp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]),
    "tbx_field_get": (i32, [vp, cp, vp, vp]),
    "tbx_field_set": (i32, [vp, cp, vp, vp, vp]),
    "tbx_wrap_create": (i32, [vp, i32, i32, i32, i32, i32, i32, i32, i32, u64, u64, C.POINTER(vp)]),
    "tbx_wrap_destroy": (i32, [vp]),
    "tbx_wrap_set_stack_mode": (i32, [vp, i32]),
    "tbx_wrap_set_obs_mode": (i32, [vp, i32]),
    "tbx_wrap_set_episode_outputs": (i32, [vp, vp, vp]),
    "tbx_wrap_set_sticky_actions": (i32, [vp, C.c_double, u64]),
    "tbx_wrap_set_time_limit": (i32, [vp, i32, vp]),
    "tbx_wrap_set_final_observations": (i32, [vp, vp]),
    "tbx_wrap_step": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, C.POINTER(i32), vp]),
    "tbx_state_rows": (i32, [vp]),
    "tbx_wrap_state_rows": (i32, [vp]),
    "tbx_state_tables": (i32, [vp, vp, sz, C.POINTER(sz)]),
    "tbx_wrap_state_tables": (i32, [vp, vp, sz, C.POINTER(sz)]),
    "tbx_state_save": (i32, [vp, vp, i32, vp, vp]),
    "tbx_wrap_state_save": (i32, [vp, vp, i32, vp, vp]),
    "tbx_state_load": (i32, [vp, vp, i32, vp, vp, i32, vp, sz, vp]),
    "tbx_wrap_state_load": (i32, [vp, vp, i32, vp, vp, i32, vp, sz, vp]),
}
EXPORTS = sorted(SIGNATURES)


class ToyboxError(RuntimeError):
    pass


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(_SO):
        raise ToyboxError("toybox_b200: %s is missing -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)" % _SO)
    L = C.CDLL(_SO)
    for name, (res, args) in SIGNATURES.items():
        f = getattr(L, name)          # AttributeError here = the header and the library disagree
        f.restype = res
        f.argtypes = args
    _LIB = L
    return L


def check(rc):
    if rc != 0:
        msg = lib().tbx_last_error().decode()
        if rc == 5:
            raise ValueError(msg)            # the reference raises ValueError for a refused action
        raise ToyboxError("toybox_b200 error %d: %s" % (rc, msg))


def take_str(ptr):
    s = C.string_at(ptr).decode()
    lib().tbx_free_str(ptr)
    return s
