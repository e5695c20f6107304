"""ctypes binding of the C-ABI shared library (include/hrl_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` (``_cabi.build``) with nvcc for
sm_100a.  There is NO fallback: if the library is missing or no CUDA device is present the
calls raise.
"""
import ctypes as C
import os
import subprocess

from .config import HrlConfig

_HERE = os.path.dirname(os.path.abspath(__file__))
# HRL_B200_LIB selects another build of the SAME sources (A/B runs: `_cabi.build(defines=..., out=...)`, tools/gpu_round.sh)
LIB_PATH = os.environ.get("HRL_B200_LIB") or os.path.join(_HERE, "libhrl_b200.so")
SRC_DIR = os.path.join(_HERE, "csrc")
INCLUDE_DIR = os.path.join(os.path.dirname(_HERE), "include")
_lib = None

# -prec-div / -prec-sqrt off: fp32 divisions and square roots become MUFU + one Newton step (2 ulp) without their IEEE
# slow paths - fewer instruction bytes per launch (43.9 -> 43.15 us), every parity test unchanged; float64 (the sensor
# decisions, the lidar) is not affected by these switches
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-shared",
              "-Xcompiler", "-fPIC", "-prec-div=false", "-prec-sqrt=false"]

# every symbol include/hrl_b200.h declares (checked by tests/test_cabi_symbols.py)
SYMBOLS = ["hrl_default_config", "hrl_obs_dim", "hrl_act_dim", "hrl_create", "hrl_destroy", "hrl_reset", "hrl_step",
           "hrl_step_host", "hrl_set_host_mode", "hrl_host_layout", "hrl_get_state", "hrl_set_state", "hrl_observe", "hrl_gather_sensor", "hrl_sense_walls", "hrl_gae",
           "hrl_obs_moments", "hrl_reward_scale", "hrl_substeps", "hrl_rollout_mlp", "hrl_rollout_mlp_ex", "hrl_rollout_mlp_norm", "hrl_evaluate_mlp", "hrl_flagrun_next_target", "hrl_get_stats", "hrl_stream_gate", "hrl_set_lanes_per_env", "hrl_get_lanes_per_env", "hrl_set_compact_rows",
           "hrl_get_compact_rows", "hrl_launch_count", "hrl_last_error", "hrl_version"]


class HrlError(RuntimeError):
    pass


def build(force=False, verbose=False, defines=None, out=None):
    """nvcc -> hrl_pybullet_envs_b200/libhrl_b200.so (cross-compiles without a GPU).
    `defines` (e.g. {"HRL_ENVS_PER_WARP": 4}) and `out` build a tuning variant beside it."""
    out = out or LIB_PATH
    srcs = [os.path.join(SRC_DIR, f) for f in os.listdir(SRC_DIR)] + [os.path.join(INCLUDE_DIR, "hrl_b200.h")]
    if not force and os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in srcs):
        return out
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = "nvcc"
    dflags = ["-D%s=%s" % kv for kv in sorted((defines or {}).items())]
    cmd = [nvcc] + NVCC_FLAGS + dflags + (["-Xptxas", "-v"] if verbose else []) + ["-o", out, os.path.join(SRC_DIR, "hrl_b200.cu")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise HrlError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return out


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise HrlError("%s not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(no CPU fallback exists)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32, f32 = C.c_void_p, C.c_int32, C.c_float
    L.hrl_default_config.argtypes = [i32, i32, C.POINTER(HrlConfig)]
    L.hrl_obs_dim.argtypes = [C.POINTER(HrlConfig)]
    L.hrl_act_dim.argtypes = [C.POINTER(HrlConfig)]
    L.hrl_create.argtypes = [C.POINTER(HrlConfig), i32, C.POINTER(vp)]
    L.hrl_destroy.argtypes = [vp]
    L.hrl_reset.argtypes = [vp, vp, vp, vp]
    L.hrl_step.argtypes = [vp] + [vp] * 7
    L.hrl_step_host.argtypes = [vp] + [vp] * 6
    L.hrl_set_host_mode.argtypes = [vp, i32]
    L.hrl_host_layout.argtypes = [C.POINTER(HrlConfig)] + [C.POINTER(C.c_size_t)] * 4
    L.hrl_get_state.argtypes = [vp, vp, vp, vp]
    L.hrl_set_state.argtypes = [vp, vp, vp, vp]
    L.hrl_observe.argtypes = [vp, vp, vp]
    L.hrl_gather_sensor.argtypes = [i32, i32, f32, f32, vp, vp, vp, vp, vp, vp, vp]
    L.hrl_sense_walls.argtypes = [i32, i32, f32, f32, i32, vp, vp, vp, vp, vp]
    L.hrl_gae.argtypes = [i32, i32, f32, f32] + [vp] * 8
    L.hrl_substeps.argtypes = [vp, vp, i32, vp]
    L.hrl_rollout_mlp.argtypes = [vp, i32, vp, i32, f32, C.c_uint64, vp, vp, vp, vp, vp]
    L.hrl_rollout_mlp_ex.argtypes = [vp, i32, vp, i32, f32, vp, C.c_uint64, vp, vp, vp, vp, vp, vp, vp]
    L.hrl_rollout_mlp_norm.argtypes = [vp, i32, vp, i32, f32, vp, C.c_uint64, vp, vp, f32, vp, vp, vp, vp, vp, vp, vp]
    L.hrl_evaluate_mlp.argtypes = [vp, i32, i32, vp, i32, f32, vp, C.c_uint64, vp, vp, f32, vp, vp, vp, vp]
    L.hrl_obs_moments.argtypes = [i32, i32, vp, vp, f32, vp, vp, vp]
    L.hrl_reward_scale.argtypes = [i32, i32, f32, f32, f32] + [vp] * 7
    L.hrl_flagrun_next_target.argtypes = [vp, vp, vp]
    L.hrl_get_stats.argtypes = [vp, vp, C.c_int]
    L.hrl_set_lanes_per_env.argtypes = [vp, i32]
    L.hrl_get_lanes_per_env.argtypes = [vp]
    L.hrl_set_compact_rows.argtypes = [vp, i32]
    L.hrl_get_compact_rows.argtypes = [vp]
    L.hrl_stream_gate.argtypes = [vp, C.c_uint32, C.c_uint64, vp]
    L.hrl_launch_count.restype = C.c_int64
    L.hrl_last_error.restype = C.c_char_p
    L.hrl_version.restype = C.c_char_p
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise HrlError("hrl_b200 error %d: %s" % (rc, lib().hrl_last_error().decode()))


def default_config(kind, num_envs):
    cfg = HrlConfig()
    check(lib().hrl_default_config(int(kind), int(num_envs), C.byref(cfg)))
    return cfg
