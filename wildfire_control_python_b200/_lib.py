"""ctypes binding of libwildfire_b200.so (include/wildfire.h).

Same FFI style the reference uses for its only native component (pyastar/pyastar.py:9-22:
``ctypes.cdll.LoadLibrary`` + typed ``argtypes``).  There is NO fallback: if the shared library
has not been built (``python -c 'import __graft_entry__ as g; g.build()'`` or
``make -C wildfire_control_python_b200/csrc``) importing this module's ``lib()`` raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("WILDFIRE_B200_LIB") or os.path.join(HERE, "libwildfire_b200.so")  # override: experiments
CSRC = os.path.join(HERE, "csrc")

WF_OK, WF_ERR_INVALID, WF_ERR_CUDA, WF_ERR_STATE = 0, -1, -2, -3
WF_OBS_U8, WF_OBS_F32, WF_OBS_BF16, WF_OBS_BITS = 0, 1, 2, 3
WF_POLICY_STREAM, WF_POLICY_WALK, WF_POLICY_MLP = 0, 1, 2
WF_NSCALARS = 16
(S_ALIVE, S_AX, S_AY, S_DEAD, S_DIGGING, S_VISIBLE, S_RUNNING, S_FIRE_AT_BORDER, S_LATCHED, S_EPISODE, S_T,
 S_WIND_ID, S_WIND_X, S_WIND_Y, S_N_BURNING, S_RESERVED) = range(16)


def obs_bits_words(width: int, height: int) -> int:
    """uint32 words of one env's WF_OBS_BITS observation: ceil(W*H*3 / 32) (include/wildfire.h)."""
    return (int(width) * int(height) * 3 + 31) // 32


class WfConfig(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("n_actions", C.c_int32), ("a_speed", C.c_int32),
        ("allow_dig_toggle", C.c_int32), ("make_rivers", C.c_int32), ("containment_wins", C.c_int32),
        ("wind_random", C.c_int32), ("wind_x", C.c_int32), ("wind_y", C.c_int32), ("fuel", C.c_int32),
        ("radius", C.c_int32), ("extra_ignitions", C.c_int32), ("auto_reset", C.c_int32),
        ("wind_speed", C.c_double), ("death_penalty", C.c_double), ("contained_bonus", C.c_double),
        ("default_reward", C.c_double), ("heat", C.c_double), ("threshold", C.c_double),
        ("seed", C.c_uint64), ("env_id_base", C.c_int64),
    ]


class WfInit(C.Structure):
    _fields_ = [("ax", C.c_int32), ("ay", C.c_int32)]


class WfMlpShape(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("hidden", C.c_int32), ("n_actions", C.c_int32),
                ("dueling", C.c_int32), ("batch", C.c_int32)]


class WfFitParams(C.Structure):
    _fields_ = [("gamma", C.c_double), ("lr", C.c_double), ("beta_1", C.c_double), ("beta_2", C.c_double),
                ("epsilon", C.c_double), ("clipvalue", C.c_double), ("adam_t", C.c_int64), ("target_every", C.c_int32),
                ("phase", C.c_int32)]


class WfFitLearner(C.Structure):
    """``wf_fit_learner``: one learner of ``wf_replay_fit_many`` (device pointers travel as integers)."""
    _fields_ = [("params", C.c_void_p), ("target", C.c_void_p), ("adam_m", C.c_void_p), ("adam_v", C.c_void_p),
                ("s_row", C.c_void_p), ("sp_row", C.c_void_p), ("action", C.c_void_p), ("next_action", C.c_void_p),
                ("reward", C.c_void_p), ("done", C.c_void_p), ("loss", C.c_void_p), ("hp", WfFitParams)]


MAX_LEARNERS = 64  # wf_replay_fit_many's n_learners and wf_set_policy_mlp_nets_dev's n_nets


def mlp_param_count(width: int, height: int, hidden: int, n_actions: int, dueling: bool) -> int:
    """Floats of wf_replay_fit's flat parameter buffer (include/wildfire.h): parameters_to_vector(model.parameters())."""
    n_in = int(width) * int(height) * 3
    n = hidden * (n_in + 1 + n_actions) + n_actions
    return n + (hidden * (n_in + 2) + 1 if dueling else 0)


class WildfireError(RuntimeError):
    pass


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile libwildfire_b200.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "wildfire.h")]
    newest = max(os.path.getmtime(p) for p in srcs)
    if force or not os.path.isfile(LIB_PATH) or os.path.getmtime(LIB_PATH) < newest:
        r = subprocess.run(["make", "-j4", "-C", CSRC], capture_output=True, text=True)
        if verbose or r.returncode != 0:
            print(r.stdout[-4000:], r.stderr[-8000:])
        if r.returncode != 0:
            raise WildfireError("building libwildfire_b200.so failed")
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise WildfireError(
            f"{LIB_PATH} is missing: build it with `make -C {CSRC}` (nvcc, sm_100a). "
            "This package has no CPU or PyTorch fallback.")
    L = C.CDLL(LIB_PATH)
    vp, u8p, i32p, f64p = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p  # device pointers travel as integers
    L.wf_default_config.argtypes = [C.POINTER(WfConfig), C.c_int32]
    L.wf_default_config.restype = None
    L.wf_create.argtypes = [C.POINTER(WfConfig), C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]
    L.wf_destroy.argtypes = [vp]
    L.wf_destroy.restype = None
    L.wf_last_error.restype = C.c_char_p
    L.wf_abi_version.restype = C.c_int
    L.wf_kernel_family.argtypes = [vp]
    L.wf_kernel_family.restype = C.c_char_p
    L.wf_reset.argtypes = [vp, u8p, vp, vp, C.c_int32, vp]
    L.wf_step.argtypes = [vp, i32p, vp, C.c_int32, f64p, u8p, vp]
    L.wf_rollout.argtypes = [vp, C.c_int32, i32p, vp, C.c_int32, f64p, u8p, vp]
    L.wf_rollout_policy.argtypes = [vp, C.c_int32, C.c_int32, i32p, vp, C.c_int32, f64p, u8p, vp]
    L.wf_set_policy_mlp.argtypes = [vp, vp, vp, vp, vp, C.c_int32, C.c_double]
    L.wf_set_policy_mlp_dev.argtypes = [vp, vp, vp, vp, vp, C.c_int32, C.c_double, vp]
    L.wf_set_policy_mlp_dev.restype = C.c_int
    L.wf_replay_fit.argtypes = [C.POINTER(WfMlpShape), C.POINTER(WfFitParams), C.c_int32, vp, vp, vp, vp, vp, C.c_int64,
                                vp, vp, vp, vp, vp, vp, vp, vp]
    L.wf_replay_fit.restype = C.c_int
    L.wf_replay_fit_large.argtypes = L.wf_replay_fit.argtypes
    L.wf_replay_fit_large.restype = C.c_int
    L.wf_replay_fit_many.argtypes = [C.POINTER(WfMlpShape), C.c_int32, C.POINTER(WfFitLearner), C.c_int32, vp, C.c_int64, vp]
    L.wf_replay_fit_many.restype = C.c_int
    L.wf_set_policy_mlp_nets_dev.argtypes = [vp, C.POINTER(WfMlpShape), C.c_int32, vp, C.POINTER(C.c_double), vp]
    L.wf_set_policy_mlp_nets_dev.restype = C.c_int
    L.wf_step_host.argtypes = [vp, i32p, vp, C.c_int32, f64p, u8p]
    L.wf_reset_host.argtypes = [vp, u8p, vp, vp, C.c_int32]
    L.wf_host_session.argtypes = [vp, C.c_int32]
    L.wf_host_session_active.argtypes = [vp]
    L.wf_host_session_active.restype = C.c_int
    L.wf_get_state.argtypes = [vp, u8p, u8p, u8p, u8p, u8p, u8p, i32p, vp]
    L.wf_set_state.argtypes = [vp, u8p, u8p, u8p, u8p, u8p, i32p, vp]
    L.wf_set_fire_to.argtypes = [vp, i32p, vp]
    L.wf_get_a_iter.argtypes = [vp, C.POINTER(C.c_int32)]
    L.wf_set_a_iter.argtypes = [vp, C.c_int32]
    L.wf_get_obs.argtypes = [vp, vp, C.c_int32, vp]
    L.wf_get_wind_table.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int32),
                                    C.POINTER(C.c_int32)]
    L.wf_stats.argtypes = [vp, C.POINTER(C.c_int64), vp]
    L.wf_stats_reset.argtypes = [vp, vp]
    L.wf_philox_kat.argtypes = [C.c_int32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
    L.wf_philox_kat.restype = C.c_int
    L.wf_tile_geometry.argtypes = [vp, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    L.wf_launch_count.argtypes = [vp]
    L.wf_launch_count.restype = C.c_int64
    L.wf_host_threads.argtypes = [vp]
    L.wf_host_threads.restype = C.c_int
    L.wf_expand_packed_obs.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32]
    L.wf_expand_packed_obs.restype = C.c_int
    L.wf_apply_change_blocks.argtypes = [vp, vp, C.c_int32, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_double,
                                         C.c_double, C.c_int32]
    L.wf_apply_change_blocks.restype = C.c_int
    L.wf_unpack_obs_bits.argtypes = [vp, C.c_int64, vp, C.c_int64, C.c_int32, C.c_int32, vp, C.c_int32, vp]
    L.wf_unpack_obs_bits.restype = C.c_int
    L.wf_state_bytes_per_env.argtypes = [vp]
    L.wf_state_bytes_per_env.restype = C.c_int64
    for name in ("wf_create", "wf_reset", "wf_step", "wf_rollout", "wf_rollout_policy", "wf_set_policy_mlp", "wf_step_host", "wf_get_state", "wf_set_state",
                 "wf_set_fire_to", "wf_get_obs", "wf_get_wind_table", "wf_stats", "wf_stats_reset", "wf_get_a_iter", "wf_set_a_iter", "wf_reset_host", "wf_tile_geometry", "wf_host_session"):
        getattr(L, name).restype = C.c_int
    _lib = L
    return L


def check(rc: int):
    if rc != WF_OK:
        raise WildfireError(f"libwildfire_b200 error {rc}: {lib().wf_last_error().decode()}")


EXPORTED_SYMBOLS = [
    "wf_default_config", "wf_create", "wf_destroy", "wf_last_error", "wf_abi_version", "wf_kernel_family",
    "wf_reset", "wf_step", "wf_rollout", "wf_rollout_policy", "wf_set_policy_mlp", "wf_step_host", "wf_get_state", "wf_set_state", "wf_set_fire_to",
    "wf_get_obs", "wf_get_wind_table", "wf_stats", "wf_stats_reset", "wf_philox_kat", "wf_launch_count",
    "wf_state_bytes_per_env", "wf_host_threads", "wf_expand_packed_obs", "wf_apply_change_blocks", "wf_get_a_iter", "wf_set_a_iter", "wf_reset_host", "wf_tile_geometry", "wf_host_session", "wf_host_session_active",
    "wf_unpack_obs_bits", "wf_set_policy_mlp_dev", "wf_replay_fit", "wf_replay_fit_many", "wf_set_policy_mlp_nets_dev",
    "wf_replay_fit_large",
]
