"""ctypes binding of the C ABI in include/uavenv_b200.h (lib/libuavenv_b200.so).

This is the only place the shared library is loaded.  There is no CPU fallback: when the library is
missing and cannot be built, or when it reports a failure, an exception is raised.
"""
import ctypes as C
import os

import torch

from . import _build

STATE_DIM = 14
SEQ_LEN = 5

c_f64p = C.POINTER(C.c_double)
c_f32p = C.POINTER(C.c_float)
c_i32p = C.POINTER(C.c_int32)
c_u8p = C.POINTER(C.c_uint8)


class UavenvCfg(C.Structure):
    _fields_ = [("num_uavs", C.c_int32), ("num_targets", C.c_int32), ("num_nfz", C.c_int32),
                ("num_interceptors", C.c_int32), ("reset_episodes", C.c_int32), ("auto_reset", C.c_int32),
                ("param_zeta_d", C.c_double), ("param_k", C.c_double),
                ("param_c1", C.c_double), ("param_c2", C.c_double), ("param_c3", C.c_double),
                ("param_c4", C.c_double), ("cost_weight_omega", C.c_double),
                ("weather_speed_factor", C.c_double), ("weather_load_factor", C.c_double),
                ("map_width", C.c_double), ("map_height", C.c_double),
                ("uav_gen_x_lo", C.c_double), ("uav_gen_x_hi", C.c_double),
                ("target_gen_x_lo", C.c_double), ("target_gen_x_hi", C.c_double),
                ("intercept_rad", C.c_double), ("tie_band", C.c_double)]


class UavenvInfo(C.Structure):
    _fields_ = [("d_J_val", C.c_void_p), ("d_num_assigned", C.c_void_p), ("d_is_valid_action", C.c_void_p),
                ("d_avg_p_dmg", C.c_void_p), ("d_avg_p_final", C.c_void_p), ("d_reward_f64", C.c_void_p)]


class UavenvEpisodeAcc(C.Structure):
    _fields_ = [("d_ret", C.c_void_p), ("d_length", C.c_void_p), ("d_assigns", C.c_void_p), ("d_valid", C.c_void_p),
                ("d_episodes", C.c_void_p), ("d_envs_complete", C.c_void_p)]


# uavenv_episode_t (40 bytes, C layout)
EPISODE_FIELDS = [("ret", "<f8"), ("J_val", "<f4"), ("avg_p_dmg", "<f4"), ("avg_p_final", "<f4"), ("length", "<i4"),
                  ("num_assigned", "<i4"), ("assigns", "<i4"), ("valid", "<i4")]
EPISODE_BYTES = 40

SCENE_FIELDS = [("uav_x", "f8", "N"), ("uav_y", "f8", "N"), ("uav_vx", "f8", "N"), ("uav_vy", "f8", "N"),
                ("uav_load", "f8", "N"), ("uav_cost", "f8", "N"), ("uav_type", "i4", "N"),
                ("tgt_x", "f8", "M"), ("tgt_y", "f8", "M"), ("tgt_vx", "f8", "M"), ("tgt_vy", "f8", "M"),
                ("tgt_value", "f8", "M"), ("tgt_id", "i4", "M"),
                ("nfz_x", "f8", "K1"), ("nfz_y", "f8", "K1"), ("nfz_radius", "f8", "K1"),
                ("int_x", "f8", "K2"), ("int_y", "f8", "K2"), ("int_vx", "f8", "K2"), ("int_vy", "f8", "K2")]


class UavenvScene(C.Structure):
    _fields_ = [(name, C.c_void_p) for name, _, _ in SCENE_FIELDS]


STATE_FIELDS = [("uav_idx", "i4", "1"), ("target_idx", "i4", "1"), ("assigned_target_id", "i4", "N"),
                ("lock_count", "i4", "M"), ("not_hit", "f8", "M"), ("not_hit_pure", "f8", "M"),
                ("J_val", "f8", "1"), ("episode", "i4", "1"), ("scene_index", "i4", "1"), ("finished", "u1", "1")]


class UavenvState(C.Structure):
    _fields_ = [(name, C.c_void_p) for name, _, _ in STATE_FIELDS]


class UavenvError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("uavenv error %d: %s" % (code, message))
        self.code = code


_lib = None


def lib_path():
    return _build.LIB_PATH


def _open(path, override_var, abi_fn, abi_version):
    """The library at `path`, built first when it is stale, or the build named by $override_var (timing experiments
    only: an ablation / diagnostic build of the same ABI).  Raises ImportError on any failure."""
    name = os.path.basename(path)
    override = os.environ.get(override_var)
    if override:
        path = override
    elif not _build.up_to_date(path):
        try:
            _build.build(lib=path)
        except Exception as exc:  # no nvcc on this host, or a compile error: never load a binary older than its sources
            raise ImportError("%s is %s and could not be (re)built (%s); there is no CPU fallback" % (
                name, "stale" if os.path.isfile(path) else "missing", exc)) from exc
    L = C.CDLL(path)
    getattr(L, abi_fn).restype = C.c_int
    if getattr(L, abi_fn)() != abi_version:
        raise ImportError("%s ABI version mismatch" % name)
    return L


def load():
    """Load (building first if the sources are newer) the sm_100a library.  Raises on any failure."""
    global _lib
    if _lib is not None:
        return _lib
    L = _open(_build.LIB_PATH, "UAVENV_LIB_OVERRIDE", "uavenv_abi_version", 2)
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    L.uavenv_default_cfg.argtypes = [C.POINTER(UavenvCfg)]
    L.uavenv_default_cfg.restype = None
    L.uavenv_create.argtypes = [C.POINTER(UavenvCfg), i32, i32, u64, u64, C.POINTER(vp)]
    L.uavenv_destroy.argtypes = [vp]
    L.uavenv_last_error.argtypes = [vp]
    L.uavenv_last_error.restype = C.c_char_p
    L.uavenv_num_envs.argtypes = [vp]
    L.uavenv_num_envs.restype = i32
    L.uavenv_reset.argtypes = [vp, i32, vp, vp, vp]
    L.uavenv_step.argtypes = [vp, vp, vp, vp, vp, C.POINTER(UavenvInfo), vp]
    L.uavenv_step_host.argtypes = [vp, vp, vp, vp, vp, vp]
    L.uavenv_step_host_i8.argtypes = [vp, vp, vp, vp, vp, vp]
    L.uavenv_step_host_i8.restype = C.c_int
    L.uavenv_obs_buffer.argtypes = [vp]
    L.uavenv_obs_buffer.restype = vp
    L.uavenv_load_scene.argtypes = [vp, C.POINTER(UavenvScene), i32, i32, vp]
    L.uavenv_load_scene_device.argtypes = [vp, C.POINTER(UavenvScene), i32, i32, i32, vp, vp]
    L.uavenv_group_best.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, vp, vp]
    L.uavenv_improve_allocation.argtypes = [vp, i32, i32, i32, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    L.uavenv_improve_workspace_bytes.argtypes = [vp]
    L.uavenv_improve_workspace_bytes.restype = C.c_size_t
    L.uavenv_upper_bound.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp, vp, vp]
    L.uavenv_get_scene.argtypes = [vp, C.POINTER(UavenvScene), i32, i32]
    L.uavenv_get_state.argtypes = [vp, C.POINTER(UavenvState), i32, i32]
    L.uavenv_set_episode_counters.argtypes = [vp, vp, i32, i32]
    L.uavenv_set_episode_counters.restype = C.c_int
    L.uavenv_score_matrix.argtypes = [vp, vp, vp, vp]
    L.uavenv_score_matrix_f64.argtypes = [vp, vp, vp, vp]
    L.uavenv_recompute_objective.argtypes = [vp, c_f64p, vp]
    L.uavenv_random_actions.argtypes = [vp, u64, u64, vp, vp]
    L.uavenv_best_target_actions.argtypes = [vp, vp, vp, vp]
    L.uavenv_episode_accumulate.argtypes = [i32, vp, vp, C.POINTER(UavenvInfo), i32, C.POINTER(UavenvEpisodeAcc), vp, i32, vp]
    L.ppo_gae_advantages.argtypes = [vp, vp, vp, vp, i32, i32, C.c_float, C.c_float, vp, vp, i32, vp, i32, vp]
    L.ppo_normalize_advantages.argtypes = [vp, i64, vp, i32, vp]
    L.ppo_attn5_forward.argtypes = [vp, i64, vp, vp, i64, vp, i64, i32, vp, i32, vp]
    L.ppo_attn5_backward.argtypes = [vp, i64, vp, vp, i64, vp, i64, i32, vp, vp, vp, vp, i32, vp]
    L.ppo_clip_adam_step.argtypes = [vp, vp, vp, vp, i64, C.POINTER(i64), C.POINTER(C.c_float), i32, C.c_float, C.c_float,
                                     C.c_float, C.c_float, C.c_float, vp, vp, vp, i32, vp]
    L.ppo_clip_adam_step.restype = C.c_int
    L.ppo_optim_partials.restype = C.c_int
    L.ppo_attn5_forward.restype = C.c_int
    L.ppo_attn5_backward.restype = C.c_int
    for name in ("uavenv_create", "uavenv_destroy", "uavenv_reset", "uavenv_step", "uavenv_step_host",
                 "uavenv_load_scene", "uavenv_get_scene", "uavenv_get_state", "uavenv_score_matrix",
                 "uavenv_score_matrix_f64", "uavenv_recompute_objective", "uavenv_random_actions", "uavenv_best_target_actions",
                 "uavenv_episode_accumulate", "ppo_gae_advantages", "ppo_normalize_advantages",
                 "uavenv_load_scene_device", "uavenv_group_best", "uavenv_improve_allocation", "uavenv_upper_bound"):
        getattr(L, name).restype = C.c_int
    _lib = L
    return L


def check(rc, handle=None, last_error=None):
    """Raises UavenvError with the library's message when rc != 0: last_error(handle), by default the env library's
    uavenv_last_error, which with no handle reports this thread's last create or handle-free call that failed."""
    if rc != 0:
        msg = (last_error or load().uavenv_last_error)(handle)
        raise UavenvError(rc, msg.decode() if msg else "(no message)")


def cuda_device(device, what):
    """The torch.device `what` runs on: `device` (None: the current CUDA device), which must be a CUDA device."""
    dev = torch.device("cuda" if device is None else device)
    if dev.type != "cuda" or not torch.cuda.is_available():
        raise RuntimeError("%s runs on a CUDA device (sm_100a) only; there is no CPU fallback" % what)
    return torch.device("cuda", torch.cuda.current_device()) if dev.index is None else dev


class Handle:
    """One library handle on a CUDA device: created with <prefix>_create, every call checked through
    <prefix>_last_error, work enqueued on the device's current stream, <prefix>_destroy on close."""

    def __init__(self, load_lib, prefix, device, what):
        self._h = None
        self.device = cuda_device(device, what)
        self._lib, self._prefix = load_lib(), prefix
        self._last_error = getattr(self._lib, prefix + "_last_error")

    def _create(self, *args):
        h = C.c_void_p()
        self._chk(getattr(self._lib, self._prefix + "_create")(*args, C.byref(h)))
        self._h = h

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _chk(self, rc):
        check(rc, self._h, self._last_error)

    def close(self):
        if getattr(self, "_h", None):
            getattr(self._lib, self._prefix + "_destroy")(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- policy rollout forward (include/uavpolicy_b200.h, lib/libuavpolicy_b200.so) ---------------------------------
_policy_lib = None
NUM_PARAMS = 419267   # UAVPOLICY_NUM_PARAMS: length of the flat parameter vector of include/uavpolicy_b200.h


def load_policy():
    """Load (building first if stale) the tcgen05 policy-forward library.  Raises on any failure."""
    global _policy_lib
    if _policy_lib is not None:
        return _policy_lib
    L = _open(_build.POLICY_LIB_PATH, "UAVPOLICY_LIB_OVERRIDE", "uavpolicy_abi_version", 3)
    vp, i32, u64 = C.c_void_p, C.c_int32, C.c_uint64
    L.uavpolicy_create.argtypes = [i32, i32, C.POINTER(vp)]
    L.uavpolicy_destroy.argtypes = [vp]
    L.uavpolicy_last_error.argtypes = [vp]
    L.uavpolicy_last_error.restype = C.c_char_p
    L.uavpolicy_set_weights.argtypes = [vp, vp, vp]
    L.uavpolicy_get_action.argtypes = [vp, vp, i32, u64, u64, u64, vp, vp, vp, vp, vp, vp]
    L.uavpolicy_act.argtypes = [vp, vp, i32, i32, u64, u64, u64, vp, vp, vp, vp]        # include/uavpolicy_eval_b200.h
    L.uavpolicy_selftest_gemm_tile.argtypes = [vp, vp, vp, i32, i32, vp]
    i64 = C.c_int64
    L.uavpolicy_selftest_wgrad.argtypes = [vp, i64, vp, i64, i32, i32, i32, vp, vp, vp]
    L.uavpolicy_selftest_dense.argtypes = [vp, i64, vp, vp, vp, i64, vp, i32, i32, i32, i32, vp]
    L.uavpolicy_selftest_dense_ln.argtypes = [vp, i64, vp, vp, vp, i64, vp, vp, vp, vp, vp, i32, i32, vp]
    L.uavtrain_create.argtypes = [i32, i32, C.POINTER(vp)]
    L.uavtrain_destroy.argtypes = [vp]
    L.uavtrain_last_error.argtypes = [vp]
    L.uavtrain_last_error.restype = C.c_char_p
    L.uavtrain_forward.argtypes = [vp, vp, vp, i32, vp, vp]
    L.uavtrain_backward.argtypes = [vp, vp, vp, vp]
    L.uavtrain_forward_heads.argtypes = [vp, vp, vp, i32, vp, vp, vp]
    L.uavtrain_backward_heads.argtypes = [vp, vp, vp, vp, vp]
    L.uavtrain_ppo_loss.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i32, C.c_float, C.c_float, C.c_float, vp, vp, vp, vp]
    for name in ("uavpolicy_create", "uavpolicy_destroy", "uavpolicy_set_weights", "uavpolicy_get_action",
                 "uavpolicy_act", "uavpolicy_selftest_gemm_tile", "uavpolicy_selftest_wgrad", "uavpolicy_selftest_dense",
                 "uavpolicy_selftest_dense_ln", "uavtrain_create",
                 "uavtrain_destroy", "uavtrain_forward", "uavtrain_backward", "uavtrain_forward_heads",
                 "uavtrain_backward_heads", "uavtrain_ppo_loss"):
        getattr(L, name).restype = C.c_int
    _policy_lib = L
    return L
