"""ctypes binding of libshems_b200.so — exactly the symbols include/shems_b200.h declares.

There is no CPU fallback: if the shared library is missing this module raises at load time,
and every compute entry point returns SHEMS_ERR_CUDA on a box without a CUDA device.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SHEMS_B200_LIB", os.path.join(HERE, "libshems_b200.so"))  # override: kernel-variant sweeps (tools/)

OK, ERR_INVALID, ERR_CUDA, ERR_BOUNDS, ERR_KEY, ERR_STATE = 0, -1, -2, -3, -4, -5
RESET_DETERMINISTIC, RESET_HOST_DRAWS, RESET_DEVICE_PHILOX = 0, 1, 2
POLICY_RULE, POLICY_RANDOM, POLICY_TAPE = 0, 1, 2
ENV_LU1, ENV_LU7, ENV_LU1_INPUT0607 = 0, 1, 2
NET_ACTOR, NET_CRITIC, NET_ACTOR_TARGET, NET_CRITIC_TARGET, NET_ACTOR_BEST = 0, 1, 2, 3, 4
DP_HANDLE_BYTES = 192


class ShemsParams(C.Structure):
    _fields_ = [
        ("pv_eta", C.c_float), ("b_eta", C.c_float), ("b_soc_min", C.c_float), ("b_soc_max", C.c_float),
        ("b_rate_max", C.c_double), ("b_loss", C.c_float), ("ev_soc_min", C.c_float), ("ev_soc_max", C.c_float),
        ("ev_rate_max", C.c_float), ("penalty_weight", C.c_float), ("sell_discount", C.c_double),
        ("discomfort_weight_ev", C.c_double), ("disc_pot", C.c_double),
        ("penalty_weight_f64", C.c_double), ("penalty_in_f64", C.c_int32), ("reward_form", C.c_int32),
    ]


class DdpgParams(C.Structure):
    _fields_ = [
        ("state_size", C.c_int32), ("action_size", C.c_int32), ("l1", C.c_int32), ("l2", C.c_int32),
        ("batch", C.c_int32), ("gamma", C.c_float), ("tau", C.c_float), ("lr_actor", C.c_float),
        ("lr_critic", C.c_float), ("adam_beta1", C.c_double), ("adam_beta2", C.c_double), ("adam_eps", C.c_double),
        ("act_lo", C.c_float * 2), ("act_hi", C.c_float * 2), ("use_tensor_cores", C.c_int32), ("population", C.c_int32),
    ]


class ShemsRolloutArgs(C.Structure):
    _fields_ = [
        ("policy", C.c_int32), ("n_steps", C.c_int32), ("seed", C.c_uint64), ("env_id_base", C.c_int64),
        ("tape_dev", C.c_void_p), ("ep_return_dev", C.c_void_p), ("replay", C.c_void_p), ("trace_dev", C.c_void_p),
        ("obs_traj_dev", C.c_void_p), ("reward_traj_dev", C.c_void_p), ("tape_unscaled", C.c_int32),
    ]


EXPLOIT_MAX_GROUPS = 16


class DdpgExploitParams(C.Structure):
    _fields_ = [
        ("frac", C.c_double), ("factor_lo", C.c_float), ("factor_hi", C.c_float), ("keys", C.c_int32), ("round", C.c_uint32),
        ("seed", C.c_uint64), ("n_groups", C.c_int32), ("group_start", C.c_int32 * (EXPLOIT_MAX_GROUPS + 1)),
    ]


class ShemsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[{code}] {msg}")
        self.code = code


class ShemsBoundsError(ShemsError, IndexError):
    """Julia BoundsError of next_state! (shems_LU1.jl:266-268)."""


class ShemsKeyError(ShemsError, KeyError):
    """Julia KeyError of capacities[charger_id] (shems_LU1.jl:95)."""


VP, PF, PI, PD = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_double)
I32, I64, U64, F32 = C.c_int32, C.c_int64, C.c_uint64, C.c_float

# name -> (restype, argtypes); every SHEMS_API symbol of include/shems_b200.h
SIGNATURES = {
    "shems_last_error": (C.c_char_p, []),
    "shems_version": (I32, []),
    "shems_device_count": (I32, []),
    "shems_env_kernel_launches": (I64, []),
    "shems_rollout_pair_launches": (I64, []),
    "shems_params_for_charger": (I32, [I32, C.POINTER(ShemsParams)]),
    "shems_params_for_env": (I32, [I32, I32, C.POINTER(ShemsParams)]),
    "shems_series_from_csv": (I32, [C.c_char_p, PF, I32, PI]),
    "shems_create": (I32, [C.POINTER(ShemsParams), PF, I32, I32, I64, I32, C.POINTER(VP)]),
    "shems_create_groups": (I32, [C.POINTER(ShemsParams), I32, C.POINTER(I64), PF, I32, I32, I32, I32, C.POINTER(VP)]),
    "shems_destroy": (I32, [VP]),
    "shems_set_stream": (I32, [VP, VP]),
    "shems_sync": (I32, [VP]),
    "shems_reset": (I32, [VP, I32, PI, PF, U64, I64]),
    "shems_step": (I32, [VP, VP, I32, VP, VP, VP, VP]),
    "shems_action_rule": (I32, [VP, VP]),
    "shems_action_drl": (I32, [VP, VP, VP]),
    "shems_finished": (I32, [VP, PI]),
    "shems_state_ptr": (I32, [VP, C.POINTER(VP), C.POINTER(VP)]),
    "shems_get_state": (I32, [VP, PF, PI]),
    "shems_set_state": (I32, [VP, PF, PI]),
    "shems_get_step": (I32, [VP, PI]),
    "shems_num_envs": (I64, [VP]),
    "shems_num_rows": (I32, [VP]),
    "shems_rollout": (I32, [VP, C.POINTER(ShemsRolloutArgs)]),
    "replay_create": (I32, [I64, I32, C.POINTER(VP)]),
    "replay_destroy": (I32, [VP]),
    "replay_set_stream": (I32, [VP, VP]),
    "replay_length": (I64, [VP]),
    "replay_capacity": (I64, [VP]),
    "replay_head": (I64, [VP]),
    "replay_series_count": (I32, [VP]),
    "replay_push": (I32, [VP, VP, VP, VP, VP, VP, I64]),
    "replay_push_groups": (I32, [C.POINTER(VP), I32, VP, VP, VP, VP, VP, I64]),
    "replay_sample": (I32, [VP, I32, PI, U64, VP, VP, VP, VP, VP]),
    "replay_minmax": (I32, [VP, I64, PI, U64, PF, PF]),
    "replay_get": (I32, [VP, PF, PF, PF, PF, PF]),
    "replay_enable_priorities": (I32, [VP]),
    "replay_get_priorities": (I32, [VP, PF, PF]),
    "replay_set_priorities": (I32, [VP, PF, F32]),
    "replay_sample_prioritized": (I32, [VP, I32, U64, F32, VP, VP]),
    "ddpg_default_params": (I32, [C.POINTER(DdpgParams)]),
    "ddpg_create": (I32, [C.POINTER(DdpgParams), I32, C.POINTER(VP)]),
    "ddpg_destroy": (I32, [VP]),
    "ddpg_set_stream": (I32, [VP, VP]),
    "ddpg_sync": (I32, [VP]),
    "ddpg_set_fused": (I32, [VP, I32]),
    "ddpg_set_prioritized": (I32, [VP, I32, F32, F32, F32]),
    "ddpg_get_prioritized": (I32, [VP, PI, PF, PF, PF]),
    "ddpg_init": (I32, [VP, U64]),
    "ddpg_set_layer": (I32, [VP, I32, I32, PF, PF]),
    "ddpg_get_layer": (I32, [VP, I32, I32, PF, PF]),
    "ddpg_get_grad": (I32, [VP, I32, I32, PF, PF]),
    "ddpg_num_params": (I64, [VP, I32]),
    "ddpg_set_norm": (I32, [VP, PF, PF]),
    "ddpg_act": (I32, [VP, VP, I64, F32, U64, I64, I64, VP, VP, VP]),
    "ddpg_act_soa": (I32, [VP, VP, I64, F32, U64, I64, I64, VP, VP, VP]),
    "ddpg_act_ou": (I32, [VP, VP, I64, F32, F32, F32, F32, VP, U64, I64, I64, VP, VP, VP]),
    "ddpg_set_noise": (I32, [VP, I32, F32, F32, F32]),
    "ddpg_episode": (I32, [VP, VP, C.POINTER(VP), I32, I32, F32, U64, I32, I64, VP, VP]),
    "ddpg_update": (I32, [VP, VP, I32, PI, U64]),
    "ddpg_update_phase": (I32, [VP, VP, I32, PI, U64, F32]),
    "ddpg_update_batch": (I32, [VP, VP, VP, VP, VP, VP]),
    "ddpg_dp_export": (I32, [VP, VP]),
    "ddpg_dp_connect": (I32, [VP, I32, I32, VP]),
    "ddpg_dp_prepare": (I32, [VP, I64]),
    "ddpg_update_dp": (I32, [VP, VP, I32, PI, U64]),
    "ddpg_dp_status": (I32, [VP, PI]),
    "ddpg_get_losses": (I32, [VP, PF, PF]),
    "ddpg_select_learner": (I32, [VP, I32]),
    "ddpg_population": (I32, [VP]),
    "ddpg_update_population": (I32, [VP, C.POINTER(VP), I32, PI, C.POINTER(U64)]),
    "ddpg_set_hparams": (I32, [VP, F32, F32, F32, F32, F32]),
    "ddpg_get_hparams": (I32, [VP, PF, PF, PF, PF, PF]),
    "shems_tc_gemm": (I32, [VP, I64, I32, VP, I64, I32, VP, I64, I32, I32, I32, I32, VP, VP, I64, I32, VP, VP]),
    "ddpg_grad_buffer": (I32, [VP, C.POINTER(VP), C.POINTER(I64)]),
    "ddpg_rollout": (I32, [VP, VP, I32, F32, U64, I64, VP, VP, VP]),
    "ddpg_evaluate": (I32, [VP, VP, I32, I32, I64, VP, VP, VP]),
    "ddpg_keep_best": (I32, [VP, VP, I64, I32, VP]),
    "ddpg_get_best": (I32, [VP, PD, PI]),
    "ddpg_set_best": (I32, [VP, PD, PI]),
    "ddpg_exploit": (I32, [VP, VP, C.POINTER(DdpgExploitParams), VP]),
    "ddpg_state_floats": (I64, [VP]),
    "ddpg_get_state": (I32, [VP, PF, PD]),
    "ddpg_set_state": (I32, [VP, PF, PD]),
    "ddpg_get_ou_state": (I32, [VP, PF, C.POINTER(I64)]),
    "ddpg_set_ou_state": (I32, [VP, PF, I64]),
}

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python __graft_entry__.py build` "
                "(nvcc, sm_100a).  There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(status):
    if status == OK:
        return
    msg = lib().shems_last_error().decode("utf-8", "replace")
    if status == ERR_BOUNDS:
        raise ShemsBoundsError(status, msg)
    if status == ERR_KEY:
        raise ShemsKeyError(status, msg)
    raise ShemsError(status, msg)


def params_for_charger(charger_id):
    p = ShemsParams()
    check(lib().shems_params_for_charger(int(charger_id), C.byref(p)))
    return p


def params_for_env(variant, charger_id):
    """module-level constants of shems_LU1.jl (0), shems_LU7.jl (1) or shems_LU1_input0607.jl (2) for a charger"""
    p = ShemsParams()
    check(lib().shems_params_for_env(int(variant), int(charger_id), C.byref(p)))
    return p


def default_ddpg_params(**kw):
    p = DdpgParams()
    check(lib().ddpg_default_params(C.byref(p)))
    for k, v in kw.items():
        if k in ("act_lo", "act_hi"):
            getattr(p, k)[0], getattr(p, k)[1] = v
        else:
            setattr(p, k, v)
    return p
