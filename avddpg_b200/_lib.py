"""ctypes binding of include/avddpg_b200.h (libavddpg_b200.so).

PyTorch is used by the callers for device memory and streams only; everything that crosses this
boundary is a raw pointer, a size or a POD struct.  There is NO CPU fallback: if the shared library is
missing, or no sm_100 device is visible when a compute entry point is reached, the call raises.
"""
from __future__ import annotations

import ctypes as C
import os

AVD_MAX_FOLLOWERS = 16
RING_RECORD_FLOATS = 10
ABI_VERSION = 3

RNG_RESET_VEHICLE, RNG_RESET_PLATOON, RNG_OU, RNG_LEADER_EXOG, RNG_REPLAY, RNG_INIT = range(6)

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libavddpg_b200.so")

f32p = C.POINTER(C.c_float)


class EnvParams(C.Structure):
    _fields_ = [
        ("M", C.c_int32), ("num_states", C.c_int32), ("model_a", C.c_int32), ("can_terminate", C.c_int32),
        ("centralized", C.c_int32), ("rand_uniform", C.c_int32), ("reset_mode", C.c_int32),
        ("steps_per_episode", C.c_int32),
        ("T", C.c_float), ("h", C.c_float), ("max_ep", C.c_float), ("max_ev", C.c_float),
        ("action_high", C.c_float), ("action_low", C.c_float),
        ("rew_ep", C.c_float), ("rew_ev", C.c_float), ("rew_u", C.c_float), ("rew_jerk", C.c_float),
        ("re_scalar", C.c_float), ("terminal_reward", C.c_float),
        ("reset_ep", C.c_float), ("reset_ev", C.c_float), ("reset_a", C.c_float),
        ("reset_leader_a", C.c_float), ("reset_u", C.c_float),
        ("ou_theta", C.c_float), ("ou_dt", C.c_float), ("ou_sigma", C.c_float), ("ou_mean", C.c_float),
        ("A", (C.c_float * 16) * AVD_MAX_FOLLOWERS),
        ("B", (C.c_float * 4) * AVD_MAX_FOLLOWERS),
        ("C", (C.c_float * 4) * AVD_MAX_FOLLOWERS),
    ]


class Clock(C.Structure):
    _fields_ = [("step_tick", C.c_uint64), ("ring_count", C.c_uint64), ("update_tick", C.c_uint64),
                ("reserved", C.c_uint64)]


class EnvIO(C.Structure):
    _fields_ = [
        ("P", C.c_int64), ("platoon_id_base", C.c_int64), ("seed", C.c_uint64),
        ("x_in", C.c_void_p), ("x_out", C.c_void_p), ("prev_a", C.c_void_p), ("cum_accel", C.c_void_p),
        ("action_mu", C.c_void_p), ("ou_state", C.c_void_p), ("action_out", C.c_void_p),
        ("leader_exog", C.c_void_p), ("front_u", C.c_void_p), ("front_accel", C.c_void_p),
        ("reward", C.c_void_p), ("done", C.c_void_p),
        ("jerk", C.c_void_p), ("velocity", C.c_void_p), ("headway", C.c_void_p),
        ("ring", C.c_void_p), ("ring_capacity", C.c_int64),
        ("episode", C.c_void_p), ("step_in_episode", C.c_void_p), ("ep_reward", C.c_void_p),
        ("stats", C.c_void_p), ("clock", C.c_void_p),
        ("gen_exog", C.c_int32), ("auto_reset", C.c_int32), ("clip_actions", C.c_int32), ("ep_hist_window", C.c_int32),
        ("last_ep_reward", C.c_void_p), ("ep_hist", C.c_void_p),
    ]


class NetDims(C.Structure):
    _fields_ = [("ns", C.c_int32), ("l1", C.c_int32), ("la", C.c_int32), ("l2", C.c_int32)]


class LearnIO(C.Structure):
    _fields_ = [
        ("dims", NetDims), ("A", C.c_int32), ("apply_updates", C.c_int32), ("rows_per_agent", C.c_int64),
        ("gamma", C.c_float), ("action_high", C.c_float), ("tau", C.c_float), ("actor_lr", C.c_float), ("critic_lr", C.c_float),
        ("adam_beta1", C.c_float), ("adam_beta2", C.c_float), ("adam_eps", C.c_float),
        ("s", C.c_void_p), ("a", C.c_void_p), ("r", C.c_void_p), ("s2", C.c_void_p),
        ("actor", C.c_void_p), ("critic", C.c_void_p), ("t_actor", C.c_void_p), ("t_critic", C.c_void_p),
        ("actor_grad", C.c_void_p), ("critic_grad", C.c_void_p),
        ("actor_m", C.c_void_p), ("actor_v", C.c_void_p), ("critic_m", C.c_void_p), ("critic_v", C.c_void_p),
        ("actor_t", C.c_void_p), ("critic_t", C.c_void_p),
        ("apply_mask", C.c_void_p), ("loss", C.c_void_p),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64),
        ("precision", C.c_int32), ("s_stride", C.c_int32),
    ]


AVD_MAX_PEERS = 16


class PeerComm(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("reserved0", C.c_uint32), ("reserved1", C.c_uint32),
                ("peer_base", C.c_uint64 * AVD_MAX_PEERS), ("multicast_base", C.c_uint64)]


class FedApplyIO(C.Structure):
    _fields_ = [
        ("comm", PeerComm), ("flag_offset", C.c_int64), ("data_offset", C.c_int64), ("local_sums", C.c_void_p), ("ctrl", C.c_void_p),
        ("pitch", C.c_int64), ("n_systems", C.c_int32), ("n_members", C.c_int32), ("member_stride_s", C.c_int64), ("member_stride_x", C.c_int64),
        ("A", C.c_int32), ("reserved0", C.c_int32),
        ("actor", C.c_void_p), ("t_actor", C.c_void_p), ("actor_m", C.c_void_p), ("actor_v", C.c_void_p), ("actor_step", C.c_void_p),
        ("actor_grad_out", C.c_void_p), ("actor_total", C.c_int64), ("actor_train", C.c_int64),
        ("critic", C.c_void_p), ("t_critic", C.c_void_p), ("critic_m", C.c_void_p), ("critic_v", C.c_void_p), ("critic_step", C.c_void_p),
        ("critic_grad_out", C.c_void_p), ("critic_total", C.c_int64), ("critic_train", C.c_int64),
        ("apply_mask", C.c_void_p), ("wsum_out", C.c_void_p),
        ("actor_lr", C.c_float), ("critic_lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float), ("tau", C.c_float),
    ]


class AvdError(RuntimeError):
    pass


_STATUS_EXC = {-1: ValueError, -2: RuntimeError, -3: NotImplementedError, -4: RuntimeError}

_lib = None

# name -> (restype, argtypes); the exported-symbol test checks every one of these against the header
SIGNATURES = {
    "avd_abi_version": (C.c_int, []),
    "avd_last_error": (C.c_char_p, []),
    "avd_kernel_launches": (C.c_int64, []),
    "avd_sizeof": (C.c_int64, [C.c_int]),
    "avd_device_info": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int64)]),
    "avd_clock_advance": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]),
    "avd_env_build_matrices": (C.c_int, [C.POINTER(EnvParams), C.c_int, C.c_double, C.c_double, C.c_double, C.c_double]),
    "avd_env_reset": (C.c_int, [C.POINTER(EnvParams), C.POINTER(EnvIO), C.c_void_p, C.c_void_p]),
    "avd_env_step": (C.c_int, [C.POINTER(EnvParams), C.POINTER(EnvIO), C.c_void_p]),
    "avd_ou_sample": (C.c_int, [C.POINTER(EnvParams), C.c_void_p, C.c_void_p, C.c_int64, C.c_uint64, C.c_uint64,
                                C.c_uint32, C.c_void_p]),
    "avd_env_step_host": (C.c_int, [C.POINTER(EnvParams), C.POINTER(EnvIO), C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p]),
    "avd_replay_add": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p]),
    "avd_replay_sample": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_uint64, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "avd_replay_sample_indices": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int64, C.c_uint64,
                                            C.c_void_p, C.c_void_p]),
    "avd_replay_gather": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "avd_replay_fill_synthetic": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_uint64, C.c_void_p]),
    "avd_ddpg_param_counts": (C.c_int, [C.POINTER(NetDims), C.POINTER(C.c_int64)]),
    "avd_ddpg_workspace_bytes": (C.c_int64, [C.POINTER(NetDims), C.c_int32, C.c_int64, C.c_int32]),
    "avd_forward_workspace_bytes": (C.c_int64, [C.POINTER(NetDims), C.c_int32, C.c_int64, C.c_int32, C.c_int32]),
    "avd_ddpg_learn": (C.c_int, [C.POINTER(LearnIO), C.c_void_p]),
    "avd_actor_forward": (C.c_int, [C.POINTER(NetDims), C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                    C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "avd_critic_forward": (C.c_int, [C.POINTER(NetDims), C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "avd_adam_apply": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_int32, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p]),
    "avd_polyak_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_void_p]),
    "avd_fed_reduce": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int64,
                                 C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "avd_adam_polyak_apply2": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                         C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_int64, C.c_float, C.c_void_p, C.c_int32, C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p]),
    "avd_fed_reduce2": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32,
                                  C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "avd_fed_broadcast2": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int32,
                                     C.c_int32, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "avd_fed_weights_from_history": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p]),
    "avd_fed_finalize": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p]),
    "avd_fed_exchange_peer": (C.c_int, [C.POINTER(PeerComm), C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int64,
                                        C.c_void_p]),
    "avd_fed_apply_gradients": (C.c_int, [C.POINTER(FedApplyIO), C.c_void_p]),
    "avd_fed_broadcast": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int64,
                                    C.c_void_p, C.c_int64, C.c_void_p]),
    "avd_gemm_bf16": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64,
                                C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p]),
    "avd_gemm_f16kind": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64,
                                   C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "avd_gemm_bf16x3": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64,
                                  C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p]),
    "avd_rng_words": (C.c_int, [C.c_void_p, C.c_int64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p]),
    "avd_rng_normals": (C.c_int, [C.c_void_p, C.c_int64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p]),
}


def lib_path() -> str:
    return _LIB_PATH


def load():
    """dlopen the library (once) and bind every declared symbol.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise AvdError(f"{_LIB_PATH} is missing: build it with `python -m avddpg_b200.build` "
                       "(needs nvcc; there is no CPU fallback)")
    lib = C.CDLL(_LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here == symbol not exported
        fn.restype, fn.argtypes = res, args
    if lib.avd_abi_version() != ABI_VERSION:
        raise AvdError(f"ABI mismatch: library {lib.avd_abi_version()} vs binding {ABI_VERSION}")
    for which, st in enumerate((EnvParams, EnvIO, Clock, NetDims, LearnIO, PeerComm, FedApplyIO)):
        if lib.avd_sizeof(which) != C.sizeof(st):
            raise AvdError(f"struct layout mismatch for {st.__name__}: C {lib.avd_sizeof(which)} vs ctypes {C.sizeof(st)}")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().avd_last_error().decode("utf-8", "replace")
        raise _STATUS_EXC.get(rc, AvdError)(f"libavddpg_b200: {msg} (status {rc})")


def require_device():
    """Fail loudly when there is no B200-class device: the product path never falls back to the CPU."""
    lib = load()
    sm, cc, mem = C.c_int(0), C.c_int(0), C.c_int64(0)
    check(lib.avd_device_info(C.byref(sm), C.byref(cc), C.byref(mem)))
    return sm.value, cc.value, mem.value


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
