"""ctypes binding of libom_b200.so (the C ABI declared in include/om_b200.h).

There is no CPU implementation behind these calls: if the shared library is missing, or no CUDA device
is present, every compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libom_b200.so"

c_f32p = C.c_void_p      # device pointers travel as integers
_lib = None


class OmModelDesc(C.Structure):
    _fields_ = [("name", C.c_char_p),
                ("nbody", C.c_int), ("njnt", C.c_int), ("nsite", C.c_int), ("nq", C.c_int), ("nv", C.c_int),
                ("body_parentid", C.c_void_p), ("body_rootid", C.c_void_p), ("body_jntadr", C.c_void_p),
                ("body_jntnum", C.c_void_p), ("body_pos", C.c_void_p), ("body_quat", C.c_void_p),
                ("body_ipos", C.c_void_p), ("body_mass", C.c_void_p), ("jnt_type", C.c_void_p),
                ("jnt_qposadr", C.c_void_p), ("jnt_dofadr", C.c_void_p), ("jnt_axis", C.c_void_p),
                ("jnt_pos", C.c_void_p), ("qpos0", C.c_void_p), ("site_bodyid", C.c_void_p),
                ("site_pos", C.c_void_p), ("site_quat", C.c_void_p)]


class OmH1Spec(C.Structure):
    _fields_ = [("n_obs_q", C.c_int), ("obs_perm", C.c_int32 * 32), ("x_vel_idx", C.c_int),
                ("target_velocity", C.c_float), ("use_absorbing_states", C.c_int)]


class OmPlayState(C.Structure):
    _fields_ = [("traj_no", C.c_void_p), ("step_no", C.c_void_p), ("reset_count", C.c_void_p),
                ("xy_off", C.c_void_p), ("curr_qpos", C.c_void_p), ("pending", C.c_void_p),
                ("prev_x_vel", C.c_void_p)]


class OmPlayOut(C.Structure):
    _fields_ = [("xpos", C.c_void_p), ("xquat", C.c_void_p), ("site_xpos", C.c_void_p), ("cvel", C.c_void_p),
                ("obs", C.c_void_p), ("reward", C.c_void_p), ("fallen", C.c_void_p), ("traj_no_t", C.c_void_p),
                ("step_no_t", C.c_void_p), ("obs_moments", C.c_void_p)]


class OmLiveState(C.Structure):
    _fields_ = [("traj_no", C.c_void_p), ("step_no", C.c_void_p), ("reset_count", C.c_void_p), ("xy_off", C.c_void_p),
                ("prev_x_vel", C.c_void_p)]


class OmLiveOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("qpos", "qvel", "xpos", "xquat", "site_xpos", "cvel", "obs", "reward",
                                          "absorbing", "wrapped")]


class OmH1ResetArgs(C.Structure):
    _fields_ = [("mask", C.c_void_p), ("absorbing", C.c_void_p), ("horizon", C.c_int), ("forced_traj", C.c_int),
                ("forced_step", C.c_int), ("traj_no", C.c_void_p), ("step_no", C.c_void_p), ("reset_count", C.c_void_p),
                ("xy_off", C.c_void_p), ("qpos", C.c_void_p), ("qvel", C.c_void_p), ("obs_in", C.c_void_p),
                ("obs", C.c_void_p), ("obs_dim", C.c_int), ("prev_x_vel", C.c_void_p), ("episode_step", C.c_void_p),
                ("last", C.c_void_p), ("grf", C.c_void_p), ("n_grf", C.c_int), ("partial_resets", C.c_void_p),
                ("model_index", C.c_void_p), ("mass", C.c_void_p), ("n_models", C.c_int), ("random", C.c_int),
                ("masses_host", C.c_void_p)]


class OmA3TaskDesc(C.Structure):
    _fields_ = [("period", C.c_int), ("delay_frames", C.c_int), ("target_radius", C.c_double),
                ("goal_height_ref", C.c_double), ("goal_speed_ref", C.c_double), ("total_mass", C.c_double),
                ("clock_lut_host", C.c_void_p), ("init_qpos_host", C.c_void_p)]


class OmA3State(C.Structure):
    _fields_ = [("ints", C.c_void_p), ("sequence", C.c_void_p)]


class OmA3Out(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("terms", C.c_void_p), ("reward", C.c_void_p), ("done", C.c_void_p),
                ("xpos", C.c_void_p), ("xquat", C.c_void_p), ("site_xpos", C.c_void_p), ("site_xmat", C.c_void_p),
                ("cvel", C.c_void_p)]


class OmA3Returns(C.Structure):
    _fields_ = [("values", C.c_void_p), ("v_next", C.c_void_p), ("v_last", C.c_void_p), ("path_end", C.c_void_p),
                ("gamma", C.c_float), ("ret", C.c_void_p), ("adv", C.c_void_p)]


class OmA3AutoResetArgs(C.Structure):
    _fields_ = [("done", C.c_void_p), ("max_traj_len", C.c_int), ("iteration_count", C.c_double),
                ("reset_count", C.c_void_p), ("traj_len", C.c_void_p), ("qpos", C.c_void_p), ("qvel", C.c_void_p),
                ("state", OmA3State), ("obs_in", C.c_void_p), ("obs", C.c_void_p), ("last", C.c_void_p),
                ("path_end", C.c_void_p)]


class OmDiscDesc(C.Structure):
    _fields_ = [("kind", C.c_int), ("n_in", C.c_int), ("n_h1", C.c_int), ("n_h2", C.c_int), ("z_size", C.c_int)] + \
               [(k, C.c_void_p) for k in ("w1", "b1", "w2", "b2", "wmu", "bmu", "wlv", "blv", "wd", "bd")]


class OmActionSpec(C.Structure):
    _fields_ = [("nu", C.c_int), ("delta", C.c_float * 32), ("mean", C.c_float * 32)]


class OmPdSpec(C.Structure):
    _fields_ = [("nu", C.c_int), ("qposadr", C.c_int32 * 32), ("dofadr", C.c_int32 * 32), ("kp", C.c_float * 32),
                ("kd", C.c_float * 32), ("gear", C.c_float * 32), ("offset", C.c_float * 32)]


class OmMirrorSpec(C.Structure):
    _fields_ = [("numel", C.c_int), ("index", C.c_int32 * 64), ("sign", C.c_float * 64), ("negate", C.c_uint8 * 64)]


_P, _I, _F, _D = C.c_void_p, C.c_int, C.c_float, C.c_double
_U64, _U32 = C.c_uint64, C.c_uint32

# name -> (restype, argtypes); kept in the order of include/om_b200.h
PROTOTYPES = {
    "om_last_error": (C.c_char_p, []),
    "om_abi_version": (_I, []),
    "om_launch_count": (C.c_longlong, []),
    "om_reset_launch_count": (None, []),
    "om_debug_set": (_I, [C.c_char_p, _I]),
    "om_model_create": (_I, [C.POINTER(OmModelDesc), C.POINTER(_P)]),
    "om_model_destroy": (None, [_P]),
    "om_model_is_specialised": (_I, [_P]),
    "om_model_h1_variant": (_I, [_P]),
    "om_model_bind_env_body_mass": (_I, [_P, _I, _P, _I]),
    "om_fk": (_I, [_P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _I, _P]),
    "om_h1_step": (_I, [_P, C.POINTER(OmH1Spec), _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "om_set_sim_state": (_I, [_P, C.POINTER(OmH1Spec), _P, _I, _I, _P, _P, _P]),
    "om_h1_has_fallen": (_I, [_P, _I, _I, _P, _P]),
    "om_traj_create": (_I, [_P, _I, _I, _I, C.POINTER(_P)]),
    "om_traj_destroy": (None, [_P]),
    "om_traj_reset": (_I, [_P, _U64, _U32, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _P]),
    "om_traj_current": (_I, [_P, _P, _P, _P, _P, _I, _I, _P]),
    "om_traj_next": (_I, [_P, _U64, _U32, _I, _P, _P, _P, _P, _P, _P, _I, _I, _P]),
    "om_h1_play_from_velocity": (_I, [_P, C.POINTER(OmH1Spec), _P, _U64, _U32, _D, _I, _I,
                                      C.POINTER(OmPlayState), C.POINTER(OmPlayOut), _I, _I, _P]),
    "om_h1_live_step": (_I, [_P, C.POINTER(OmH1Spec), _P, _U64, _U32, C.POINTER(OmLiveState), C.POINTER(OmLiveOut), _I, _I, _P]),
    "om_h1_draw_models": (_I, [_U64, _U32, _U32, _I, _I, _P, _P, _P, _I, _P]),
    "om_h1_reset_envs": (_I, [_P, C.POINTER(OmH1Spec), _P, _U64, _U32, C.POINTER(OmH1ResetArgs), _I, _I, _P]),
    "om_a3_task_create": (_I, [C.POINTER(OmA3TaskDesc), C.POINTER(_P)]),
    "om_a3_task_destroy": (None, [_P]),
    "om_a3_task_step": (_I, [_P, _P, _P, _P, _P, _I, C.POINTER(OmA3State), C.POINTER(OmA3Out), _I, _I, _P]),
    "om_a3_task_rollout": (_I, [_P, _P, _P, _P, _P, _I, C.POINTER(OmA3State), C.POINTER(OmA3Out), C.POINTER(OmA3Returns), _I, _I, _P]),
    "om_a3_reset": (_I, [_P, _P, _U64, _U32, _P, _P, _D, _P, _P, C.POINTER(OmA3State), _P, _I, _I, _P]),
    "om_a3_autoreset": (_I, [_P, _P, _U64, _U32, C.POINTER(OmA3AutoResetArgs), _I, _I, _P]),
    "om_disc_create": (_I, [C.POINTER(OmDiscDesc), C.POINTER(_P)]),
    "om_disc_destroy": (None, [_P]),
    "om_disc_reward": (_I, [_P, _P, _P, _P, _P, _I, _I, _P, _P, _P]),
    "om_disc_forward": (_I, [_P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P]),
    "om_disc_loss_stats": (_I, [_P, _P, _P, _I, _I, _F, _P, _P, _P]),
    "om_expert_minibatch": (_I, [_P, _I, _I, _I, _U64, _U32, _I, _P, _P, _P, _I, _P]),
    "om_action_affine": (_I, [C.POINTER(OmActionSpec), _P, _I, _I, _P, _P]),
    "om_pd_torque": (_I, [C.POINTER(OmPdSpec), _P, _P, _P, _P, _I, _I, _I, _P, _P]),
    "om_mirror": (_I, [C.POINTER(OmMirrorSpec), _P, _I, _I, _P, _P]),
    "om_ppo_loss_stats": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, C.POINTER(OmMirrorSpec), _I, _I, _I, _F, _F, _P, _P, _P, _P]),
    "om_h1_play_trajectory": (_I, [_P, C.POINTER(OmH1Spec), _P, _U64, _U32, _I, _I,
                                   C.POINTER(OmPlayState), C.POINTER(OmPlayOut), _I, _I, _P]),
    "om_ppo_returns": (_I, [_P, _P, _P, _P, _P, _F, _I, _I, _I, _P, _P, _P]),
    "om_gae": (_I, [_P, _P, _P, _P, _P, _F, _F, _I, _I, _I, _P, _P, _P]),
    "om_moments": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "om_adv_stats": (_I, [_P, _I, _D, _P, _P]),
    "om_moment_stats": (_I, [_P, _I, _I, _P, _P, _P, _P, _P]),
    "om_normalize": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "om_mailbox_create": (_I, [_I, _I, C.POINTER(_P), _P]),
    "om_mailbox_connect": (_I, [_P, _P]),
    "om_mailbox_allreduce": (_I, [_P, _P, _P, _I, _P]),
    "om_mailbox_set_timeout_ms": (_I, [_P, _D]),
    "om_mailbox_timed_out": (_I, [_P, C.POINTER(_I)]),
    "om_mailbox_destroy": (None, [_P]),
}


class OmError(RuntimeError):
    pass


def load():
    """Load the shared library (once) and declare every prototype.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise OmError(f"{LIB_PATH} is missing: run `python -m olympics_mujoco_b200.build` "
                      "(nvcc, sm_100a).  This package has no CPU fallback.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise OmError(load().om_last_error().decode())


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise OmError("no CUDA device: olympics_mujoco_b200 computes only on the GPU (no CPU fallback)")
