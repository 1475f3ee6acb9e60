"""ctypes wrapper of oracle/c/libom_oracle.so (TEST INFRASTRUCTURE): the plain-C float64 restatement used
for cross-checking the NumPy oracle and as the CPU baseline."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

DIR = Path(__file__).resolve().parent / "c"
LIB = DIR / "libom_oracle.so"
_lib = None


class OrModel(C.Structure):
    _fields_ = [("nbody", C.c_int), ("njnt", C.c_int), ("nsite", C.c_int), ("nq", C.c_int), ("nv", C.c_int)] + \
               [(k, C.c_void_p) for k in ("body_parentid", "body_rootid", "body_jntadr", "body_jntnum", "jnt_type",
                                          "jnt_qposadr", "jnt_dofadr", "jnt_bodyid", "site_bodyid", "body_pos",
                                          "body_quat", "body_ipos", "body_mass", "jnt_axis", "jnt_pos", "qpos0",
                                          "site_pos", "site_quat")]


def lib():
    global _lib
    if _lib is None:
        # every time, not only when the .so is missing: a no-op when it is up to date, and a stale library would
        # otherwise test the old C code
        subprocess.check_call(["make", "-s", "-C", str(DIR)])
        _lib = C.CDLL(str(LIB))
        _lib.or_num_threads.restype = C.c_int
    return _lib


class CModel:
    def __init__(self, km):
        self.km = km
        i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)
        f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        self.keep = dict(body_parentid=i32(km.body_parentid), body_rootid=i32(km.body_rootid),
                         body_jntadr=i32(km.body_jntadr), body_jntnum=i32(km.body_jntnum), jnt_type=i32(km.jnt_type),
                         jnt_qposadr=i32(km.jnt_qposadr), jnt_dofadr=i32(km.jnt_dofadr), jnt_bodyid=i32(km.jnt_bodyid),
                         site_bodyid=i32(km.site_bodyid), body_pos=f64(km.body_pos), body_quat=f64(km.body_quat),
                         body_ipos=f64(km.body_ipos), body_mass=f64(km.body_mass), jnt_axis=f64(km.jnt_axis),
                         jnt_pos=f64(km.jnt_pos), qpos0=f64(km.qpos0), site_pos=f64(km.site_pos), site_quat=f64(km.site_quat))
        self.c = OrModel(nbody=km.nbody, njnt=km.njnt, nsite=km.nsite, nq=km.nq, nv=km.nv,
                         **{k: v.ctypes.data for k, v in self.keep.items()})


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def forward(cm, qpos, qvel):
    km = cm.km
    qpos, qvel = np.ascontiguousarray(qpos, np.float64), np.ascontiguousarray(qvel, np.float64)
    n = qpos.shape[0]
    out = dict(xpos=np.zeros((n, km.nbody, 3)), xquat=np.zeros((n, km.nbody, 4)), site_xpos=np.zeros((n, km.nsite, 3)),
               site_xmat=np.zeros((n, km.nsite, 3, 3)), cvel=np.zeros((n, km.nbody, 6)), subtree_com=np.zeros((n, km.nbody, 3)))
    lib().or_forward_batch(C.byref(cm.c), _p(qpos), _p(qvel), n, _p(out["xpos"]), _p(out["xquat"]), _p(out["site_xpos"]),
                           _p(out["site_xmat"]), _p(out["cvel"]), _p(out["subtree_com"]))
    return out


def h1_play_buffers(km, K, n_env, n_steps):
    """Output arrays of ``h1_play(record=True)`` (``n_steps``: all episodes' steps); allocate once and pass as ``out=`` to
    keep page faults and zero fills out of a timed region."""
    return dict(xpos=np.zeros((n_env, n_steps, km.nbody * 3)), xquat=np.zeros((n_env, n_steps, km.nbody * 4)),
                site_xpos=np.zeros((n_env, n_steps, km.nsite * 3)), cvel=np.zeros((n_env, n_steps, km.nbody * 6)),
                obs=np.zeros((n_env, n_steps, K - 2)), reward=np.zeros((n_env, n_steps)),
                fallen=np.zeros((n_env, n_steps), np.uint8), traj_no=np.zeros((n_env, n_steps), np.int32),
                step_no=np.zeros((n_env, n_steps), np.int32), checksum=np.zeros(n_env))


class OrPlayState(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("traj_no", "step_no", "reset_count", "xy_off", "curr_qpos", "pending",
                                          "prev_x_vel")]


def play_state(K, n_env):
    """The per-env state one playback call hands the next (the device's OmPlayState), env-major, float64 where the
    device keeps float32: traj_no, step_no, reset_count [n_env], xy_off [n_env, 2], curr_qpos [n_env, K/2], pending
    [n_env, K] (the loop's stale ``sample``), prev_x_vel [n_env].  All zero = a fresh env; its first call must reset."""
    return dict(traj_no=np.zeros(n_env, np.int32), step_no=np.zeros(n_env, np.int32),
                reset_count=np.zeros(n_env, np.uint32), xy_off=np.zeros((n_env, 2)), curr_qpos=np.zeros((n_env, K // 2)),
                pending=np.zeros((n_env, K)), prev_x_vel=np.zeros(n_env))


def h1_play(cm, perm, table, seed, env_id0, n_env, n_steps, dt=0.01, target=1.25, record=True, out=None, n_episodes=1,
            state=None, start_reset=True):
    """``play_trajectory_from_velocity`` for envs ``env_id0 ..`` ``env_id0 + n_env - 1``: ``n_episodes`` episodes of
    ``n_steps``, each ending with reset() (outputs [n_env, n_episodes * n_steps, ...]).  ``state`` (``play_state``) is
    read at the start and updated in place; ``None`` = fresh envs, final state dropped.  ``start_reset=False`` continues
    the state's episode instead of beginning with reset()."""
    km = cm.km
    table = np.ascontiguousarray(table, np.float64)
    K, n_traj, T = table.shape
    perm = np.ascontiguousarray(perm, np.int32)
    n_slots = n_episodes * n_steps
    if out is None:
        out = h1_play_buffers(km, K, n_env, n_slots) if record else dict(checksum=np.zeros(n_env))
    else:
        assert out["checksum"].shape == (n_env,) and ("reward" not in out or out["reward"].shape == (n_env, n_slots))
    if state is None:
        assert start_reset, "a fresh env begins with reset()"
        ps = None
    else:
        want = play_state(K, n_env)
        for k, v in want.items():
            a = state[k]
            assert isinstance(a, np.ndarray) and a.shape == v.shape and a.dtype == v.dtype and a.flags.c_contiguous, k
        ps = C.byref(OrPlayState(**{k: state[k].ctypes.data for k in want}))
    g = lambda k: _p(out.get(k))
    lib().or_h1_play_chain(C.byref(cm.c), _p(perm), _p(table), K, n_traj, T, C.c_uint64(seed), C.c_uint32(env_id0), n_env,
                           n_episodes, n_steps, int(bool(start_reset)), C.c_double(dt), C.c_double(target), ps, g("xpos"),
                           g("xquat"), g("site_xpos"), g("cvel"), g("obs"), g("reward"), g("fallen"), g("traj_no"),
                           g("step_no"), _p(out["checksum"]))
    return out


def gae_buffers(n_env, n_steps):
    return np.zeros((n_env, n_steps)), np.zeros((n_env, n_steps))


def gae(r, v, v_next, absorbing, last, gamma, lam, out=None):
    """Env-major [n_env, T] arrays.  ``out`` = (adv, v_target) preallocated (``gae_buffers``)."""
    r, v, v_next = (np.ascontiguousarray(a, np.float64) for a in (r, v, v_next))
    absorbing = np.ascontiguousarray(absorbing, np.uint8)
    last = np.ascontiguousarray(last, np.uint8)
    adv, vt = (np.zeros_like(r), np.zeros_like(r)) if out is None else out
    lib().or_gae(_p(r), _p(v), _p(v_next), _p(absorbing), _p(last), C.c_double(gamma), C.c_double(lam), r.shape[0], r.shape[1],
                 _p(adv), _p(vt))
    return vt, adv


def num_threads():
    return int(lib().or_num_threads())


def use_all_cores():
    """Undo an inherited OMP_NUM_THREADS=1 (torchrun sets it for every rank): one thread per usable host CPU."""
    import os
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    lib().or_set_num_threads(int(n))
    return num_threads()
