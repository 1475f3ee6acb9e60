"""Torch-level wrappers over the C ABI: torch provides device memory and streams, nothing else.

Layout contract (include/om_b200.h): every per-env array is a 2-D ``[C, n]`` tensor (component-major,
env index contiguous); rollout buffers are ``[T, C, n]``.  ``env_major`` gives the reference's logical
shapes (``[n, nbody, 3]`` ...) as zero-copy permuted views.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import (OmA3AutoResetArgs, OmA3Out, OmA3Returns, OmA3State, OmA3TaskDesc, OmActionSpec, OmDiscDesc, OmH1ResetArgs, OmH1Spec, OmLiveOut, OmLiveState, OmMirrorSpec,
                   OmPdSpec, OmModelDesc, OmPlayOut, OmPlayState, check)
from .mjcf import KinematicModel


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t, dtype=None, rows=None):
    """Device pointer of a tensor laid out [.., C, ld] with unit stride on the last axis."""
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.OmError("expected a CUDA tensor (this package has no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"expected {dtype}, got {t.dtype}")
    if t.dim() >= 1 and t.stride(-1) != 1 and t.shape[-1] > 1:
        raise ValueError("last axis (envs) must be contiguous")
    if t.dim() >= 2 and not t.is_contiguous():
        raise ValueError("SoA arrays must be contiguous [.., C, n] tensors")
    return C.c_void_p(t.data_ptr())


def soa(c, n, dtype=torch.float32, device="cuda", t=None):
    shape = (c, n) if t is None else (t, c, n)
    return torch.empty(shape, dtype=dtype, device=device)


def env_major(x, *comp_shape):
    """[C, n] -> [n, *comp_shape] view (or [T, C, n] -> [T, n, *comp_shape])."""
    if x.dim() == 2:
        return x.view(*comp_shape, x.shape[-1]).permute(len(comp_shape), *range(len(comp_shape)))
    t = x.shape[0]
    v = x.view(t, *comp_shape, x.shape[-1])
    return v.permute(0, len(comp_shape) + 1, *range(1, len(comp_shape) + 1))


def to_soa(x):
    """[n, C] (any float dtype, host or device) -> contiguous float32 [C, n] CUDA tensor."""
    x = torch.as_tensor(x)
    return x.to(device="cuda", dtype=torch.float32).t().contiguous()


# ------------------------------------------------------------------------------------------- model
class DeviceModel:
    """OmModel handle for a KinematicModel."""

    def __init__(self, km: KinematicModel):
        _lib.require_cuda()
        lib = _lib.load()
        self.km = km
        i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)
        f64 = lambda a: np.ascontiguousarray(a, dtype=np.float64)
        keep = dict(body_parentid=i32(km.body_parentid), body_rootid=i32(km.body_rootid),
                    body_jntadr=i32(km.body_jntadr), body_jntnum=i32(km.body_jntnum), body_pos=f64(km.body_pos),
                    body_quat=f64(km.body_quat), body_ipos=f64(km.body_ipos), body_mass=f64(km.body_mass),
                    jnt_type=i32(km.jnt_type), jnt_qposadr=i32(km.jnt_qposadr), jnt_dofadr=i32(km.jnt_dofadr),
                    jnt_axis=f64(km.jnt_axis), jnt_pos=f64(km.jnt_pos), qpos0=f64(km.qpos0),
                    site_bodyid=i32(km.site_bodyid), site_pos=f64(km.site_pos), site_quat=f64(km.site_quat))
        desc = OmModelDesc(name=km.name.encode(), nbody=km.nbody, njnt=km.njnt, nsite=km.nsite, nq=km.nq, nv=km.nv,
                           **{k: v.ctypes.data for k, v in keep.items()})
        h = C.c_void_p()
        check(lib.om_model_create(C.byref(desc), C.byref(h)))
        self.handle = h
        self.specialised = bool(lib.om_model_is_specialised(h))
        # UnitreeH1 model with fused playback / live-step kernels: 1 the default, 2.. its other variants, 0 none
        self.h1_variant = int(lib.om_model_h1_variant(h))

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                _lib.load().om_model_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


def bind_env_body_mass(dm: DeviceModel, body, mass):
    """``om_model_bind_env_body_mass``: from now on every FK of ``dm`` (a UnitreeH1 carry model) reads body ``body``'s mass
    of env i from ``mass[i]`` (float32 [n] CUDA tensor, updated in place by its owner).  For the model's life: the tensor
    is kept alive by ``dm``."""
    check(_lib.load().om_model_bind_env_body_mass(dm.handle, int(body), _p(mass, torch.float32), max(mass.numel(), 1)))
    dm.env_mass = mass


def h1_draw_models(seed, env_id0, count, body_masses, idx, mass, random=True):
    """``om_h1_draw_models``: the per-env model switch of one MultiMuJoCo reset (counter ``count``) into ``idx`` (int32
    [n]) and ``mass`` (float32 [n], ``body_masses[idx]``), on the device, in place."""
    bm = np.ascontiguousarray(body_masses, dtype=np.float64)
    n = idx.numel()
    assert mass.numel() == n
    check(_lib.load().om_h1_draw_models(int(seed), int(env_id0), int(count), len(bm), int(bool(random)), bm.ctypes.data,
                                        _p(idx, torch.int32), _p(mass, torch.float32), n, _stream()))


def h1_reset_envs(dm, spec, traj, qpos, qvel, mask=None, absorbing=None, horizon=0, forced_traj=-1, forced_step=-1,
                  obs_in=None, obs=None, prev_x_vel=None, episode_step=None, last=None, grf=None, partial_resets=None,
                  model_index=None, mass=None, masses=(), random=True, n=None):
    """``om_h1_reset_envs``: LocoEnvBase.reset for the envs of ``mask`` ([ld] bool / uint8), or -- ``mask=None`` -- the
    auto-reset after a step: ``episode_step += 1``, ``last = absorbing | (episode_step >= horizon)``, reset where ``last``.
    Everything is updated in place on the current stream: the trajectory state of ``traj``, qpos [nq, ld], qvel [nv, ld],
    obs [D, ld] (from ``obs_in`` for the envs that do not reset), prev_x_vel, episode_step, last [ld] uint8, grf [G, ld]
    and -- per-env models -- partial_resets, model_index (int32), mass (float32) from the host list ``masses``.
    ld = ``traj.n`` (the width of its state tensors); ``n`` (default ld) envs are processed."""
    _lib.require_cuda()
    ld = traj.n
    n = ld if n is None else int(n)
    for name, t in (("qpos", qpos), ("qvel", qvel), ("obs_in", obs_in), ("obs", obs), ("grf", grf)):
        if t is not None and t.shape[-1] != ld:
            raise ValueError(f"{name} must be a [C, {ld}] SoA tensor")
    if mask is not None and (mask.dtype not in (torch.bool, torch.uint8) or mask.shape != (ld,)):
        raise ValueError(f"mask must be a [{ld}] bool or uint8 tensor")
    i32, f32, u8 = torch.int32, torch.float32, torch.uint8
    bm = np.ascontiguousarray(masses, dtype=np.float64)
    v = lambda t, dt_=None: None if t is None else _p(t, dt_).value
    a = OmH1ResetArgs(mask=v(mask), absorbing=v(absorbing, u8), horizon=int(horizon), forced_traj=int(forced_traj),
                      forced_step=int(forced_step), traj_no=v(traj.traj_no, i32), step_no=v(traj.step_no, i32),
                      reset_count=v(traj.reset_count, i32), xy_off=v(traj.xy_off, torch.float64), qpos=v(qpos, f32),
                      qvel=v(qvel, f32), obs_in=v(obs_in, f32), obs=v(obs, f32), obs_dim=0 if obs is None else obs.shape[0],
                      prev_x_vel=v(prev_x_vel, f32), episode_step=v(episode_step, i32), last=v(last, u8), grf=v(grf, f32),
                      n_grf=0 if grf is None else grf.shape[0], partial_resets=v(partial_resets, i32),
                      model_index=v(model_index, i32), mass=v(mass, f32), n_models=len(bm), random=int(bool(random)),
                      masses_host=bm.ctypes.data if len(bm) else None)
    check(_lib.load().om_h1_reset_envs(dm.handle, C.byref(spec), traj.handle, traj.seed, traj.env_id0, C.byref(a), n, ld,
                                       _stream()))


def fk(dm: DeviceModel, qpos, qvel=None, want=("xpos", "xquat", "site_xpos", "site_xmat", "cvel", "subtree_com"),
       force_generic=False, out=None):
    """K1.  qpos [nq,n], qvel [nv,n] -> dict of SoA tensors."""
    km = dm.km
    n = qpos.shape[-1]
    assert qpos.shape[0] == km.nq and (qvel is None or qvel.shape == (km.nv, n))
    sizes = dict(xpos=km.nbody * 3, xquat=km.nbody * 4, site_xpos=km.nsite * 3, site_xmat=km.nsite * 9,
                 cvel=km.nbody * 6, subtree_com=3)
    out = dict(out or {})
    for k in want:
        if k not in out:
            out[k] = soa(sizes[k], n, device=qpos.device)
    g = lambda k: _p(out.get(k), torch.float32)
    check(_lib.load().om_fk(dm.handle, _p(qpos, torch.float32), _p(qvel, torch.float32), n, qpos.stride(0) if n > 1 else max(n, 1),
                            g("xpos"), g("xquat"), g("site_xpos"), g("site_xmat"), g("cvel"), g("subtree_com"),
                            int(force_generic), _stream()))
    return out


# ------------------------------------------------------------------------------------------- H1
def make_h1_spec(perm, x_vel_idx, target_velocity=1.25, use_absorbing_states=True):
    s = OmH1Spec()
    s.n_obs_q = len(perm)
    for k, v in enumerate(perm):
        s.obs_perm[k] = int(v)
    s.x_vel_idx = int(x_vel_idx)
    s.target_velocity = float(target_velocity)
    s.use_absorbing_states = int(bool(use_absorbing_states))
    return s


def h1_step(dm, spec, qpos, qvel, prev_x_vel, want_fk=True, out=None):
    """K1+K2 fused: FK + observation + absorbing + reward for n envs."""
    km = dm.km
    n = qpos.shape[-1]
    nobs = 2 * spec.n_obs_q - 2
    out = dict(out or {})
    dev = qpos.device
    if want_fk:
        for k, c in (("xpos", km.nbody * 3), ("xquat", km.nbody * 4), ("site_xpos", km.nsite * 3), ("cvel", km.nbody * 6)):
            out.setdefault(k, soa(c, n, device=dev))
    out.setdefault("obs", soa(nobs, n, device=dev))
    out.setdefault("reward", torch.empty(n, device=dev))
    out.setdefault("absorbing", torch.empty(n, dtype=torch.uint8, device=dev))
    g = lambda k: _p(out.get(k), torch.float32)
    check(_lib.load().om_h1_step(dm.handle, C.byref(spec), _p(qpos, torch.float32), _p(qvel, torch.float32),
                                 _p(prev_x_vel, torch.float32), n, max(n, 1), g("xpos"), g("xquat"), g("site_xpos"),
                                 g("cvel"), g("obs"), g("reward"), _p(out["absorbing"], torch.uint8), _stream()))
    return out


def set_sim_state(dm, spec, sample, qpos, qvel):
    """A7: sample [2*n_obs_q, n] (spec order) -> qpos [nq, n], qvel [nv, n] (MJCF order), in place."""
    n = sample.shape[-1]
    check(_lib.load().om_set_sim_state(dm.handle, C.byref(spec), _p(sample, torch.float32), n, max(n, 1),
                                       _p(qpos, torch.float32), _p(qvel, torch.float32), _stream()))


def h1_has_fallen(obs):
    n = obs.shape[-1]
    fallen = torch.empty(n, dtype=torch.uint8, device=obs.device)
    check(_lib.load().om_h1_has_fallen(_p(obs, torch.float32), n, max(n, 1), _p(fallen), _stream()))
    return fallen


# ------------------------------------------------------------------------------------------- trajectory
class DeviceTrajectory:
    """OmTraj handle + per-env integer state for n envs (K3)."""

    def __init__(self, table, n_env, seed=0, env_id0=0, device="cuda"):
        _lib.require_cuda()
        table = np.ascontiguousarray(table, dtype=np.float64)
        assert table.ndim == 3, "table must be [K, n_traj, T]"
        self.K, self.n_traj, self.T = table.shape
        h = C.c_void_p()
        check(_lib.load().om_traj_create(table.ctypes.data, self.K, self.n_traj, self.T, C.byref(h)))
        self.handle = h
        self.n, self.seed, self.env_id0 = int(n_env), int(seed), int(env_id0)
        self.traj_no = torch.zeros(n_env, dtype=torch.int32, device=device)
        self.step_no = torch.zeros(n_env, dtype=torch.int32, device=device)
        self.reset_count = torch.zeros(n_env, dtype=torch.int32, device=device)   # bits of a uint32
        self.xy_off = torch.zeros((2, n_env), dtype=torch.float64, device=device)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                _lib.load().om_traj_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def reset(self, mask=None, traj_no=None, substep_no=None, sample=None):
        if sample is None:
            sample = soa(self.K, self.n, device=self.traj_no.device)
        check(_lib.load().om_traj_reset(self.handle, self.seed, self.env_id0, _p(mask, torch.uint8),
                                        _p(traj_no, torch.int32), _p(substep_no, torch.int32), _p(self.traj_no),
                                        _p(self.step_no), _p(self.reset_count), _p(self.xy_off), _p(sample, torch.float32),
                                        self.n, max(self.n, 1), _stream()))
        return sample

    def current(self, sample=None):
        if sample is None:
            sample = soa(self.K, self.n, device=self.traj_no.device)
        check(_lib.load().om_traj_current(self.handle, _p(self.traj_no), _p(self.step_no), _p(self.xy_off),
                                          _p(sample, torch.float32), self.n, max(self.n, 1), _stream()))
        return sample

    def next(self, sample=None, wrapped=None, auto_reset=True):
        if sample is None:
            sample = soa(self.K, self.n, device=self.traj_no.device)
        check(_lib.load().om_traj_next(self.handle, self.seed, self.env_id0, int(bool(auto_reset)), _p(self.traj_no), _p(self.step_no),
                                       _p(self.reset_count), _p(self.xy_off), _p(sample, torch.float32),
                                       _p(wrapped, torch.uint8), self.n, max(self.n, 1), _stream()))
        return sample


def h1_play_from_velocity(dm, spec, traj: DeviceTrajectory, state, n_steps, dt=0.01, end_episode_reset=True,
                          want=("xpos", "xquat", "site_xpos", "cvel", "obs", "reward", "fallen", "traj_no_t", "step_no_t"),
                          out=None, forced=False, obs_moments=None, start_reset=False):
    """Fused playback of one episode (loco_env_base.py:511-557) on any UnitreeH1 model with ``dm.h1_variant != 0``.
    ``state``: dict with curr_qpos [NQ,n] f64, pending [2 NQ,n] f32, prev_x_vel [n] f32 (the trajectory indices live in
    ``traj``; NQ = ``spec.n_obs_q``, 17 for the default model).  ``forced``: play_trajectory semantics
    (loco_env_base.py:404-432), the model is set to each sample instead of integrating velocities.
    ``obs_moments``: float64 [2 nobs + 1] device buffer (nobs = 2 NQ - 2; 65 values for the default model); the kernel
    ADDS sum[nobs], sumsq[nobs], count of the observations it emits
    (S1 fused into the playback: no second pass over the observation buffer).  ``start_reset``: the call begins with
    the reference's ``reset()`` (loco_env_base.py:481), performed inside the kernel (no state tensor is read before it)."""
    km, n = dm.km, traj.n
    dev = traj.traj_no.device
    nobs = 2 * spec.n_obs_q - 2
    sizes = dict(xpos=(km.nbody * 3, torch.float32), xquat=(km.nbody * 4, torch.float32),
                 site_xpos=(km.nsite * 3, torch.float32), cvel=(km.nbody * 6, torch.float32),
                 obs=(nobs, torch.float32), reward=(None, torch.float32), fallen=(None, torch.uint8),
                 traj_no_t=(None, torch.int32), step_no_t=(None, torch.int32))
    out = dict(out or {})
    for k in want:
        if k not in out:
            c, dt_ = sizes[k]
            out[k] = torch.empty((n_steps, n) if c is None else (n_steps, c, n), dtype=dt_, device=dev)
    cq = state.get("curr_qpos")
    ps = OmPlayState(traj_no=traj.traj_no.data_ptr(), step_no=traj.step_no.data_ptr(),
                     reset_count=traj.reset_count.data_ptr(), xy_off=traj.xy_off.data_ptr(),
                     curr_qpos=None if cq is None else _p(cq, torch.float64).value,
                     pending=_p(state["pending"], torch.float32).value,
                     prev_x_vel=_p(state["prev_x_vel"], torch.float32).value)
    po = OmPlayOut(**{k: (out[k].data_ptr() if k in out else None) for k in sizes})
    if obs_moments is not None:
        if obs_moments.numel() != 2 * nobs + 1:
            raise ValueError(f"obs_moments must hold 2 * {nobs} + 1 float64 values")
        po.obs_moments = _p(obs_moments, torch.float64).value
    flags = (1 if end_episode_reset else 0) | (2 if start_reset else 0)
    if forced:
        check(_lib.load().om_h1_play_trajectory(dm.handle, C.byref(spec), traj.handle, traj.seed, traj.env_id0, int(n_steps),
                                                flags, C.byref(ps), C.byref(po), n, max(n, 1), _stream()))
    else:
        check(_lib.load().om_h1_play_from_velocity(dm.handle, C.byref(spec), traj.handle, traj.seed, traj.env_id0, float(dt),
                                                   int(n_steps), flags, C.byref(ps), C.byref(po), n, max(n, 1), _stream()))
    return out


class H1LiveStep:
    """``om_h1_live_step`` with every argument bound once: one fused kernel per env step (next sample / wrap reset +
    set_sim_state + FK + observation + has_fallen + reward), one ctypes call per step with no per-call marshalling --
    the eager Python loop stays within a few microseconds of host time per step.  ``out``: dict of SoA tensors (any of
    qpos, qvel, xpos, xquat, site_xpos, cvel, obs, reward, absorbing, wrapped); missing FK / mirror outputs are not
    computed.  ``prev_x_vel`` [n] float32 is carried in place.  Graph-capturable.  ``keys``: (components, dtype) of
    each output for this model (``KEYS``: the default model's)."""

    KEYS = dict(qpos=(17, torch.float32), qvel=(17, torch.float32), xpos=(63, torch.float32), xquat=(84, torch.float32),
                site_xpos=(3, torch.float32), cvel=(126, torch.float32), obs=(32, torch.float32), reward=(None, torch.float32),
                absorbing=(None, torch.uint8), wrapped=(None, torch.uint8))

    @staticmethod
    def keys_for(dm, spec):
        km = dm.km
        return dict(H1LiveStep.KEYS, qpos=(km.nq, torch.float32), qvel=(km.nv, torch.float32),
                    xpos=(km.nbody * 3, torch.float32), xquat=(km.nbody * 4, torch.float32),
                    site_xpos=(km.nsite * 3, torch.float32), cvel=(km.nbody * 6, torch.float32),
                    obs=(2 * spec.n_obs_q - 2, torch.float32))

    def __init__(self, dm, spec, traj: DeviceTrajectory, prev_x_vel, out=None,
                 want=("xpos", "xquat", "site_xpos", "cvel", "obs", "reward", "absorbing")):
        n, dev = traj.n, traj.traj_no.device
        self.dm, self.spec, self.traj, self.n = dm, spec, traj, n
        self.keys = self.keys_for(dm, spec)
        self.prev_x_vel = prev_x_vel
        self.out = dict(out or {})
        for k in want:
            if k not in self.out:
                c, dt_ = self.keys[k]
                self.out[k] = torch.empty((n,) if c is None else (c, n), dtype=dt_, device=dev)
        self._fn = _lib.load().om_h1_live_step
        self.rebind()

    def rebind(self, out=None, stream=None):
        """Point the call at other output tensors (e.g. the next time slot of a rollout buffer) / another stream."""
        if out is not None:
            self.out.update(out)
        traj = self.traj
        self._state = OmLiveState(traj_no=traj.traj_no.data_ptr(), step_no=traj.step_no.data_ptr(),
                                  reset_count=traj.reset_count.data_ptr(), xy_off=traj.xy_off.data_ptr(),
                                  prev_x_vel=_p(self.prev_x_vel, torch.float32).value)
        self._out = OmLiveOut(**{k: _p(v, self.keys[k][1]).value for k, v in self.out.items()})
        st = torch.cuda.current_stream().cuda_stream if stream is None else stream
        self._args = (self.dm.handle, C.byref(self.spec), traj.handle, traj.seed, traj.env_id0, C.byref(self._state),
                      C.byref(self._out), self.n, max(self.n, 1), C.c_void_p(st))
        return self

    def __call__(self):
        if self._fn(*self._args):
            check(1)
        return self.out


# ------------------------------------------------------------------------------------------- A3
A3_NINT, A3_MAX_STEPS, A3_NOBS = 7, 20, 41
A3_FK_SIZES = dict(xpos=17 * 3, xquat=17 * 4, site_xpos=2 * 3, site_xmat=2 * 9, cvel=17 * 6)


class A3Task:
    """OmA3Task handle (constants of the WalkingTask) + per-env task state for n envs."""

    def __init__(self, dm: DeviceModel, n_env, clock_lut, init_qpos, period=88, delay_frames=30, target_radius=0.20,
                 goal_height_ref=0.80, goal_speed_ref=0.0, seed=0, env_id0=0, device="cuda"):
        _lib.require_cuda()
        lut = np.ascontiguousarray(clock_lut, dtype=np.float64)
        iq = np.ascontiguousarray(init_qpos, dtype=np.float64)
        assert lut.shape == (period, 4) and iq.shape == (dm.km.nq,)
        desc = OmA3TaskDesc(period=period, delay_frames=delay_frames, target_radius=target_radius,
                            goal_height_ref=goal_height_ref, goal_speed_ref=goal_speed_ref,
                            total_mass=float(dm.km.total_mass), clock_lut_host=lut.ctypes.data, init_qpos_host=iq.ctypes.data)
        h = C.c_void_p()
        check(_lib.load().om_a3_task_create(C.byref(desc), C.byref(h)))
        self.handle, self.dm = h, dm
        self.n, self.seed, self.env_id0 = int(n_env), int(seed), int(env_id0)
        self.ints = torch.zeros((A3_NINT, n_env), dtype=torch.int32, device=device)
        self.sequence = torch.zeros((A3_MAX_STEPS * 4, n_env), dtype=torch.float32, device=device)
        self.reset_count = torch.zeros(n_env, dtype=torch.int32, device=device)          # bits of a uint32

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                _lib.load().om_a3_task_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def _state(self):
        return OmA3State(ints=self.ints.data_ptr(), sequence=self.sequence.data_ptr())

    def reset(self, qpos, qvel, mask=None, iteration_count=0.0, obs=None):
        """reset_model + WalkingTask.reset for the masked envs: fills qpos [25,n], qvel [24,n], the task state and obs."""
        if obs is None:
            obs = soa(A3_NOBS, self.n, device=self.ints.device)
        st = self._state()
        check(_lib.load().om_a3_reset(self.dm.handle, self.handle, self.seed, self.env_id0, _p(mask, torch.uint8),
                                      _p(self.reset_count), float(iteration_count), _p(qpos, torch.float32),
                                      _p(qvel, torch.float32), C.byref(st), _p(obs, torch.float32), self.n, max(self.n, 1),
                                      _stream()))
        return obs

    def autoreset(self, qpos, qvel, done, traj_len, obs_in, obs, last, path_end, max_traj_len=None, iteration_count=0.0,
                  n=None):
        """``om_a3_autoreset``: the PPO sampler's path bookkeeping after a one-step ``step`` (rl/algos/ppo.py:150-198):
        ``traj_len += 1``; a path ends on ``done`` or at ``max_traj_len`` (None = never); ``last`` = it ended, ``path_end`` =
        1 (done) / 2 (truncated) / 0, the codes of ``ppo_returns``; an env whose path ended is reset as ``reset(mask=last)``
        resets it and ``traj_len`` restarts at 0.  ``obs`` = ``obs_in`` (the step's observation) where no reset happened, the
        new first observation where one did.  Everything in place on the current stream: qpos [25, ld], qvel [24, ld], the
        task state, reset_count, traj_len (int32 [ld]), obs [41, ld], last / path_end ([ld] uint8 or bool).  done ([ld]
        uint8 or bool), obs_in [41, ld].  ld = ``self.n``; ``n`` (default ld) envs are processed."""
        ld = self.n
        n = ld if n is None else int(n)
        if not 0 <= n <= ld:
            raise ValueError(f"n = {n} outside [0, {ld}]")
        if max_traj_len is not None and int(max_traj_len) < 1:
            raise ValueError(f"max_traj_len must be None or >= 1, got {max_traj_len}")
        for name, t, rows in (("qpos", qpos, 25), ("qvel", qvel, 24), ("obs_in", obs_in, A3_NOBS), ("obs", obs, A3_NOBS)):
            if t.shape != (rows, ld) or t.dtype != torch.float32:
                raise ValueError(f"{name} must be a float32 [{rows}, {ld}] SoA tensor")
        for name, t, dts in (("done", done, (torch.uint8, torch.bool)), ("last", last, (torch.uint8, torch.bool)),
                             ("path_end", path_end, (torch.uint8,)), ("traj_len", traj_len, (torch.int32,))):
            if t.shape != (ld,) or t.dtype not in dts:
                raise ValueError(f"{name} must be a [{ld}] {' or '.join(str(d) for d in dts)} tensor")
        _lib.require_cuda()
        v = lambda t: _p(t).value
        a = OmA3AutoResetArgs(done=v(done), max_traj_len=0 if max_traj_len is None else int(max_traj_len),
                              iteration_count=float(iteration_count), reset_count=v(self.reset_count), traj_len=v(traj_len),
                              qpos=v(qpos), qvel=v(qvel), state=self._state(), obs_in=v(obs_in), obs=v(obs), last=v(last),
                              path_end=v(path_end))
        check(_lib.load().om_a3_autoreset(self.dm.handle, self.handle, self.seed, self.env_id0, C.byref(a), n, max(ld, 1),
                                          _stream()))

    def step(self, qpos, qvel, contact, want=("obs", "terms", "reward", "done"), out=None, returns=None):
        """The StickFigureA3.step tail on post-physics states.  qpos [25,n] (one step) or [T,25,n] (replay of T
        recorded steps); qvel / contact ([4,n]: l_grf, r_grf, min contact z, flags) likewise.
        ``returns``: dict(values [T,n], gamma, v_next=None, v_last=None, path_end=None) -- the rollout is finished with
        PPOBuffer.finish_path's discounted returns by the same call (``om_a3_task_rollout``); ``out`` then also holds
        ``ret`` and ``adv`` [T,n]."""
        T = 1 if qpos.dim() == 2 else qpos.shape[0]
        n, dev = self.n, qpos.device
        assert qpos.shape[-2:] == (25, n) and qvel.shape[-2:] == (24, n) and contact.shape[-2:] == (4, n)
        sizes = dict(obs=(A3_NOBS, torch.float32), terms=(6, torch.float32), reward=(None, torch.float32),
                     done=(None, torch.uint8), **{k: (c, torch.float32) for k, c in A3_FK_SIZES.items()})
        out = dict(out or {})
        for k in want:
            if k not in out:
                c, dt_ = sizes[k]
                shape = ((n,) if c is None else (c, n)) if qpos.dim() == 2 else ((T, n) if c is None else (T, c, n))
                out[k] = torch.empty(shape, dtype=dt_, device=dev)
        for k, t in out.items():
            _p(t, torch.float32 if k in ("ret", "adv") else sizes[k][1])
        po = OmA3Out(**{k: (out[k].data_ptr() if k in out else None) for k in sizes})
        st = self._state()
        if returns is not None:
            assert qpos.dim() == 3 and "reward" in out and "done" in out
            for k in ("ret", "adv"):
                if k not in out:
                    out[k] = torch.empty((T, n), dtype=torch.float32, device=dev)
            g = lambda k, dt_=torch.float32: None if returns.get(k) is None else _p(returns[k], dt_).value
            pr = OmA3Returns(values=g("values"), v_next=g("v_next"), v_last=g("v_last"), path_end=g("path_end", torch.uint8),
                             gamma=float(returns["gamma"]), ret=out["ret"].data_ptr(), adv=out["adv"].data_ptr())
            check(_lib.load().om_a3_task_rollout(self.dm.handle, self.handle, _p(qpos, torch.float32), _p(qvel, torch.float32),
                                                 _p(contact, torch.float32), T, C.byref(st), C.byref(po), C.byref(pr), n,
                                                 max(n, 1), _stream()))
            return out
        check(_lib.load().om_a3_task_step(self.dm.handle, self.handle, _p(qpos, torch.float32), _p(qvel, torch.float32),
                                          _p(contact, torch.float32), T, C.byref(st), C.byref(po), n, max(n, 1), _stream()))
        return out


# ------------------------------------------------------------------------------------------- actions (N1)
def make_action_spec(delta, mean):
    sp = OmActionSpec()
    sp.nu = len(delta)
    for a, (d, m) in enumerate(zip(delta, mean)):
        sp.delta[a], sp.mean[a] = float(d), float(m)
    return sp


def make_pd_spec(qposadr, dofadr, kp, kd, gear, offset):
    sp = OmPdSpec()
    sp.nu = len(qposadr)
    for a in range(sp.nu):
        sp.qposadr[a], sp.dofadr[a] = int(qposadr[a]), int(dofadr[a])
        sp.kp[a], sp.kd[a], sp.gear[a], sp.offset[a] = float(kp[a]), float(kd[a]), float(gear[a]), float(offset[a])
    return sp


def action_affine(spec, action, out=None):
    """_preprocess_action: action [nu, n] in [-1, 1] -> ctrl [nu, n]."""
    n = action.shape[-1]
    out = torch.empty_like(action) if out is None else out
    check(_lib.load().om_action_affine(C.byref(spec), _p(action, torch.float32), n, max(n, 1), _p(out, torch.float32), _stream()))
    return out


def pd_torque(spec, target, qpos, qvel, vel_target=None, add_offset=True, out=None):
    """robot.py do_simulation inner body: target [nu, n] (+ motor offset), qpos [nq, n], qvel [nv, n] -> ctrl [nu, n]."""
    n = target.shape[-1]
    out = torch.empty_like(target) if out is None else out
    check(_lib.load().om_pd_torque(C.byref(spec), _p(target, torch.float32), _p(vel_target, torch.float32),
                                   _p(qpos, torch.float32), _p(qvel, torch.float32), int(bool(add_offset)), n, max(n, 1),
                                   _p(out, torch.float32), _stream()))
    return out


def make_mirror_spec(mirrored, clock_inds=()):
    """``mirrored`` as the reference writes it (signed indices, 0 encoded as +-0.1; StickFigureA3.py:118-129)."""
    sp = OmMirrorSpec()
    sp.numel = len(mirrored)
    for i, m in enumerate(mirrored):
        sp.index[i] = int(abs(int(m)))
        sp.sign[i] = float(np.sign(m))
    for c in clock_inds:
        sp.negate[int(c)] = 1
    return sp


def mirror(spec, x, out=None):
    """SymmetricEnv.mirror_observation / mirror_action (/ mirror_clock_observation with clock_inds): x [numel, n]."""
    n = x.shape[-1]
    out = torch.empty_like(x) if out is None else out
    check(_lib.load().om_mirror(C.byref(spec), _p(x, torch.float32), n, max(n, 1), _p(out, torch.float32), _stream()))
    return out


def ppo_loss_stats(logp, old_logp, adv, clip, mask=None, values=None, returns=None, vf_coeff=0.5, entropy=None, act=None,
                   act_mirror=None, action_mirror=None, want_grad=True, out=None):
    """N3: PPO.update_policy's losses in one pass (layout in include/om_b200.h) -> (sums float64 [7], dlogp, dvalues)."""
    n = logp.numel()
    nu = 0 if act is None and entropy is None else (act if act is not None else entropy).shape[0]
    if out is None:
        out = torch.zeros(7, dtype=torch.float64, device=logp.device)
    dlogp = torch.empty(n, device=logp.device) if want_grad else None
    dvalues = torch.empty(n, device=logp.device) if (want_grad and values is not None) else None
    check(_lib.load().om_ppo_loss_stats(_p(logp, torch.float32), _p(old_logp, torch.float32), _p(adv, torch.float32),
                                        _p(mask, torch.float32), _p(values, torch.float32), _p(returns, torch.float32),
                                        _p(entropy, torch.float32), _p(act, torch.float32), _p(act_mirror, torch.float32),
                                        C.byref(action_mirror) if action_mirror is not None else None, int(nu), n, max(n, 1),
                                        float(clip), float(vf_coeff), _p(out, torch.float64), _p(dlogp), _p(dvalues),
                                        _stream()))
    return out, dlogp, dvalues


# ------------------------------------------------------------------------------------------- discriminator (K4)
class Discriminator:
    """OmDisc handle.  ``params``: dict of float32 arrays in torch.nn.Linear layout ([out, in] weights):
    VAIL  w1 b1 w2 b2 wmu bmu wlv blv wd bd   (n_in-256-128-z128-1)
    GAIL  w1 b1 w2 b2 w3 b3                   (n_in-512-256-1)
    ``n_in`` (the columns of w1) is 1..64: the kinematic observation of any UnitreeH1 variant,
    ``env.get_kinematic_obs_mask()`` (32 for the default model, 30 without the back joint, 48 with arms, 46 with arms
    and without the back joint)."""

    def __init__(self, kind, params):
        _lib.require_cuda()
        kind = {"vail": 0, "gail": 1}[kind.lower()] if isinstance(kind, str) else int(kind)
        f = lambda k: np.ascontiguousarray(params[k], dtype=np.float32)
        keep = dict(w1=f("w1"), b1=f("b1"), w2=f("w2"), b2=f("b2"))
        if kind == 0:
            keep.update(wmu=f("wmu"), bmu=f("bmu"), wlv=f("wlv"), blv=f("blv"), wd=f("wd"), bd=f("bd"))
        else:
            keep.update(wd=f("w3"), bd=f("b3"))
        n_h1, n_in = keep["w1"].shape
        n_h2 = keep["w2"].shape[0]
        assert keep["w2"].shape[1] == n_h1
        z = keep["wmu"].shape[0] if kind == 0 else 0
        desc = OmDiscDesc(kind=kind, n_in=n_in, n_h1=n_h1, n_h2=n_h2, z_size=z,
                          **{k: v.ctypes.data for k, v in keep.items()})
        h = C.c_void_p()
        check(_lib.load().om_disc_create(C.byref(desc), C.byref(h)))
        self.handle, self.kind, self.n_in, self.z = h, kind, n_in, z

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                _lib.load().om_disc_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def reward(self, s, mean, std, eps=None, want_d=False):
        """s [n_in, n] observations (SoA), mean / std [n_in] float32 device tensors, eps [z, n] or None -> reward [n]
        (and the raw logit d [n] when ``want_d``)."""
        n = s.shape[-1]
        assert s.shape == (self.n_in, n) and (eps is None or eps.shape == (self.z, n))
        assert mean.numel() == self.n_in and std.numel() == self.n_in
        reward = torch.empty(n, device=s.device)
        d = torch.empty(n, device=s.device) if want_d else None
        check(_lib.load().om_disc_reward(self.handle, _p(s, torch.float32), _p(mean, torch.float32), _p(std, torch.float32),
                                         _p(eps, torch.float32), n, max(n, 1), _p(reward), _p(d), _stream()))
        return (reward, d) if want_d else reward


    def forward(self, s, mean, std, eps=None, want_reward=False, want_kl=None):
        """The forward pass of the discriminator FIT (gail_TRPO.py:167-220): -> dict(logit [n], kl [n] (VAIL),
        reward [n] if asked) for s [n_in, n].  Same kernel as ``reward``; the KL term is VDBLoss.kl_divergence per sample."""
        n = s.shape[-1]
        assert s.shape == (self.n_in, n) and (eps is None or eps.shape == (self.z, n))
        assert mean.numel() == self.n_in and std.numel() == self.n_in
        want_kl = (self.kind == 0) if want_kl is None else want_kl
        out = dict(logit=torch.empty(n, device=s.device))
        if want_kl:
            out["kl"] = torch.empty(n, device=s.device)
        if want_reward:
            out["reward"] = torch.empty(n, device=s.device)
        check(_lib.load().om_disc_forward(self.handle, _p(s, torch.float32), _p(mean, torch.float32), _p(std, torch.float32),
                                          _p(eps, torch.float32), n, max(n, 1), _p(out.get("reward")), _p(out["logit"]),
                                          _p(out.get("kl")), _stream()))
        return out


def disc_loss_stats(logit, n_plcy, target=None, kl=None, entcoeff=1e-3, want_grad=False, out=None):
    """N2: statistics of one discriminator-fit batch (layout in include/om_b200.h) accumulated into a float64 [9]
    buffer; with ``want_grad`` also d(sum bce - entcoeff * sum entropy)/d logit per sample."""
    n = logit.numel()
    if out is None:
        out = torch.zeros(9, dtype=torch.float64, device=logit.device)
    grad = torch.empty_like(logit) if want_grad else None
    check(_lib.load().om_disc_loss_stats(_p(logit, torch.float32), _p(target, torch.float32), _p(kl, torch.float32),
                                         int(n_plcy), int(n - n_plcy), float(entcoeff), _p(out, torch.float64), _p(grad),
                                         _stream()))
    return (out, grad) if want_grad else out


def expert_minibatch(src, n_src, seed, draw, batch, want_next=False, want_idx=False):
    """N2: src [D, >= n_src (+1)] device-resident expert states -> (states [D, batch], next_states | None, idx | None)
    by the keyed-permutation contract of om_expert_minibatch."""
    d, ld = src.shape
    out = torch.empty((d, batch), device=src.device)
    nxt = torch.empty((d, batch), device=src.device) if want_next else None
    idx = torch.empty(batch, dtype=torch.int32, device=src.device) if want_idx else None
    check(_lib.load().om_expert_minibatch(_p(src, torch.float32), int(n_src), ld, d, int(seed), int(draw), int(batch),
                                          _p(out), _p(nxt), _p(idx, torch.int32), max(batch, 1), _stream()))
    return out, nxt, idx


# ------------------------------------------------------------------------------------------- learner side
def ppo_returns(rewards, values, gamma, path_end=None, v_next=None, v_last=None):
    """K5a over a [T, n] buffer -> (returns, advantages)."""
    T, n = rewards.shape
    ret, adv = torch.empty_like(rewards), torch.empty_like(rewards)
    check(_lib.load().om_ppo_returns(_p(rewards, torch.float32), _p(values, torch.float32), _p(path_end, torch.uint8),
                                     _p(v_next, torch.float32), _p(v_last, torch.float32), float(gamma), T, n, max(n, 1),
                                     _p(ret), _p(adv), _stream()))
    return ret, adv


def gae(rewards, v, v_next, absorbing, last, gamma, lam):
    """K5b over a [T, n] buffer -> (v_target, adv) (the order compute_gae returns)."""
    T, n = rewards.shape
    adv, vt = torch.empty_like(rewards), torch.empty_like(rewards)
    check(_lib.load().om_gae(_p(rewards, torch.float32), _p(v, torch.float32), _p(v_next, torch.float32),
                             _p(absorbing, torch.uint8), _p(last, torch.uint8), float(gamma), float(lam), T, n, max(n, 1),
                             _p(adv), _p(vt), _stream()))
    return vt, adv


def moments(x, out=None):
    """K6.  x [C, n] or [rows, C, n] -> float64 [2C+1] = (sum[C], sumsq[C], count), accumulated into ``out``."""
    if x.dim() == 1:
        x = x.view(1, 1, -1)
    elif x.dim() == 2:
        x = x.view(1, *x.shape)
    rows, c, n = x.shape
    if out is None:
        out = torch.zeros(2 * c + 1, dtype=torch.float64, device=x.device)
    if out.numel() != 2 * c + 1:
        raise ValueError(f"moments of {c} components need a {2 * c + 1}-element output, got {out.numel()}")
    check(_lib.load().om_moments(_p(x, torch.float32), rows, c, n, max(n, 1), _p(out, torch.float64), _stream()))
    return out


def moments_scalar(x, out=None):
    """K6 for a single-component buffer ([n] or [T, n], e.g. advantages) -> float64 [3] = (sum, sumsq, count)."""
    x3 = x.reshape(1, 1, -1) if x.dim() == 1 else x.unsqueeze(1)
    if out is not None and out.numel() != 3:
        raise ValueError("moments_scalar needs a 3-element output")
    return moments(x3, out=out)


def adv_stats(mom, unbiased, eps):
    stats = torch.empty(2, dtype=torch.float64, device=mom.device)
    check(_lib.load().om_adv_stats(_p(mom, torch.float64), int(bool(unbiased)), float(eps), _p(stats), _stream()))
    return stats


MOMENT_KINDS = dict(standardizer=0, ppo_obs=1, adv_ppo=2, adv_gail=3)


def moment_stats(mom, kind, want32=False):
    """(mean [C], denominator [C]) float64 from a moment buffer [sum[C], sumsq[C], count] in one kernel (the formulas of
    ``distributed.mean_std_from_moments``); with ``want32`` also float32 copies (what ``Discriminator.reward`` takes)."""
    c = (mom.numel() - 1) // 2
    mean = torch.empty(c, dtype=torch.float64, device=mom.device)
    denom = torch.empty(c, dtype=torch.float64, device=mom.device)
    m32 = torch.empty(c, dtype=torch.float32, device=mom.device) if want32 else None
    d32 = torch.empty(c, dtype=torch.float32, device=mom.device) if want32 else None
    check(_lib.load().om_moment_stats(_p(mom, torch.float64), c, MOMENT_KINDS[kind], _p(mean), _p(denom), _p(m32), _p(d32),
                                      _stream()))
    return (mean, denom, m32, d32) if want32 else (mean, denom)


def normalize(x, stats, out=None):
    """(x - stats[0]) / stats[1] over a [rows, n] buffer."""
    x2 = x.view(1, -1) if x.dim() == 1 else x
    rows, n = x2.shape
    out = torch.empty_like(x) if out is None else out
    check(_lib.load().om_normalize(_p(x2, torch.float32), _p(stats, torch.float64), rows, n, max(n, 1),
                                   _p(out, torch.float32), _stream()))
    return out


def debug_set(knob, value):
    """Tuning / test hook (``om_debug_set``): force a kernel variant; -1 / 0 = automatic."""
    check(_lib.load().om_debug_set(knob.encode(), int(value)))


def launch_count():
    return int(_lib.load().om_launch_count())


def reset_launch_count():
    _lib.load().om_reset_launch_count()
