"""GPU: the benchmarked H1 rollouts at FULL size against the float64 C oracle (oracle/c), every env and every step.

* configs[1]: ``bench.py``'s ``hot_step`` three times in a row on one environment (4096 envs x 500 steps on the bench's
  [34, 4, 500] table): the first call resets through the Python API, the later ones inside the kernel; the observation
  moments are fused into the playback; GAE, the advantage moments, ``adv_stats`` and the in-place ``normalize`` follow.
* configs[4]: one shard of the 1 M-env run (131072 envs at env_id0 = 917504), two rollouts of two 32-step calls (the
  second continues the first's episode), the observation moments and ``moment_stats(.., "ppo_obs")``.

The oracle plays the same calls on a carried per-env state (``c_oracle.play_state``) in env blocks, and each block is
compared on the device.  Tolerance: ``|a - ref| <= 1e-5 max(|ref|, 1)`` unless an array names a tighter bound; the one
looser bound, the linear part of ``cvel``, is written out and derived at ``CVEL_LIN_ROUNDINGS``.  Every array's worst
error, where it is and its error / tolerance are printed (run with ``-rP`` to keep them in the log)."""
import time

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BLOCK_ENV_STEPS = 1 << 18          # oracle block: ~256 k env-steps, ~650 MB of float64 outputs


class Worst:
    """Largest error of one array over every comparison made, and the first place it breaks its bound.  The bound is
    ``max(atol, rtol |ref|)`` (the default: 1e-5 max(|ref|, 1)); ``exact=True`` asks for equality."""

    def __init__(self, name, rtol=1e-5, atol=1e-5, exact=False, bound=None):
        self.name, self.rtol, self.atol, self.exact = name, rtol, atol, exact
        self.bound = bound or f"max({atol:g}, {rtol:g} |ref|)"
        self.ratio, self.err, self.ref, self.where, self.first_bad, self.n_bad, self.count = 0.0, 0.0, 0.0, "-", None, 0, 0

    def add(self, a, ref, where, axes=("env", "step", "ch"), env0=0, extra=None):
        """a, ref: float64 device tensors of one shape, axes named by ``axes`` (the env axis first); ``env0`` is the
        global index of env 0; ``where`` names the call; ``extra``: a written error term added to the bound."""
        import torch
        err = (a - ref).abs()
        if self.exact:
            bad = a != ref
            ratio = err
        else:
            tol = torch.clamp(self.rtol * ref.abs(), min=self.atol)
            ratio = err / (tol if extra is None else tol + extra)
            ratio = torch.nan_to_num(ratio, nan=float("inf"))
            bad = ratio > 1.0
        self.count += a.numel()

        def loc(flat):
            idx = np.unravel_index(int(flat), tuple(a.shape))
            parts = [f"{n} {i + (env0 if n == 'env' else 0)}" for n, i in zip(axes, idx)]
            return " ".join([where] + parts)
        flat = int(torch.argmax(ratio))
        r = float(ratio.reshape(-1)[flat])
        if r > self.ratio or self.where == "-":
            self.ratio, self.err, self.ref = r, float(err.reshape(-1)[flat]), float(ref.reshape(-1)[flat])
            self.where = loc(flat)
        nb = int(bad.sum())
        if nb:
            self.n_bad += nb
            if self.first_bad is None:                   # the earliest step that breaks the bound, its lowest env
                if len(axes) > 1 and axes[1] == "step":
                    per_step = bad.reshape(bad.shape[0], bad.shape[1], -1).any(dim=2)    # [env, step]
                    s = int(per_step.any(dim=0).nonzero()[0])
                    e = int(per_step[:, s].nonzero()[0])
                    self.first_bad = f"{where} env {e + env0} step {s}"
                else:
                    self.first_bad = loc(int(bad.reshape(-1).nonzero()[0]))

    def line(self):
        if self.exact:
            return (f"{self.name:<24} exact: {self.n_bad} of {self.count} values differ, worst |err| {self.err:.3g} "
                    f"at {self.where}" + (f"; first at {self.first_bad}" if self.first_bad else ""))
        return (f"{self.name:<24} worst |err| {self.err:.3g} (ref {self.ref:.4g}) at {self.where}, err/tol {self.ratio:.3g} "
                f"(bound {self.bound}, {self.count} values)"
                + (f"; {self.n_bad} over, first at {self.first_bad}" if self.first_bad else ""))

    @property
    def ok(self):
        return self.n_bad == 0


class Report:
    def __init__(self, title):
        self.title, self.arrays, self.t0 = title, {}, time.perf_counter()

    def __call__(self, name, **kw):
        if name not in self.arrays:
            self.arrays[name] = Worst(name, **kw)
        return self.arrays[name]

    def finish(self):
        print(f"== {self.title}: {time.perf_counter() - self.t0:.1f} s")
        for w in self.arrays.values():
            print(f"{self.title} {w.line()}")
        bad = [w.line() for w in self.arrays.values() if not w.ok and "reported only" not in w.bound]
        assert not bad, "\n".join(bad)


@pytest.fixture(scope="module")
def bench_setup():
    """The bench's model and table (built once: ~14 s), the table as the device stores it (channels >= 2 rounded to fp32,
    x and y float64) and the oracle's model."""
    import bench
    from oracle import c_oracle
    from oracle import h1 as OH
    model, table = bench.build_table()
    tab = table.copy()
    tab[2:] = tab[2:].astype(np.float32).astype(np.float64)
    c_oracle.use_all_cores()
    return model, table, tab, c_oracle.CModel(model), OH.perm(model)


def _pinned_buffers(model, K, n, T):
    """c_oracle.h1_play_buffers in page-locked host memory (the blocks are copied to the device for the comparison)."""
    import torch
    f = lambda *s, dt=torch.float64: torch.empty(s, dtype=dt, pin_memory=True).numpy()
    return dict(xpos=f(n, T, model.nbody * 3), xquat=f(n, T, model.nbody * 4), site_xpos=f(n, T, model.nsite * 3),
                cvel=f(n, T, model.nbody * 6), obs=f(n, T, K - 2), reward=f(n, T), fallen=f(n, T, dt=torch.uint8),
                traj_no=f(n, T, dt=torch.int32), step_no=f(n, T, dt=torch.int32), checksum=np.zeros(n))


def _play_and_compare(rep, where, setup, seed, env_id0, state, start_reset, out, play_state, n_steps):
    """The oracle's side of one playback call, block by block, against the device's rollout buffers ``out`` ([T, C, n])
    and carried state ``play_state``; updates the oracle ``state`` in place.  Returns the float64 sums and sums of squares
    of the oracle's observations (the call's moment sums)."""
    import torch
    from oracle import c_oracle
    model, _, tab, cm, perm = setup
    K = tab.shape[0]
    n = state["traj_no"].shape[0]
    blk = max(128, BLOCK_ENV_STEPS // n_steps // 128 * 128)
    buf = _pinned_buffers(model, K, min(blk, n), n_steps)
    dev = lambda a: torch.from_numpy(a).to("cuda").double()
    s1 = np.zeros(K - 2)
    s2 = np.zeros(K - 2)
    for e0 in range(0, n, blk):
        e1 = min(n, e0 + blk)
        b = {k: v[:e1 - e0] for k, v in buf.items()}
        c_oracle.h1_play(cm, perm, tab, seed, env_id0 + e0, e1 - e0, n_steps, out=b, start_reset=start_reset,
                         state={k: v[e0:e1] for k, v in state.items()})
        o = b["obs"]
        s1 += o.sum(axis=(0, 1))
        s2 += np.einsum("etc,etc->c", o, o)
        got = lambda k: out[k][..., e0:e1].movedim(-1, 0).double()                      # [T, (C,) n] -> [n, T, (C)]
        for k, kk in (("traj_no_t", "traj_no"), ("step_no_t", "step_no"), ("fallen", "fallen"), ("obs", "obs")):
            rep(kk, exact=True).add(got(k), dev(b[kk]), where, env0=env_id0 + e0)
        rep("reward").add(got("reward"), dev(b["reward"]), where, env0=env_id0 + e0)
        for k in ("xpos", "xquat", "site_xpos"):
            rep(k).add(got(k), dev(b[k]), where, env0=env_id0 + e0)
        _compare_cvel(rep, where, got("cvel"), dev(b["cvel"]), dev(b["xpos"]), env_id0 + e0)
    # the state the next call starts from (device: [C, n]; reset_count holds the bits of a uint32)
    d = dict(play_state, reset_count=play_state["reset_count"].long() & 0xFFFFFFFF)
    for k, kw in (("traj_no", dict(exact=True)), ("step_no", dict(exact=True)), ("reset_count", dict(exact=True)),
                  ("xy_off", dict(exact=True)), ("curr_qpos", dict(rtol=1e-12, atol=1e-12)),
                  ("pending", dict(exact=True)), ("prev_x_vel", dict(exact=True))):
        ref = torch.from_numpy(state[k].astype(np.float64)).cuda()
        if k == "pending":     # float32 on the device: x, y re-centred in float64 and rounded, the rest float32 numbers
            ref = ref.float().double()
        rep("state." + k, **kw).add(d[k].t().double(), ref, where, axes=("env", "ch")[:ref.dim()], env0=env_id0)
    return s1, s2


# cvel = [w; v] of each body about the subtree centre of mass.  The kernels form the centre of mass and every joint anchor
# in world coordinates in fp32 and take their differences from the root position (codegen.generate_fk), so once the root
# has walked |P| metres from the origin each difference carries about eps32 |P| of rounding per operation of the kinematic
# chain (16 bounds the roundings along the deepest H1 chain), and w x (com - P) and axis x (P - anchor) turn it into a
# linear-velocity error of that size times the angular velocities: 16 eps32 (|P| + 1) max_b |w_b| on top of the
# north-star bound.  In exact arithmetic cvel does not depend on P; the angular part carries no such term.
CVEL_LIN_ROUNDINGS = 16


def _compare_cvel(rep, where, got, ref, ref_xpos, env0):
    """cvel [env, step, 6 nbody]: the angular part at the north-star bound, the linear part with the term above."""
    import torch
    nb = ref.shape[-1] // 6
    g6, r6 = got.reshape(*got.shape[:-1], nb, 6), ref.reshape(*ref.shape[:-1], nb, 6)
    rep("cvel.angular").add(g6[..., :3].flatten(-2), r6[..., :3].flatten(-2), where, env0=env0)
    root = ref_xpos[..., 3:6].norm(dim=-1)                                              # body 1 (the root) position
    w_max = r6[..., :3].norm(dim=-1).amax(dim=-1)                                       # [env, step]
    extra = (CVEL_LIN_ROUNDINGS * float(np.finfo(np.float32).eps) * (root + 1.0) * w_max)[..., None]
    rep("cvel.linear", bound=f"max(1e-05, 1e-05 |ref|) + {CVEL_LIN_ROUNDINGS} eps32 (|root| + 1) max|w|").add(
        g6[..., 3:].flatten(-2), r6[..., 3:].flatten(-2), where, env0=env0, extra=extra)
    rep("cvel (north-star bound)", bound="max(1e-05, 1e-05 |ref|), reported only").add(got, ref, where, env0=env0)


def _device_state(env):
    tr, ps = env.trajectories.device_state, env._play_state
    return dict(traj_no=tr.traj_no, step_no=tr.step_no, reset_count=tr.reset_count, xy_off=tr.xy_off,
                curr_qpos=ps["curr_qpos"], pending=ps["pending"], prev_x_vel=ps["prev_x_vel"])


def _compare_moments(rep, where, mom, s1, s2, count):
    """Float64 moment sums the kernel accumulated against the oracle's observations (same bound as test_gpu_env.py)."""
    import torch
    ref = torch.as_tensor(np.concatenate([s1, s2, [count]]), device="cuda")
    rep("obs_moments", rtol=1e-12, atol=1e-9).add(mom, ref, where, axes=("ch",))


def test_bench_hot_step_matches_float64_oracle(bench_setup):
    """configs[1] exactly as bench.py's hot_step runs it (the world-1 all-reduce, a no-op, left out), three calls."""
    import torch
    import bench
    from olympics_mujoco_b200 import kernels as Kn
    from olympics_mujoco_b200.environments import LocoEnvBase
    from oracle import c_oracle
    model, table, tab, cm, perm = bench_setup
    n, T, seed = bench.N_ENVS, bench.HORIZON, 1234
    rep = Report("configs[1]")
    env = LocoEnvBase.make("UnitreeH1.walk.real", n_envs=n, traj_params=dict(table=table), seed=seed, env_id0=0)
    roll = env.make_rollout_buffers(T)
    g = torch.Generator(device="cuda").manual_seed(7)
    values = torch.randn((T + 1, n), device="cuda", generator=g)
    last = torch.zeros((T, n), dtype=torch.uint8, device="cuda")
    mom = torch.zeros(3 + 65, dtype=torch.float64, device="cuda")
    mom_adv, mom_obs = mom[:3], mom[3:]
    state = c_oracle.play_state(tab.shape[0], n)
    v64 = values.double().cpu().numpy().T                                               # [n, T + 1]
    last_np = np.zeros((n, T), np.uint8)
    for call in (1, 2, 3):
        where = f"call {call}"
        mom.zero_()
        out = env.play_trajectory_from_velocity(n_episodes=1, n_steps_per_episode=T, render=False, out=roll,
                                                obs_moments=mom_obs)
        vt, adv = Kn.gae(out["reward"], values[:-1], values[1:], out["fallen"], last, bench.GAMMA, bench.LAM)
        Kn.moments_scalar(adv, out=mom_adv)
        adv_raw = adv.clone()
        stats = Kn.adv_stats(mom_adv, unbiased=False, eps=1e-8)
        Kn.normalize(adv, stats, out=adv)
        torch.cuda.synchronize()
        # the oracle: the first call starts from a fresh env, every call begins with reset() (the Python API's on the
        # first call, the kernel's on the later ones) and ends with one
        s1, s2 = _play_and_compare(rep, where, bench_setup, seed, 0, state, True, out, _device_state(env), T)
        _compare_moments(rep, where, mom_obs, s1, s2, n * T)
        # GAE in float64 on the device's own rewards and flags: only the scan's error is measured
        r64 = out["reward"].double().cpu().numpy().T
        ab = out["fallen"].cpu().numpy().T
        ref_vt, ref_adv = c_oracle.gae(r64, v64[:, :-1], v64[:, 1:], ab, last_np, bench.GAMMA, bench.LAM)
        cu = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device="cuda")
        rep("v_target").add(vt.t().double(), cu(ref_vt), where, axes=("env", "step"))
        rep("adv").add(adv_raw.t().double(), cu(ref_adv), where, axes=("env", "step"))
        rep("adv_moments.count", exact=True).add(mom_adv[2:], cu([float(n * T)]), where, axes=("ch",))
        mean, std = ref_adv.mean(), ref_adv.std()                                        # population std (ddof 0)
        rep("adv_normalized").add(adv.t().double(), cu((ref_adv - mean) / (std + 1e-8)), where, axes=("env", "step"))
    rep.finish()


def test_sharded_1m_rollouts_match_float64_oracle(bench_setup):
    """One configs[4] shard as bench.sharded_1m runs it: two 64-step rollouts, each two 32-step calls into the same
    buffers (the second continues the episode), observation moments fused, then moment_stats(.., "ppo_obs").  The second
    rollout's first call resets inside the kernel at a nonzero env_id0."""
    import torch
    from olympics_mujoco_b200 import distributed as D
    from olympics_mujoco_b200 import kernels as Kn
    from olympics_mujoco_b200.environments import LocoEnvBase
    from oracle import c_oracle
    model, table, tab, cm, perm = bench_setup
    seed, t_call = 1234, 32
    env_id0, n = D.env_shard(1 << 20, 7, 8)
    assert (env_id0, n) == (917504, 131072)
    rep = Report("configs[4]")
    env = LocoEnvBase.make("UnitreeH1.walk.real", n_envs=n, traj_params=dict(table=table), seed=seed, env_id0=env_id0)
    roll = env.make_rollout_buffers(t_call)
    mom = torch.zeros(65, dtype=torch.float64, device="cuda")
    state = c_oracle.play_state(tab.shape[0], n)
    for rollout in (1, 2):
        mom.zero_()
        s1, s2 = np.zeros(32), np.zeros(32)
        for c in range(2):
            where = f"rollout {rollout} call {c + 1}"
            env.play_trajectory_from_velocity(n_episodes=1, n_steps_per_episode=t_call, render=False, out=roll,
                                              continue_episode=c > 0, obs_moments=mom)
            torch.cuda.synchronize()
            a1, a2 = _play_and_compare(rep, where, bench_setup, seed, env_id0, state, c == 0, roll, _device_state(env),
                                       t_call)
            s1 += a1
            s2 += a2
        where = f"rollout {rollout}"
        mean, denom = Kn.moment_stats(mom, "ppo_obs")
        torch.cuda.synchronize()
        cnt = n * 2 * t_call
        _compare_moments(rep, where, mom, s1, s2, cnt)
        ref_mean = s1 / cnt                                                              # MOMENT_KINDS["ppo_obs"]
        ref_denom = np.sqrt(np.maximum(s2 / cnt - ref_mean * ref_mean, 0.0) + 1e-8)
        cu = lambda a: torch.as_tensor(np.asarray(a, dtype=np.float64), device="cuda")
        rep("ppo_obs.mean").add(mean, cu(ref_mean), where, axes=("ch",))
        rep("ppo_obs.denominator").add(denom, cu(ref_denom), where, axes=("ch",))
    rep.finish()
