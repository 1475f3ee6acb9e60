"""GPU: fused playback and live step of the UnitreeH1 constructor variants (no back joint, arms with / without the back
joint, a carried weight of each valid mass) against the oracle, the per-step kernels of the base class and the
three-kernel live-step chain."""
import numpy as np
import pytest

from conftest import GOLDEN, assert_close

pytestmark = pytest.mark.gpu

VARIANTS = dict(noback=dict(disable_back_joint=True), arms=dict(disable_arms=False),
                arms_noback=dict(disable_arms=False, disable_back_joint=True),
                carry_0p1=dict(hold_weight=True, weight_mass=0.1), carry_1=dict(hold_weight=True, weight_mass=1.0),
                carry_5=dict(hold_weight=True, weight_mass=5.0), carry_10=dict(hold_weight=True, weight_mass=10.0))


def _golden():
    tab = np.load(GOLDEN / "trajectory_ref.npz")["table"].copy()
    tab[2:] = tab[2:].astype(np.float32).astype(np.float64)
    return tab


def _model(name):
    from olympics_mujoco_b200 import mjcf
    return mjcf.unitree_h1_variant(**VARIANTS[name])


def _table(model):
    """The golden 3 x 50 table restricted to the model's keys; with arms, a synthetic 3 x 50 table of all 50 keys."""
    from oracle import h1 as OH
    keys = OH.keys(model)
    if any(a in k for k in keys for a in OH.ARM_JOINTS):
        from olympics_mujoco_b200 import synthetic
        d = synthetic.h1_walk_dataset(n_traj=3, t_raw=50, seed=4, model=model)
        tab = np.stack([np.asarray(d[k]).reshape(3, 50) for k in keys])
    else:
        full = ["q_" + j for j in OH._SPEC_JOINTS] + ["dq_" + j for j in OH._SPEC_JOINTS]
        full = [k for k in full if not any(a in k for a in OH.ARM_JOINTS)]
        tab = _golden()[[full.index(k) for k in keys]]
    tab[2:] = tab[2:].astype(np.float32).astype(np.float64)
    return tab


def _spec(model):
    from olympics_mujoco_b200 import kernels as Kn
    from oracle import h1 as OH
    return Kn.make_h1_spec([int(p) for p in OH.perm(model)], OH.x_vel_idx(model))


def _env(name, n, seed=77, **kw):
    import olympics_mujoco_b200 as om
    model = _model(name) if name else _model("carry_1")
    args = dict(VARIANTS[name]) if name else dict(hold_weight=True)
    return om.LocoEnvBase.make("UnitreeH1.walk.real", n_envs=n, traj_params=dict(table=_table(model)), seed=seed,
                               **args, **kw)


def test_variant_models_are_recognised():
    from olympics_mujoco_b200 import kernels as Kn, mjcf
    ids = {}
    for name in VARIANTS:
        dm = Kn.DeviceModel(_model(name))
        assert not dm.specialised, name
        ids[name] = dm.h1_variant
    assert len(set(ids.values())) == len(VARIANTS) and 0 not in ids.values() and 1 not in ids.values(), ids
    assert Kn.DeviceModel(mjcf.load_builtin("unitree_h1")).h1_variant == 1
    odd = mjcf.unitree_h1_variant(hold_weight=True, weight_mass=2.5)
    assert Kn.DeviceModel(odd).h1_variant == 0
    # an unlisted weight keeps the base-class playback and raises on the fused live step
    import olympics_mujoco_b200 as om
    import torch
    from olympics_mujoco_b200.environments.loco_env_base import LocoEnvBase as Base
    mk = lambda: om.LocoEnvBase.make("UnitreeH1.walk.real", n_envs=5, traj_params=dict(table=_table(odd)), seed=3,
                                     hold_weight=True, weight_mass=2.5)
    env, twin = mk(), mk()
    res = env.play_trajectory_from_velocity(1, 20, render=False)
    ref = Base.play_trajectory_from_velocity(twin, 1, 20)
    assert set(res) == {"obs", "has_fallen"} and torch.equal(res["obs"], ref["obs"])
    with pytest.raises(NotImplementedError):
        env.step_trajectory()


@pytest.mark.parametrize("forced", [False, True])
@pytest.mark.parametrize("n_episodes,n_steps", [(1, 120), (3, 37)])
@pytest.mark.parametrize("name", list(VARIANTS))
def test_variant_playback_kernel_parity(name, n_episodes, n_steps, forced, om_knob):
    """Kn.h1_play_from_velocity on the variant against oracle/h1.py, for the time-parallel kernel (chunks 1 and 7) and the
    sequential one: integer state, fallen and obs bit for bit; FK and reward to fp32 rounding; final carried state."""
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    from oracle import h1 as OH
    model = _model(name)
    tab = _table(model)
    nq, n, seed = model.nq, 24, 99
    refs = [(OH.play_trajectory if forced else OH.play_trajectory_from_velocity)(model, tab, n_episodes, n_steps, seed=seed,
                                                                                 env_id=e) for e in range(n)]
    dm, spec = Kn.DeviceModel(model), _spec(model)
    for chunk in (1, 7, 100000):
        om_knob("play_chunk", chunk)
        dt = Kn.DeviceTrajectory(tab, n, seed=seed)
        sample = dt.reset()
        state = dict(pending=sample.clone(), prev_x_vel=sample[nq].clone())
        if not forced:
            state["curr_qpos"] = sample[:nq].double().contiguous()
        outs = []
        for _ in range(n_episodes):
            o = Kn.h1_play_from_velocity(dm, spec, dt, state, n_steps, dt=0.01, end_episode_reset=True, forced=forced)
            torch.cuda.synchronize()
            outs.append({k: v.cpu().numpy() for k, v in o.items()})
        cat = {k: np.concatenate([o[k] for o in outs], axis=0) for k in outs[0]}
        nb = model.nbody
        for e, ref in enumerate(refs):
            msg = f"{name} chunk {chunk} env {e}"
            assert np.array_equal(cat["traj_no_t"][:, e], ref["traj_no"]), msg
            assert np.array_equal(cat["step_no_t"][:, e], ref["step_no"]), msg
            assert np.array_equal(cat["fallen"][:, e].astype(bool), ref["fallen"]), msg
            assert np.array_equal(cat["obs"][:, :, e], ref["obs"].astype(np.float32)), msg
            assert_close(cat["reward"][:, e], ref["reward"], "reward")
            assert_close(cat["xpos"][:, :, e], ref["xpos"].reshape(-1, nb * 3), "xpos")
            assert_close(cat["xquat"][:, :, e], ref["xquat"].reshape(-1, nb * 4), "xquat")
            assert_close(cat["site_xpos"][:, :, e], ref["site_xpos"].reshape(-1, 3 * model.nsite), "site_xpos")
            assert_close(cat["cvel"][:, :, e], ref["cvel"].reshape(-1, nb * 6), "cvel")
            fin = ref["final"]
            assert int(dt.traj_no[e]) == fin["traj_no"] and int(dt.step_no[e]) == fin["step_no"], msg
            assert int(dt.reset_count[e]) == fin["reset_count"], msg
            assert_close(state["pending"][:, e].cpu().numpy(), fin["pending_sample"], "pending", rtol=1e-6, atol=1e-6)
            if not forced:
                assert_close(state["curr_qpos"][:, e].cpu().numpy(), fin["curr_qpos"], "curr_qpos", rtol=1e-6, atol=1e-6)


def _env_state(env):
    tr = env.trajectories.device_state
    return [tr.traj_no.clone(), tr.step_no.clone(), tr.reset_count.clone(), tr.xy_off.clone(), env._obs.clone(),
            env._current_model_idx, env._model_resets]


def _same(a, b):
    import torch
    return all(torch.equal(x, y) if isinstance(x, torch.Tensor) else x == y for x, y in zip(a, b))


@pytest.mark.parametrize("case", list(VARIANTS) + ["multi_random", "multi_round_robin"])
def test_variant_playback_api_equals_base_class(case):
    """env.play_trajectory_from_velocity / play_trajectory (fused) return what the base class's per-step path returns on a
    twin env (last obs, has_fallen) and leave the same env state -- over two calls, so that the second call's reset runs
    inside the kernel; with MultiMuJoCo every reset() of the call moves the env to the same next model."""
    import torch
    from olympics_mujoco_b200.environments.loco_env_base import LocoEnvBase as Base
    n, T = 6, 45
    name = None if case.startswith("multi") else case
    kw = dict(random_env_reset=case == "multi_random") if name is None else {}
    for method in ("play_trajectory_from_velocity", "play_trajectory"):
        env, twin = _env(name, n, seed=21, **kw), _env(name, n, seed=21, **kw)
        if name is None:
            assert len(env._models) == 4 and all(dm.h1_variant for dm in env._dms)
        for call in range(2):
            res = getattr(env, method)(2, T, render=False)
            ref = getattr(Base, method)(twin, 2, T)
            assert set(res) == {"obs", "has_fallen"}, (case, method)
            assert torch.equal(res["obs"], ref["obs"]), (case, method, call)
            assert torch.equal(res["has_fallen"], ref["has_fallen"]), (case, method, call)
            assert _same(_env_state(env), _env_state(twin)), (case, method, call)


@pytest.mark.parametrize("name", ["arms", "carry_5"])
def test_variant_call_semantics(name):
    """Every call begins with a reset (two calls == the oracle called twice on one trajectory state);
    continue_episode=True == one two-episode call; obs_moments (2 nobs + 1 values) == float64 moments and accumulates."""
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    from oracle import h1 as OH
    n, T = 6, 70
    for steps in (T, 400):                                            # sequential, time-parallel kernel
        env = _env(name, n)
        model, tab = env._model, _table(env._model)
        want = ("obs", "traj_no_t", "step_no_t", "reward", "xpos")
        a = {k: v.clone() for k, v in env.play_trajectory_from_velocity(1, steps, render=False, want=want).items()}
        b = env.play_trajectory_from_velocity(1, steps, render=False, want=want)
        for e in range(n):
            r1 = OH.play_trajectory_from_velocity(model, tab, 1, steps, seed=77, env_id=e, record_fk=(e == 0))
            r2 = OH.play_trajectory_from_velocity(model, tab, 1, steps, seed=77, env_id=e, record_fk=(e == 0),
                                                  traj_state=r1["final"]["traj_state"])
            for out, ref in ((a, r1), (b, r2)):
                assert np.array_equal(out["traj_no_t"][:, e].cpu().numpy(), ref["traj_no"])
                assert np.array_equal(out["step_no_t"][:, e].cpu().numpy(), ref["step_no"])
                assert np.array_equal(out["obs"][:, :, e].cpu().numpy(), ref["obs"].astype(np.float32))
                assert_close(out["reward"][:, e].cpu().numpy(), ref["reward"], "reward")
                if e == 0:
                    assert_close(out["xpos"][:, :, e].cpu().numpy(), ref["xpos"].reshape(steps, -1), "xpos")
            assert int(env.trajectories.device_state.reset_count[e]) == r2["final"]["reset_count"]
    env1, env2 = _env(name, n), _env(name, n)
    want = ("obs", "traj_no_t", "step_no_t", "reward", "xpos")
    two = env1.play_trajectory_from_velocity(2, T, render=False, want=want)
    env2.play_trajectory_from_velocity(1, T, render=False, want=want)
    cont = env2.play_trajectory_from_velocity(1, T, render=False, want=want, continue_episode=True)
    for k in want:
        assert torch.equal(two[k], cont[k]), k
    nobs = 2 * env1._model.nq - 2
    for n, T in ((40, 33), (300, 260)):
        env = _env(name, n)
        mom = torch.zeros(2 * nobs + 1, dtype=torch.float64, device="cuda")
        out = env.play_trajectory_from_velocity(1, T, render=False, obs_moments=mom)
        torch.cuda.synchronize()
        o = out["obs"].double()
        exact = torch.cat([o.sum(dim=(0, 2)), (o * o).sum(dim=(0, 2)),
                           torch.tensor([float(n * T)], dtype=torch.float64, device="cuda")])
        assert float(mom[-1]) == n * T and (name != "arms" or mom.numel() == 97)
        assert_close(mom.cpu().numpy(), exact.cpu().numpy(), "fused moments", rtol=1e-12, atol=1e-9)
        assert_close(mom.cpu().numpy(), Kn.moments(out["obs"]).cpu().numpy(), "vs om_moments", rtol=1e-12, atol=1e-9)
        env.play_trajectory_from_velocity(1, T, render=False, obs_moments=mom)
        assert float(mom[-1]) == 2 * n * T
        with pytest.raises(ValueError):
            env.play_trajectory_from_velocity(1, T, render=False, obs_moments=torch.zeros(65 if nobs != 32 else 61,
                                                                                           dtype=torch.float64, device="cuda"))


@pytest.mark.parametrize("name", list(VARIANTS))
def test_variant_live_step(name):
    """step_trajectory (one kernel, generated FK) == om_traj_next -> om_set_sim_state -> om_h1_step (table-driven FK for a
    variant): ints, obs, absorbing and reward bit for bit, FK to fp32 rounding; against the oracle; step_graph replays ==
    eager steps."""
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    from oracle import h1 as OH
    from oracle.trajectory import TrajectoryState
    n, steps = 16, 110                                   # T = 50: every env wraps (and resets) at least twice
    env, env_b = _env(name, n), _env(name, n)
    env.reset()
    env_b.reset()
    model, tab = env._model, _table(env._model)
    nq, nb = model.nq, model.nbody
    trb = env_b.trajectories.device_state
    sample = Kn.soa(2 * nq, n)
    pxv = env_b._prev_x_vel.clone()
    oracle = []
    for e in range(3):
        ts = TrajectoryState(tab, seed=77, env_id=e)
        ts.reset_trajectory()
        oracle.append((ts, OH.create_observation(ts.get_current_sample())))
    for s in range(steps):
        obs, reward, absorbing, _ = env.step_trajectory()
        trb.next(sample=sample)
        Kn.set_sim_state(env_b._dm, env_b._spec, sample, env_b.data.qpos, env_b.data.qvel)
        ref = Kn.h1_step(env_b._dm, env_b._spec, env_b.data.qpos, env_b.data.qvel, pxv)
        assert torch.equal(obs, ref["obs"].t()) and torch.equal(reward, ref["reward"]), s
        assert torch.equal(absorbing, ref["absorbing"].bool())
        assert torch.equal(env.trajectories.device_state.step_no, trb.step_no)
        assert torch.equal(env.trajectories.device_state.traj_no, trb.traj_no)
        for k in ("qpos", "qvel"):
            assert torch.equal(getattr(env.data, k), getattr(env_b.data, k)), (k, s)
        for k in ("xpos", "xquat", "site_xpos", "cvel"):
            # generated FK (live step) against the table-driven FK (om_h1_step on a variant): fp32 rounding differs
            assert_close(getattr(env.data, k).cpu().numpy(), ref[k].cpu().numpy(), f"{k} step {s}")
        pxv = ref["obs"][nq - 2].clone()
        for e, (ts, prev) in enumerate(oracle):
            smp = ts.get_next_sample()
            if smp is None:
                smp = ts.reset_trajectory()
            q, v = OH.set_sim_state(model, smp.astype(np.float32).astype(np.float64))
            o = OH.step(model, q[None], v[None], prev[None])
            assert np.array_equal(obs[e].cpu().numpy(), o["obs"][0].astype(np.float32))
            assert_close(float(reward[e]), o["reward"][0], "reward")
            assert_close(env.data.xpos[:, e].cpu().numpy().reshape(nb, 3), o["xpos"][0], "xpos")
            assert_close(env.data.cvel[:, e].cpu().numpy().reshape(nb, 6), o["cvel"][0], "cvel")
            oracle[e] = (ts, o["obs"][0])
    env_g, env_e = _env(name, n), _env(name, n)
    env_g.reset(); env_e.reset()
    replay, bufs = env_g.step_graph(16, want=("obs", "reward", "absorbing", "xpos", "wrapped"))
    assert tuple(bufs["obs"].shape) == (16, 2 * nq - 2, n) and tuple(bufs["xpos"].shape) == (16, 3 * nb, n)
    for r in range(2):
        replay()
        torch.cuda.synchronize()
        for t in range(16):
            obs, reward, absorbing, _ = env_e.step_trajectory()
            assert torch.equal(bufs["obs"][t].t(), obs) and torch.equal(bufs["reward"][t], reward)
            assert torch.equal(bufs["xpos"][t], env_e.data.xpos)
    assert torch.equal(env_g.trajectories.device_state.step_no, env_e.trajectories.device_state.step_no)


def test_arms_playback_at_size(om_knob):
    """4096 envs x 500 steps with arms: the time-parallel kernel == the sequential one (ints and obs bit for bit, FK to
    fp32 rounding); 8 envs across the range against the oracle."""
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    from oracle import h1 as OH
    model = _model("arms")
    tab = _table(model)
    n, T, seed, nq = 4096, 500, 13, model.nq
    dm, spec = Kn.DeviceModel(model), _spec(model)
    res = []
    for chunk in (0, 100000):                                       # automatic (time-parallel), sequential
        om_knob("play_chunk", chunk)
        dt = Kn.DeviceTrajectory(tab, n, seed=seed)
        sample = dt.reset()
        state = dict(curr_qpos=sample[:nq].double().contiguous(), pending=sample.clone(), prev_x_vel=sample[nq].clone())
        res.append(Kn.h1_play_from_velocity(dm, spec, dt, state, T, dt=0.01, end_episode_reset=True))
        torch.cuda.synchronize()
    tp, seq = res
    for k in ("traj_no_t", "step_no_t", "fallen", "obs"):
        assert torch.equal(tp[k], seq[k]), k
    for k in ("xpos", "xquat", "site_xpos", "cvel", "reward"):
        assert_close(tp[k].cpu().numpy(), seq[k].cpu().numpy(), k, rtol=2e-5, atol=2e-5)
    nb = model.nbody
    for e in (0, 1, 700, 1365, 2048, 3001, 4094, 4095):
        ref = OH.play_trajectory_from_velocity(model, tab, 1, T, seed=seed, env_id=e)
        assert np.array_equal(tp["step_no_t"][:, e].cpu().numpy(), ref["step_no"])
        assert np.array_equal(tp["obs"][:, :, e].cpu().numpy(), ref["obs"].astype(np.float32))
        assert_close(tp["xpos"][:, :, e].cpu().numpy(), ref["xpos"].reshape(-1, nb * 3), "xpos")
        assert_close(tp["cvel"][:, :, e].cpu().numpy(), ref["cvel"].reshape(-1, nb * 6), "cvel")
