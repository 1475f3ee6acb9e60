"""GPU: the per-env carried weight of the UnitreeH1 carry task (``per_env_weight=True``): the draw contract of
``model_index`` / ``weight_body_mass``, and every path -- forward, step with dynamics, both fused playbacks, the live step
and its graph -- against the oracle run on the model each env holds."""
import numpy as np
import pytest

from conftest import GOLDEN, assert_close

pytestmark = pytest.mark.gpu

SEED = 77


def _table(model):
    from oracle import h1 as OH
    full = ["q_" + j for j in OH._SPEC_JOINTS] + ["dq_" + j for j in OH._SPEC_JOINTS]
    full = [k for k in full if not any(a in k for a in OH.ARM_JOINTS)]
    tab = np.load(GOLDEN / "trajectory_ref.npz")["table"].copy()[[full.index(k) for k in OH.keys(model)]]
    tab[2:] = tab[2:].astype(np.float32).astype(np.float64)
    return tab


def _env(n, per_env=True, random=True, env_id0=0, seed=SEED, **kw):
    import olympics_mujoco_b200 as om
    from olympics_mujoco_b200 import mjcf
    tab = _table(mjcf.unitree_h1_variant(hold_weight=True, weight_mass=1.0))
    return om.LocoEnvBase.make("UnitreeH1.carry.real", n_envs=n, traj_params=dict(table=tab), seed=seed,
                               per_env_weight=per_env, random_env_reset=random, env_id0=env_id0, **kw)


def _draw(e, k, random=True, env_id0=0):
    from olympics_mujoco_b200.utils.philox import env_model_draw
    return env_model_draw(SEED, env_id0 + e, k, 4, random)


def _masses():
    from olympics_mujoco_b200 import mjcf
    return np.float32([2.0 * w for w in mjcf.H1_VALID_WEIGHTS])


def _states(model, n, seed=3):
    """(qpos [n, nq], qvel [n, nv]) dataset-shaped, fp32-representable."""
    from olympics_mujoco_b200 import synthetic
    from oracle import h1 as OH
    d = synthetic.h1_walk_dataset(n_traj=2, t_raw=600, seed=seed, model=model)
    sample = np.stack([d[k] for k in OH.keys(model)], axis=1)[::5][:n]
    q, v = OH.set_sim_state(model, sample)
    f = lambda a: a.astype(np.float32).astype(np.float64)
    return f(q), f(v)


@pytest.mark.parametrize("random", [True, False])
def test_reset_draws_follow_the_contract(random):
    """After each reset(): model_index / weight_body_mass == the contract; env 0 == a shared twin's _current_model_idx; two
    shards reproduce the batch; every weight is present; one data / device model serve all envs; n_envs=None == shared."""
    import torch
    n = 64
    env, twin = _env(n, random=random), _env(n, per_env=False, random=random)
    a, b = _env(24, random=random), _env(40, random=random, env_id0=24)
    assert len({id(x) for x in env._dms}) == 1 and len({id(x) for x in env._datas}) == 1
    assert env.model_index.dtype == torch.int32 and env.weight_body_mass.dtype == torch.float32
    assert torch.equal(env.model_index.cpu(), torch.zeros(n, dtype=torch.int32))
    data, dm = env._data, env._dm
    for k in range(6):
        for x in (env, twin, a, b):
            x.reset()
        idx = env.model_index.cpu().numpy()
        assert idx.tolist() == [_draw(e, k, random) for e in range(n)], k
        assert np.array_equal(env.weight_body_mass.cpu().numpy(), _masses()[idx])
        assert idx[0] == twin._current_model_idx == env._current_model_idx
        assert torch.equal(torch.cat([a.model_index, b.model_index]), env.model_index)
        assert torch.equal(torch.cat([a.weight_body_mass, b.weight_body_mass]), env.weight_body_mass)
        assert set(idx.tolist()) == {0, 1, 2, 3}
        assert env._data is data and env._dm is dm
    one, shared = _env(None, random=random), _env(None, per_env=False, random=random)
    for k in range(6):
        o1, o2 = one.reset(), shared.reset()
        assert int(one.model_index[0]) == shared._current_model_idx
        assert torch.equal(o1, o2)


def test_forward_uses_each_envs_mass():
    """forward(): subtree_com and cvel per env == the oracle on that env's own model; xpos, xquat, site_xpos == shared mode."""
    from oracle import kinematics as K
    n = 40
    env, twin = _env(n), _env(n, per_env=False)
    env.reset(); env.reset(); twin.reset(); twin.reset()
    q, v = _states(env._model, n)
    env.set_state(q, v)
    twin.set_state(q, v)
    idx = env.model_index.cpu().numpy()
    assert len(set(idx.tolist())) > 1
    d, t = env.data, twin.data
    for k in ("xpos", "xquat", "site_xpos"):
        assert_close(getattr(d, k).cpu().numpy(), getattr(t, k).cpu().numpy(), k)
    nb = env._model.nbody
    for e in range(n):
        ref = K.forward(env._models[idx[e]], q[e:e + 1], v[e:e + 1])
        assert_close(d.subtree_com[:, e].cpu().numpy(), ref["subtree_com"][0, 1], f"subtree_com env {e}")
        assert_close(d.cvel[:, e].cpu().numpy().reshape(nb, 6), ref["cvel"][0], f"cvel env {e}")
        assert_close(d.xpos[:, e].cpu().numpy().reshape(nb, 3), ref["xpos"][0], f"xpos env {e}")


@pytest.mark.parametrize("soa", [False, True])
def test_step_with_dynamics(soa):
    """step() with attached dynamics: obs, absorbing and reward bit for bit == shared mode (they do not depend on the
    mass), obs == the oracle's; FK per env within tolerance of the oracle on that env's model."""
    import torch
    from oracle import h1 as OH
    n, steps = 24, 3
    env, twin = _env(n), _env(n, per_env=False)
    q, v = _states(env._model, n * steps, seed=6)
    qt, vt = torch.tensor(q, dtype=torch.float32, device="cuda"), torch.tensor(v, dtype=torch.float32, device="cuda")
    state = dict(s=0)

    def dyn(e, ctrl):
        s = state["s"]
        qq, vv = qt[s * n:(s + 1) * n], vt[s * n:(s + 1) * n]
        return (qq.t().contiguous(), vv.t().contiguous()) if soa else (qq, vv)
    for x in (env, twin):
        x.attach_dynamics(dyn, soa=soa)
        x.reset()
    nu = env.info.action_space.shape[0]
    act = torch.zeros((nu, n) if soa else (n, nu), device="cuda")
    idx = env.model_index.cpu().numpy()
    nb = env._model.nbody
    prev = env._obs.cpu().numpy().astype(np.float64)
    for s in range(steps):
        state["s"] = s
        o1, r1, a1, _ = env.step(act)
        o2, r2, a2, _ = twin.step(act)
        assert torch.equal(o1, o2) and torch.equal(r1, r2) and torch.equal(a1, a2), s
        for e in range(n):
            qq, vv = q[s * n + e][None], v[s * n + e][None]
            ref = OH.step(env._models[idx[e]], qq, vv, prev[e][None])
            assert np.array_equal(o1[e].cpu().numpy(), ref["obs"][0].astype(np.float32))
            assert bool(a1[e]) == bool(ref["absorbing"][0])
            assert_close(float(r1[e]), ref["reward"][0], "reward")
            assert_close(env.data.cvel[:, e].cpu().numpy().reshape(nb, 6), ref["cvel"][0], f"cvel env {e}")
            assert_close(env.data.xpos[:, e].cpu().numpy().reshape(nb, 3), ref["xpos"][0], f"xpos env {e}")
        prev = o1.cpu().numpy().astype(np.float64)


def _check_episode(out, e, ref, lo, model, tag):
    """One returned episode (buffers [T, C, n]) of env e against oracle records [lo, lo + T) on ``model``'s FK."""
    from oracle import kinematics as K
    T = out["obs"].shape[0]
    sl = slice(lo, lo + T)
    nb = model.nbody
    assert np.array_equal(out["traj_no_t"][:, e].cpu().numpy(), ref["traj_no"][sl]), tag
    assert np.array_equal(out["step_no_t"][:, e].cpu().numpy(), ref["step_no"][sl]), tag
    assert np.array_equal(out["fallen"][:, e].cpu().numpy().astype(bool), ref["fallen"][sl]), tag
    assert np.array_equal(out["obs"][:, :, e].cpu().numpy(), ref["obs"][sl].astype(np.float32)), tag
    assert_close(out["reward"][:, e].cpu().numpy(), ref["reward"][sl], f"reward {tag}")
    fk = K.forward(model, ref["qpos"][sl], ref["qvel"][sl])
    for k, c in (("xpos", 3), ("xquat", 4), ("cvel", 6)):
        assert_close(out[k][:, :, e].cpu().numpy(), fk[k].reshape(T, nb * c), f"{k} {tag}")
    assert_close(out["site_xpos"][:, :, e].cpu().numpy(), fk["site_xpos"].reshape(T, -1), f"site_xpos {tag}")


WANT = ("xpos", "xquat", "site_xpos", "cvel", "obs", "reward", "fallen", "traj_no_t", "step_no_t")


@pytest.mark.parametrize("chunk", [1, 7, 100000])
def test_play_from_velocity_per_env(chunk, om_knob):
    """Two calls of 2 episodes, then a continue_episode call of 1: every returned episode per env == the oracle (ints, obs,
    fallen bit for bit, reward and FK to fp32 rounding) on the model the env held in that episode; obs_moments ==
    om_moments of the obs; model_index after each call == the contract at the final counter."""
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    from oracle import h1 as OH
    om_knob("play_chunk", chunk)
    n, T = 12, 37
    env = _env(n)
    tab = _table(env._model)
    nobs = 2 * env._model.nq - 2
    # oracle per env: call 1 (2 episodes), call 2 (2 episodes) + the continue call (= a third episode of call 2);
    # draws: call 1 episodes k = 0, 1 (reset k = 2 ends it); call 2 k = 3, 4, continue call k = 5; k = 6 ends it
    refs = []
    for e in range(n):
        r1 = OH.play_trajectory_from_velocity(env._model, tab, 2, T, seed=SEED, env_id=e, record_fk=False)
        r2 = OH.play_trajectory_from_velocity(env._model, tab, 3, T, seed=SEED, env_id=e, record_fk=False,
                                              traj_state=r1["final"]["traj_state"])
        refs.append((r1, r2))
    calls = [(2, False, 0, 1, 3), (2, False, 1, 4, 6), (1, True, 1, 5, 7)]   # (episodes, continue, ref, k of the returned
    for c, (eps, cont, ri, k, resets) in enumerate(calls):                 # episode, resets after the call)
        mom = torch.zeros(2 * nobs + 1, dtype=torch.float64, device="cuda") if eps == 1 else None
        out = env.play_trajectory_from_velocity(eps, T, render=False, want=WANT, continue_episode=cont, obs_moments=mom)
        torch.cuda.synchronize()
        assert env._model_resets == resets
        idx = env.model_index.cpu().numpy()
        assert idx.tolist() == [_draw(e, resets - 1) for e in range(n)], c
        assert np.array_equal(env.weight_body_mass.cpu().numpy(), _masses()[idx])
        lo = (eps - 1) * T if ri == 0 else (T if c == 1 else 2 * T)
        for e in range(n):
            _check_episode(out, e, refs[e][ri], lo, env._models[_draw(e, k)], f"chunk {chunk} call {c} env {e}")
        if mom is not None:
            assert_close(mom.cpu().numpy(), Kn.moments(out["obs"]).cpu().numpy(), "obs_moments", rtol=1e-12, atol=1e-9)


@pytest.mark.parametrize("chunk", [1, 7, 100000])
def test_play_trajectory_per_env(chunk, om_knob):
    """play_trajectory (forced), one call of 2 episodes: the returned episode per env == the oracle on the model the env
    held; the model_index after the call == the contract."""
    import torch
    from oracle import h1 as OH
    om_knob("play_chunk", chunk)
    n, T = 12, 37
    env = _env(n)
    tab = _table(env._model)
    out = env.play_trajectory(2, T, render=False, want=WANT)
    torch.cuda.synchronize()
    assert env.model_index.cpu().numpy().tolist() == [_draw(e, 2) for e in range(n)]
    for e in range(n):
        ref = OH.play_trajectory(env._model, tab, 2, T, seed=SEED, env_id=e, record_fk=False)
        _check_episode(out, e, ref, T, env._models[_draw(e, 1)], f"chunk {chunk} env {e}")


@pytest.mark.parametrize("random", [True, False])
def test_playback_summary_equals_base_class(random):
    """Without out / want / obs_moments both playbacks return what LocoEnvBase.play_* returns on a per-env twin (its per-step
    path reaches the per-env mass through om_fk) and leave the same env state, over two calls."""
    import torch
    from olympics_mujoco_b200.environments.loco_env_base import LocoEnvBase as Base
    n, T = 6, 45
    for method in ("play_trajectory_from_velocity", "play_trajectory"):
        env, twin = _env(n, random=random, seed=21), _env(n, random=random, seed=21)
        for call in range(2):
            res = getattr(env, method)(2, T, render=False)
            ref = getattr(Base, method)(twin, 2, T)
            assert set(res) == {"obs", "has_fallen"}
            assert torch.equal(res["obs"], ref["obs"]) and torch.equal(res["has_fallen"], ref["has_fallen"]), (method, call)
            tr, tt = env.trajectories.device_state, twin.trajectories.device_state
            for x, y in ((tr.traj_no, tt.traj_no), (tr.step_no, tt.step_no), (tr.reset_count, tt.reset_count),
                         (tr.xy_off, tt.xy_off), (env._obs, twin._obs), (env.model_index, twin.model_index),
                         (env.weight_body_mass, twin.weight_body_mass)):
                assert torch.equal(x, y), (method, call)
            assert env._model_resets == twin._model_resets and env._current_model_idx == twin._current_model_idx


def test_live_step_and_graph_per_env():
    """step_trajectory == om_traj_next -> om_set_sim_state -> om_h1_step on a per-env twin (ints, obs, absorbing, reward bit
    for bit; FK to fp32 rounding) and == the oracle on each env's model; wraps keep model_index; step_graph == eager."""
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    from oracle import h1 as OH
    from oracle.trajectory import TrajectoryState
    n, steps = 16, 110                                       # T = 50: every env wraps (and resets its trajectory) twice
    env, env_b = _env(n), _env(n)
    env.reset(); env.reset(); env_b.reset(); env_b.reset()
    idx0 = env.model_index.clone()
    assert torch.equal(idx0, env_b.model_index)
    model, tab = env._model, _table(env._model)
    nq, nb = model.nq, model.nbody
    trb = env_b.trajectories.device_state
    sample = Kn.soa(2 * nq, n)
    pxv = env_b._prev_x_vel.clone()
    idx = idx0.cpu().numpy()
    oracle = []
    for e in range(3):
        ts = TrajectoryState(tab, seed=SEED, env_id=e)
        ts.reset_trajectory(); ts.reset_trajectory()
        oracle.append((ts, OH.create_observation(ts.get_current_sample())))
    for s in range(steps):
        obs, reward, absorbing, _ = env.step_trajectory()
        trb.next(sample=sample)
        Kn.set_sim_state(env_b._dm, env_b._spec, sample, env_b.data.qpos, env_b.data.qvel)
        ref = Kn.h1_step(env_b._dm, env_b._spec, env_b.data.qpos, env_b.data.qvel, pxv)
        assert torch.equal(obs, ref["obs"].t()) and torch.equal(reward, ref["reward"]), s
        assert torch.equal(absorbing, ref["absorbing"].bool())
        assert torch.equal(env.trajectories.device_state.step_no, trb.step_no)
        for k in ("xpos", "xquat", "site_xpos", "cvel"):
            assert_close(getattr(env.data, k).cpu().numpy(), ref[k].cpu().numpy(), f"{k} step {s}")
        pxv = ref["obs"][nq - 2].clone()
        for e, (ts, prev) in enumerate(oracle):
            smp = ts.get_next_sample()
            if smp is None:
                smp = ts.reset_trajectory()
            q, v = OH.set_sim_state(model, smp.astype(np.float32).astype(np.float64))
            o = OH.step(env._models[idx[e]], q[None], v[None], prev[None])
            assert np.array_equal(obs[e].cpu().numpy(), o["obs"][0].astype(np.float32))
            assert_close(env.data.cvel[:, e].cpu().numpy().reshape(nb, 6), o["cvel"][0], "cvel")
            assert_close(env.data.xpos[:, e].cpu().numpy().reshape(nb, 3), o["xpos"][0], "xpos")
            oracle[e] = (ts, o["obs"][0])
    assert int(env.trajectories.device_state.reset_count.min()) >= 4          # wraps happened ...
    assert torch.equal(env.model_index, idx0) and env._model_resets == 2       # ... and kept the weights
    env_g, env_e = _env(n), _env(n)
    env_g.reset(); env_e.reset()
    replay, bufs = env_g.step_graph(16, want=("obs", "reward", "absorbing", "xpos", "cvel"))
    for r in range(2):
        replay()
        torch.cuda.synchronize()
        for t in range(16):
            obs, reward, absorbing, _ = env_e.step_trajectory()
            assert torch.equal(bufs["obs"][t].t(), obs) and torch.equal(bufs["reward"][t], reward)
            assert torch.equal(bufs["xpos"][t], env_e.data.xpos) and torch.equal(bufs["cvel"][t], env_e.data.cvel)
    assert torch.equal(env_g.model_index, env_e.model_index)


def test_per_env_playback_at_size(om_knob):
    """4096 envs x 500 steps: the time-parallel kernel == the sequential one (ints and obs bit for bit, FK to fp32
    rounding); 8 envs across the batch against the oracle on their own models."""
    import torch
    from oracle import h1 as OH
    n, T = 4096, 500
    res = []
    for chunk in (0, 100000):
        om_knob("play_chunk", chunk)
        env = _env(n, seed=13)
        res.append({k: v.clone() for k, v in env.play_trajectory_from_velocity(1, T, render=False, want=WANT).items()})
        torch.cuda.synchronize()
    tp, seq = res
    for k in ("traj_no_t", "step_no_t", "fallen", "obs"):
        assert torch.equal(tp[k], seq[k]), k
    for k in ("xpos", "xquat", "site_xpos", "cvel", "reward"):
        assert_close(tp[k].cpu().numpy(), seq[k].cpu().numpy(), k, rtol=2e-5, atol=2e-5)
    from olympics_mujoco_b200.utils.philox import env_model_draw
    tab = _table(env._model)
    for e in (0, 1, 700, 1365, 2048, 3001, 4094, 4095):
        ref = OH.play_trajectory_from_velocity(env._model, tab, 1, T, seed=13, env_id=e, record_fk=False)
        _check_episode(tp, e, ref, 0, env._models[env_model_draw(13, e, 0, 4, True)], f"env {e}")


def test_errors():
    """Bad constructor combinations raise ValueError; binding a non-carry model, or another body, fails through
    om_last_error."""
    import torch
    import olympics_mujoco_b200 as om
    from olympics_mujoco_b200 import _lib, mjcf
    from olympics_mujoco_b200 import kernels as Kn
    with pytest.raises(ValueError):
        om.LocoEnvBase.make("UnitreeH1.walk.real", n_envs=4, per_env_weight=True)
    with pytest.raises(ValueError):
        om.LocoEnvBase.make("UnitreeH1.carry.real", n_envs=4, weight_mass=5.0, per_env_weight=True)
    mass = torch.zeros(8, device="cuda")
    for model in (mjcf.load_builtin("unitree_h1"), mjcf.unitree_h1_variant(disable_arms=False),
                  mjcf.unitree_h1_variant(hold_weight=True, weight_mass=2.5)):
        with pytest.raises(_lib.OmError, match="only the UnitreeH1 carry models"):
            Kn.bind_env_body_mass(Kn.DeviceModel(model), 21, mass)
    carry = mjcf.unitree_h1_variant(hold_weight=True, weight_mass=1.0)
    dm = Kn.DeviceModel(carry)
    with pytest.raises(_lib.OmError, match="not the weight body"):
        Kn.bind_env_body_mass(dm, 3, mass)
    Kn.bind_env_body_mass(dm, carry.body_id("weight"), mass)
    with pytest.raises(_lib.OmError, match="already bound"):
        Kn.bind_env_body_mass(dm, carry.body_id("weight"), torch.zeros(8, device="cuda"))
    with pytest.raises(_lib.OmError, match="bound body mass holds"):
        Kn.fk(dm, torch.zeros((carry.nq, 16), device="cuda"), torch.zeros((carry.nv, 16), device="cuda"))
