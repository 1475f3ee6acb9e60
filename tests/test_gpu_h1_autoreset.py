"""GPU: per-env reset (``UnitreeH1.reset(mask=...)``) and on-device auto-reset (``step(autoreset=True)``,
``om_h1_reset_envs``) against the oracle's masked reset and mushroom_rl Core loop (oracle/h1_autoreset.py).  Integers, flags,
qpos / qvel and observations bit for bit; rewards within assert_close."""
import numpy as np
import pytest

from conftest import GOLDEN, assert_close

pytestmark = pytest.mark.gpu

SEED = 2024
VARIANTS = dict(default={}, noback=dict(disable_back_joint=True), arms=dict(disable_arms=False),
                odd_weight=dict(hold_weight=True, weight_mass=2.5))


def _model(name="default"):
    from olympics_mujoco_b200 import mjcf
    return mjcf.unitree_h1_variant(**VARIANTS[name])


def _table(model):
    """The golden table restricted to the model's keys; with arms, a synthetic 3 x 50 table of all 50 keys."""
    from oracle import h1 as OH
    keys = OH.keys(model)
    if any(a in k for k in keys for a in OH.ARM_JOINTS):
        from olympics_mujoco_b200 import synthetic
        d = synthetic.h1_walk_dataset(n_traj=3, t_raw=50, seed=4, model=model)
        tab = np.stack([np.asarray(d[k]).reshape(3, 50) for k in keys])
    else:
        full = ["q_" + j for j in OH._SPEC_JOINTS] + ["dq_" + j for j in OH._SPEC_JOINTS]
        full = [k for k in full if not any(a in k for a in OH.ARM_JOINTS)]
        tab = np.load(GOLDEN / "trajectory_ref.npz")["table"].copy()[[full.index(k) for k in keys]]
    tab[2:] = tab[2:].astype(np.float32).astype(np.float64)
    return tab


def _env(n, name="default", seed=SEED, **kw):
    import olympics_mujoco_b200 as om
    args = dict(VARIANTS[name])
    args.update(kw)
    tab = _table(_model(name) if "weight_mass" in args or not args.get("hold_weight") else _model("odd_weight"))
    return om.LocoEnvBase.make("UnitreeH1.walk.real", n_envs=n, traj_params=dict(table=tab), seed=seed, **args), tab


def _f32(a):
    return np.asarray(a, dtype=np.float64).astype(np.float32)


def _snapshot(env):
    d, tr = env.data, env.trajectories.device_state
    s = dict(qpos=d.qpos, qvel=d.qvel, xpos=d.xpos, xquat=d.xquat, cvel=d.cvel, site_xpos=d.site_xpos, traj_no=tr.traj_no,
             step_no=tr.step_no, reset_count=tr.reset_count, xy_off=tr.xy_off, prev_x_vel=env._prev_x_vel,
             episode_step=env.episode_step)
    for k in ("model_index", "weight_body_mass", "partial_resets"):
        if hasattr(env, k):
            s[k] = getattr(env, k)
    if env._grf is not None:
        s["grf"] = env._grf
    return {k: v.detach().clone().cpu().numpy() for k, v in s.items()}


def _oracle_reset(env, model, tab, e, rc, grf_size=0):
    from oracle import h1_autoreset as OA
    from oracle.trajectory import TrajectoryState
    ts = TrajectoryState(tab, seed=env._seed, env_id=env._env_id0 + e)
    ts.reset_count = int(rc)
    return OA.reset_env(model, ts, env._random_start, env._init_step_no, grf_size)


def _check_masked_reset(env, model, tab, mask_np, obs_before):
    """One reset(mask=...) against the oracle; unmasked envs byte-identical, the FK mirrors untouched."""
    import torch
    before = _snapshot(env)
    mask = torch.tensor(mask_np, device="cuda")
    obs = env.reset(mask=mask)
    after = _snapshot(env)
    obs = obs.cpu().numpy()
    keep = ~mask_np.astype(bool)
    for k in before:
        if k in ("xpos", "xquat", "cvel", "site_xpos"):
            assert np.array_equal(before[k], after[k]), k
        else:
            assert np.array_equal(before[k][..., keep], after[k][..., keep]), k
    assert np.array_equal(obs[keep], obs_before[keep])
    grf_size = 0 if env._grf is None else env._grf.shape[0]
    for e in np.flatnonzero(mask_np):
        r = _oracle_reset(env, model, tab, e, before["reset_count"][e], grf_size)
        assert np.array_equal(after["qpos"][:, e], _f32(r["qpos"])), e
        assert np.array_equal(after["qvel"][:, e], _f32(r["qvel"])), e
        assert np.array_equal(obs[e], _f32(r["obs"])), e
        assert after["prev_x_vel"][e] == np.float32(r["prev_x_vel"])
        assert (after["traj_no"][e], after["step_no"][e], after["reset_count"][e]) == \
               (r["traj_no"], r["step_no"], r["reset_count"]), e
        assert np.array_equal(after["xy_off"][:, e], tab[:2, r["traj_no"], r["step_no"]])
        assert after["episode_step"][e] == 0
        if "grf" in after:
            assert not after["grf"][:, e].any()
    return obs


@pytest.mark.parametrize("start", ["random", "init_step", "neither"])
def test_masked_reset_against_oracle(start):
    """n = 300, ~30 % masked, after two full resets, fused live steps and an earlier masked reset (reset_count differs per env)."""
    kw = dict(random=dict(), init_step=dict(random_start=False, init_step_no=57), neither=dict(random_start=False))[start]
    n = 300
    env, tab = _env(n, **kw)
    model = env._model
    env.reset()
    env.reset()
    for _ in range(4):
        env.step_trajectory()
    rng = np.random.default_rng(1)
    obs = env._obs.cpu().numpy()
    for _ in range(3):
        mask = (rng.random(n) < 0.3).astype(np.uint8)
        obs = _check_masked_reset(env, model, tab, mask, obs)
    assert len(set(env.trajectories.device_state.reset_count.cpu().numpy().tolist())) > 1
    assert env._play_state is None


def test_all_ones_mask_equals_reset():
    import torch
    n = 64
    a, _ = _env(n)
    b, _ = _env(n)
    oa = a.reset(mask=torch.ones(n, dtype=torch.bool, device="cuda"))
    ob = b.reset()
    assert torch.equal(oa, ob)
    sa, sb = _snapshot(a), _snapshot(b)
    for k in ("qpos", "qvel", "traj_no", "step_no", "reset_count", "xy_off", "prev_x_vel", "episode_step"):
        assert np.array_equal(sa[k], sb[k]), k


def _scripted(model, tab, n, steps, seed=0, fall=0.1):
    """SoA post-physics states [steps, nq, n] / [steps, nv, n]: trajectory rows, ~``fall`` of them past has_fallen."""
    from oracle import h1 as OH
    rng = np.random.default_rng(seed)
    K, n_traj, T = tab.shape
    rows = tab[:, rng.integers(0, n_traj, (steps, n)), rng.integers(0, T, (steps, n))]        # [K, steps, n]
    rows = np.moveaxis(rows, 0, -1).copy()                                                     # [steps, n, K]
    falls = rng.random((steps, n)) < fall
    rows[..., 2] = np.where(falls, np.where(rng.random((steps, n)) < 0.5, -0.45, 0.25), rows[..., 2])   # q_pelvis_ty
    q, v = OH.set_sim_state(model, rows)
    q[..., [i for i in range(model.nq) if i not in OH.perm(model)]] = model.qpos0[[i for i in range(model.nq)
                                                                                  if i not in OH.perm(model)]]
    return _f32(q).astype(np.float64), _f32(v).astype(np.float64)


def _autoreset_rollout(env, model, tab, steps, horizon, seed=0, grf=False, twin=None):
    """step(autoreset=True) with SoA dynamics against core_rollout, every step, every env.  ``twin``: an identical env
    stepped on the default path with the same dynamics; its observation must equal final_obs bit for bit."""
    import torch
    from oracle import h1_autoreset as OA
    n = env.n_envs
    q, v = _scripted(model, tab, n, steps, seed)
    qt = torch.tensor(q, dtype=torch.float32, device="cuda").permute(0, 2, 1).contiguous()
    vt = torch.tensor(v, dtype=torch.float32, device="cuda").permute(0, 2, 1).contiguous()
    g = (np.random.default_rng(seed + 1).integers(-4000, 4000, (steps, n, 6)) * 125.0) if grf else None
    gt = None if g is None else torch.tensor(g, dtype=torch.float32, device="cuda")
    t_ = dict(t=0)

    def dyn(e, ctrl):
        t = t_["t"]
        return (qt[t], vt[t]) if gt is None else (qt[t], vt[t], gt[t])
    env.attach_dynamics(dyn, soa=True)
    if twin is not None:
        twin.attach_dynamics(dyn, soa=True)
        twin.reset()
    tr = env.trajectories.device_state
    rc0 = tr.reset_count.cpu().numpy().copy()
    env.reset()
    nu = env.info.action_space.shape[0]
    act = torch.zeros((nu, n), device="cuda")
    rec = {k: [] for k in ("obs", "final_obs", "reward", "absorbing", "last", "episode_step", "traj_no", "step_no",
                           "reset_count", "grf")}
    for t in range(steps):
        t_["t"] = t
        obs, reward, absorbing, info = env.step(act, autoreset=True)
        assert info["last"].dtype == torch.bool and info["final_obs"].shape == obs.shape
        for k, x in (("obs", obs), ("final_obs", info["final_obs"]), ("reward", reward), ("absorbing", absorbing),
                     ("last", info["last"]), ("episode_step", env.episode_step), ("traj_no", tr.traj_no),
                     ("step_no", tr.step_no), ("reset_count", tr.reset_count)):
            rec[k].append(x.detach().clone())
        if grf:
            rec["grf"].append(env._grf.clone())
        if twin is not None:
            assert torch.equal(twin.step(act)[0], info["final_obs"]), t
    got = {k: torch.stack(x).cpu().numpy() for k, x in rec.items() if x}
    assert got["last"].any() and not got["last"].all()
    for e in range(n):
        ref = OA.core_rollout(model, tab, list(zip(q[:, e], v[:, e])), horizon, seed=env._seed, env_id=env._env_id0 + e,
                              use_absorbing_states=env._use_absorbing_states, grfs=None if g is None else g[:, e],
                              reset_count0=rc0[e])
        nobs = 2 * len(OA.OH.perm(model)) - 2
        for k in ("obs", "final_obs"):
            assert np.array_equal(got[k][:, e, :nobs], _f32(ref[k][:, :nobs])), (k, e)
            # GRF / 1000: torch's float32 division by a scalar (the default step's op too) is not correctly rounded
            assert_close(got[k][:, e, nobs:], ref[k][:, nobs:], f"{k} GRF env {e}")
        for k in ("absorbing", "last", "episode_step", "traj_no", "step_no", "reset_count"):
            assert np.array_equal(got[k][:, e], ref[k]), (k, e)
        assert_close(got["reward"][:, e], ref["reward"], f"reward env {e}")
        if grf:
            for t in range(steps):                         # the GRF state of an env that reset is zero
                assert (not got["grf"][t][:, e].any()) if ref["last"][t] else np.array_equal(got["grf"][t][:, e],
                                                                                             _f32(g[t, e]))
    return got


@pytest.mark.parametrize("absorbing_states", [True, False])
def test_autoreset_rollout_against_core(absorbing_states):
    n = 257
    env, tab = _env(n, horizon=7, use_absorbing_states=absorbing_states)
    got = _autoreset_rollout(env, env._model, tab, 40, 7)
    assert got["absorbing"].any() == absorbing_states


def test_autoreset_foot_forces():
    env, tab = _env(96, horizon=5, use_foot_forces=True)
    twin, _ = _env(96, horizon=5, use_foot_forces=True)
    got = _autoreset_rollout(env, env._model, tab, 12, 5, seed=3, grf=True, twin=twin)
    assert got["obs"].shape[-1] == 32 + 6


@pytest.mark.parametrize("name", ["noback", "arms", "odd_weight"])
def test_variants(name):
    """Masked reset and auto-reset rollout of the variants and of a model without generated kernels."""
    env, tab = _env(70, name, horizon=4)
    model = env._model
    if name == "odd_weight":
        assert env._dm.h1_variant == 0
    env.reset()
    mask = (np.random.default_rng(5).random(70) < 0.4).astype(np.uint8)
    _check_masked_reset(env, model, tab, mask, env._obs.cpu().numpy())
    _autoreset_rollout(env, model, tab, 10, 4, seed=9)


@pytest.mark.parametrize("random", [True, False])
def test_per_env_weight_partial_draws(random):
    """Each env draws its own model at its own partial resets (stream 33 / round robin); a later full reset() keeps the
    object's k contract (stream 32); the carried weight's mass follows model_index."""
    import torch
    from olympics_mujoco_b200 import mjcf
    from olympics_mujoco_b200.utils.philox import env_model_draw, env_partial_model_draw
    n = 80
    env, tab = _env(n, "default", hold_weight=True, per_env_weight=True, random_env_reset=random, horizon=3)
    masses = np.float32([2.0 * w for w in mjcf.H1_VALID_WEIGHTS])
    env.reset()
    env.reset()
    rng = np.random.default_rng(2)
    for _ in range(3):
        before = _snapshot(env)
        mask = (rng.random(n) < 0.5).astype(np.uint8)
        env.reset(mask=torch.tensor(mask, device="cuda"))
        after = _snapshot(env)
        for e in range(n):
            if mask[e]:
                want = env_partial_model_draw(SEED, e, before["partial_resets"][e], 4, before["model_index"][e], random)
                assert after["model_index"][e] == want and after["partial_resets"][e] == before["partial_resets"][e] + 1
            else:
                assert after["model_index"][e] == before["model_index"][e]
        assert np.array_equal(after["weight_body_mass"], masses[after["model_index"]])
    assert env._model_resets == 2
    pr = env.partial_resets.clone()
    env.reset()
    idx = env.model_index.cpu().numpy()
    assert idx.tolist() == [env_model_draw(SEED, e, 2, 4, random) for e in range(n)]
    assert torch.equal(pr, env.partial_resets)
    # the auto-reset draws the same way, and the oracle still holds for the observations
    got = _autoreset_rollout(env, env._model, tab, 6, 3, seed=4)
    assert got["last"].any()
    assert np.array_equal(env.weight_body_mass.cpu().numpy(), masses[env.model_index.cpu().numpy()])


def test_shared_multimujoco_partial_reset_keeps_the_model():
    import torch
    env, tab = _env(40, "default", hold_weight=True, horizon=2)
    env.reset()
    env.reset()
    same = lambda s: s[:2] == (env._current_model_idx, env._model_resets) and all(
        a is b for a, b in zip(s[2:], (env._model, env._dm, env._data)))
    state = (env._current_model_idx, env._model_resets, env._model, env._dm, env._data)
    env.reset(mask=torch.ones(40, dtype=torch.uint8, device="cuda"))
    assert same(state)
    q = env.data.qpos.clone()

    def dyn(e, ctrl):
        return q, env.data.qvel.clone()
    env.attach_dynamics(dyn, soa=True)
    act = torch.zeros((env.info.action_space.shape[0], 40), device="cuda")
    for t in range(2):
        _, _, _, info = env.step(act, autoreset=True)
        assert bool(info["last"].all()) == (t == 1)        # horizon 2: the second step ends every episode
    assert same(state)


def _kernel_setup(n, seed=SEED, env_id0=0, ld=None):
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    from oracle import h1 as OH
    model = _model()
    tab = _table(model)
    ld = n if ld is None else ld
    dm, spec = Kn.DeviceModel(model), Kn.make_h1_spec([int(p) for p in OH.perm(model)], OH.x_vel_idx(model))
    traj = Kn.DeviceTrajectory(tab, ld, seed=seed, env_id0=env_id0)
    sample = traj.reset()
    st = dict(qpos=torch.zeros((17, ld), device="cuda"), qvel=torch.zeros((17, ld), device="cuda"),
              prev_x_vel=sample[17].clone(), episode_step=torch.zeros(ld, dtype=torch.int32, device="cuda"),
              obs=sample[2:].clone())
    Kn.set_sim_state(dm, spec, sample, st["qpos"], st["qvel"])
    return model, tab, dm, spec, traj, st


def test_graph_capture_equals_eager():
    """Kn.h1_step then Kn.h1_reset_envs (auto-reset) captured in one CUDA graph; 20 replays == 20 eager steps."""
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    n, steps, H = 300, 20, 5
    model, tab, *_ = _kernel_setup(n)
    q, v = _scripted(model, tab, n, steps, seed=11, fall=0.15)
    qs = torch.tensor(q, dtype=torch.float32, device="cuda").permute(0, 2, 1).contiguous()
    vs = torch.tensor(v, dtype=torch.float32, device="cuda").permute(0, 2, 1).contiguous()
    runs = []
    for mode in ("eager", "graph"):
        _, _, dm, spec, traj, st = _kernel_setup(n)
        o = dict(obs=torch.empty((32, n), device="cuda"), reward=torch.empty(n, device="cuda"),
                 absorbing=torch.empty(n, dtype=torch.uint8, device="cuda"))
        new, last = torch.empty((32, n), device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda")

        def step():
            Kn.h1_step(dm, spec, st["qpos"], st["qvel"], st["prev_x_vel"], want_fk=False, out=o)
            Kn.h1_reset_envs(dm, spec, traj, st["qpos"], st["qvel"], absorbing=o["absorbing"], horizon=H, obs_in=o["obs"],
                             obs=new, prev_x_vel=st["prev_x_vel"], episode_step=st["episode_step"], last=last)
        if mode == "graph":
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            g = torch.cuda.CUDAGraph()
            with torch.cuda.stream(side), torch.cuda.graph(g, stream=side):
                step()
            torch.cuda.current_stream().wait_stream(side)
            step = g.replay
        rec = []
        for t in range(steps):
            st["qpos"].copy_(qs[t])
            st["qvel"].copy_(vs[t])
            step()
            rec.append([x.clone() for x in (o["obs"], o["reward"], o["absorbing"], new, last, st["prev_x_vel"],
                                            st["episode_step"], traj.traj_no, traj.step_no, traj.reset_count, traj.xy_off,
                                            st["qpos"], st["qvel"])])
        torch.cuda.synchronize()
        runs.append(rec)
    assert any(bool(r[4].any()) for r in runs[0])
    for t in range(steps):
        for a, b in zip(runs[0][t], runs[1][t]):
            assert torch.equal(a, b), t


def test_padded_ld_and_shards():
    """ld > n through the C ABI leaves the padding alone and equals the unpadded call; two shards with env_id0 offsets
    equal the whole."""
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    n, ld = 257, 300
    rng = np.random.default_rng(8)
    mask = torch.tensor((rng.random(ld) < 0.3).astype(np.uint8), device="cuda")
    absorbing = torch.tensor((rng.random(ld) < 0.2).astype(np.uint8), device="cuda")
    es0 = torch.tensor(rng.integers(0, 6, ld).astype(np.int32), device="cuda")

    def run(n_, ld_, env_id0, lo):
        _, _, dm, spec, traj, st = _kernel_setup(ld_, env_id0=env_id0)
        sl = slice(lo, lo + ld_)
        st["episode_step"].copy_(es0[sl])
        new, last = torch.full((32, ld_), -7.0, device="cuda"), torch.full((ld_,), 9, dtype=torch.uint8, device="cuda")
        Kn.h1_reset_envs(dm, spec, traj, st["qpos"], st["qvel"], mask=mask[sl].contiguous(), obs_in=st["obs"], obs=new,
                         prev_x_vel=st["prev_x_vel"], episode_step=st["episode_step"], n=n_)
        mid = [x.clone() for x in (new, st["qpos"], st["qvel"], traj.reset_count, st["episode_step"])]
        Kn.h1_reset_envs(dm, spec, traj, st["qpos"], st["qvel"], absorbing=absorbing[sl].contiguous(), horizon=6,
                         obs_in=mid[0], obs=new, prev_x_vel=st["prev_x_vel"], episode_step=st["episode_step"], last=last,
                         n=n_)
        torch.cuda.synchronize()
        return [x for x in mid] + [x.clone() for x in (new, last, st["qpos"], st["qvel"], traj.traj_no, traj.step_no,
                                                       traj.reset_count, traj.xy_off, st["prev_x_vel"], st["episode_step"])]
    padded = run(n, ld, 0, 0)
    plain = run(n, n, 0, 0)
    for a, b in zip(padded, plain):
        assert torch.equal(a[..., :n], b), "padded"
    fresh = run(ld, ld, 0, 0)                                  # what the padding holds before any call: its reset state
    untouched = run(0, ld, 0, 0)
    for a, u in zip(padded, untouched):
        assert torch.equal(a[..., n:], u[..., n:]), "padding written"
    assert not torch.equal(fresh[3][n:], untouched[3][n:])
    s1, s2 = run(100, 100, 0, 0), run(157, 157, 100, 100)
    for whole, a, b in zip(plain, s1, s2):
        assert torch.equal(whole, torch.cat([a, b], dim=-1)), "shards"


def test_interleaved_live_step_and_masked_reset():
    """step_trajectory(), a masked reset, step_trajectory() again: the live step and the masked reset share the carried state
    (trajectory indices, prev_x_vel), and every observation / reward / index equals the oracle's."""
    import torch
    from oracle import h1 as OH
    from oracle import h1_autoreset as OA
    from oracle.trajectory import TrajectoryState
    n = 130
    env, tab = _env(n)
    model = env._model
    xv = OH.x_vel_idx(model)
    env.reset()
    mask = (np.random.default_rng(6).random(n) < 0.35).astype(np.uint8)
    seq = ["live"] * 3 + ["mask"] + ["live"] * 60          # 60 steps: every env wraps at least once (T = 50)
    got = []
    tr = env.trajectories.device_state
    for s in seq:
        if s == "mask":
            o = env.reset(mask=torch.tensor(mask, device="cuda"))
            r = None
        else:
            o, r, _, _ = env.step_trajectory()
            r = r.clone()
        got.append((o.clone().cpu().numpy(), None if r is None else r.cpu().numpy(), tr.traj_no.cpu().numpy().copy(),
                    tr.step_no.cpu().numpy().copy(), tr.reset_count.cpu().numpy().copy()))
    for e in range(n):
        ts = TrajectoryState(tab, seed=SEED, env_id=e)
        prev = OH.create_observation(ts.reset_trajectory())
        for s, (o, r, tn, sn, rc) in zip(seq, got):
            if s == "mask":
                if mask[e]:
                    cur = OA.reset_env(model, ts)["obs"]
                else:
                    cur = prev
            else:
                smp = ts.get_next_sample()
                if smp is None:
                    smp = ts.reset_trajectory()
                cur = OH.create_observation(smp)
                assert_close(r[e], np.exp(-np.square(prev[xv] - OH.TARGET_VELOCITY_WALK)), f"reward env {e}")
            assert np.array_equal(o[e], _f32(cur)), (s, e)
            assert (tn[e], sn[e], rc[e]) == (ts.traj_no, ts.step_no, ts.reset_count), (s, e)
            prev = cur
