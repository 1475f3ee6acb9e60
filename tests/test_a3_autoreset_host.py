"""CPU: the auto-reset of the batched StickFigureA3 step -- the oracle's PPO sampler loop on scripted physics (path-end
codes, resets, traj_len, per-path returns), the argument checks of ``step(autoreset=True)`` / ``A3Task.autoreset`` and the
loud failure of the new entry point without a GPU."""
import numpy as np
import pytest

SEED, ENV = 4, 3


@pytest.fixture(scope="module")
def model():
    from olympics_mujoco_b200 import mjcf
    return mjcf.load_builtin("stick_figure_a3")


@pytest.fixture(scope="module")
def lut():
    from olympics_mujoco_b200.tasks.phase_clock import phase_clock_lut
    return phase_clock_lut()


def _script(n_steps, bad_at=(), seed=0):
    """Scripted post-physics states: the env's first reset pose with small noise; bad collision (done) at ``bad_at``."""
    from oracle import a3 as OA
    rng = np.random.default_rng(seed)
    from olympics_mujoco_b200 import mjcf
    q0, v0, _, _ = OA.reset(mjcf.load_builtin("stick_figure_a3"), SEED, ENV, 0)
    out = []
    for t in range(n_steps):
        q = q0 + rng.normal(0, 0.005, q0.shape)
        v = v0 + rng.normal(0, 0.05, v0.shape)
        con = OA.Contact(l_grf=float(rng.uniform(0, 300)), r_grf=float(rng.uniform(0, 300)), min_z=0.0, foot_contact=True,
                         bad_collision=t in bad_at)
        out.append((q, v, con))
    return out


def _run(model, lut, n_steps, bad_at, max_traj_len, **kw):
    from oracle import a3_autoreset as OR
    return OR.sample(model, _script(n_steps, bad_at), lut, max_traj_len=max_traj_len, seed=SEED, env_id=ENV, **kw)


def test_sampler_path_end_codes_and_resets(model, lut):
    # done at step 1; truncation at step 5 (4 steps into the second path); done and truncation together at step 9
    r = _run(model, lut, 12, bad_at=(1, 9), max_traj_len=4)
    assert r["path_end"].tolist() == [0, 1, 0, 0, 0, 2, 0, 0, 0, 1, 0, 0]
    assert r["done"].tolist() == [t in (1, 9) for t in range(12)]
    assert r["trunc"][9] and r["done"][9]                                # done wins: bootstrap 0, as (not done) * V
    assert r["last"].tolist() == [t in (1, 5, 9) for t in range(12)]
    assert r["traj_len"].tolist() == [1, 0, 1, 2, 3, 0, 1, 2, 3, 0, 1, 2]
    assert r["reset_count"].tolist() == [1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4]
    from oracle import a3 as OA
    from oracle import a3_autoreset as OR
    for t in range(12):
        if r["last"][t]:                                                  # the new path starts from reset number rc - 1
            _, _, ts, obs = OA.reset(model, SEED, ENV, int(r["reset_count"][t]) - 1)
            assert np.array_equal(r["next_obs"][t], obs) and r["ints"][t].tolist() == OR.ints_of(ts)
            assert np.array_equal(r["sequence"][t], np.asarray(ts.sequence))
            assert not np.array_equal(r["next_obs"][t], r["final_obs"][t])
        else:
            assert np.array_equal(r["next_obs"][t], r["final_obs"][t])
        if t + 1 < 12:
            assert np.array_equal(r["obs"][t + 1], r["next_obs"][t])
    assert np.array_equal(r["obs"][0], r["initial"][3])
    assert OR.paths(r) == [(0, 2), (2, 6), (6, 10), (10, 12)]


def test_sampler_without_max_traj_len(model, lut):
    r = _run(model, lut, 9, bad_at=(6,), max_traj_len=None)
    assert r["path_end"].tolist() == [0, 0, 0, 0, 0, 0, 1, 0, 0]
    assert r["traj_len"].tolist() == [1, 2, 3, 4, 5, 6, 0, 1, 2]
    assert not r["trunc"].any()
    r1 = _run(model, lut, 3, bad_at=(), max_traj_len=1)                   # every step ends a path
    assert r1["path_end"].tolist() == [2, 2, 2] and r1["traj_len"].tolist() == [0, 0, 0]
    assert r1["reset_count"].tolist() == [2, 3, 4]
    r5 = _run(model, lut, 2, bad_at=(0,), max_traj_len=None, reset_count0=5)
    assert r5["reset_count"].tolist() == [7, 7]


def test_path_returns_equal_finish_path_and_the_buffer_form(model, lut):
    """Per path, PPOBuffer.finish_path (oracle.learner.ppo_returns with (not done) * V(state)); the same numbers from ONE
    backward pass over the buffer with the path_end codes, v_next = V(final_obs) and last_val = V(obs_T) -- what
    om_ppo_returns computes on the device."""
    from oracle import a3_autoreset as OR
    from oracle import learner as L
    r = _run(model, lut, 12, bad_at=(1, 9), max_traj_len=4)
    w = np.random.default_rng(3).normal(0, 0.1, 41)
    critic = lambda o: float(w @ o) + 0.5
    gamma = 0.9
    ret, adv = OR.path_returns(r, critic, gamma)
    for a, b in OR.paths(r):                                             # finish_path, path by path
        vals = np.array([critic(o) for o in r["obs"][a:b]])
        boot = 0.0 if r["done"][b - 1] else critic(r["final_obs"][b - 1])
        want, want_adv = L.ppo_returns(r["reward"][a:b, None], vals[:, None], False, boot, gamma)
        np.testing.assert_allclose(ret[a:b], want[:, 0], rtol=1e-12)
        np.testing.assert_allclose(adv[a:b], want_adv[:, 0], rtol=1e-12, atol=1e-12)
    v_next = np.array([critic(o) for o in r["final_obs"]])
    v_last = critic(r["next_obs"][-1])                                    # obs_T: the state after the buffer's last step
    R, buf = 0.0, np.empty(12)
    for t in range(11, -1, -1):
        pe = r["path_end"][t]
        if pe == 1:
            R = 0.0
        elif pe == 2:
            R = v_next[t]
        elif t == 11:
            R = v_last
        R = gamma * R + r["reward"][t]
        buf[t] = R
    np.testing.assert_allclose(buf, ret, rtol=1e-12)
    assert ret[1] == r["reward"][1] and ret[5] == pytest.approx(r["reward"][5] + gamma * critic(r["final_obs"][5]))


def test_autoreset_argument_checks():
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    from olympics_mujoco_b200.environments.stick_figure_a3 import StickFigureA3
    env = object.__new__(StickFigureA3)                # the checks come before any device work
    env._dynamics = None
    for bad in (0, -1):
        with pytest.raises(ValueError, match="max_traj_len"):
            env.step(np.zeros((4, 12)), autoreset=True, max_traj_len=bad)
    with pytest.raises(RuntimeError, match="attach_dynamics"):
        env.step(np.zeros((4, 12)), autoreset=True, max_traj_len=5)
    task = object.__new__(Kn.A3Task)
    task.n = 4
    f = lambda *s: torch.zeros(s)
    ok = dict(qpos=f(25, 4), qvel=f(24, 4), done=torch.zeros(4, dtype=torch.uint8), traj_len=torch.zeros(4, dtype=torch.int32),
              obs_in=f(41, 4), obs=f(41, 4), last=torch.zeros(4, dtype=torch.bool), path_end=torch.zeros(4, dtype=torch.uint8))
    for name, bad in (("qpos", f(24, 4)), ("qvel", f(24, 5)), ("obs_in", f(41, 4).double()), ("obs", f(4, 41)),
                      ("done", torch.zeros(4, dtype=torch.int32)), ("traj_len", torch.zeros(4, dtype=torch.int64)),
                      ("last", torch.zeros(3, dtype=torch.uint8)), ("path_end", torch.zeros(4, dtype=torch.bool))):
        with pytest.raises(ValueError, match=name):
            task.autoreset(**{**ok, name: bad})
    with pytest.raises(ValueError, match="max_traj_len"):
        task.autoreset(**ok, max_traj_len=0)
    with pytest.raises(ValueError, match="outside"):
        task.autoreset(**ok, n=5)


def test_autoreset_entry_point_fails_loudly_without_gpu():
    import ctypes
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from olympics_mujoco_b200 import _lib
    from olympics_mujoco_b200 import kernels as Kn
    task = object.__new__(Kn.A3Task)
    task.n = 4
    f = lambda *s: torch.zeros(s)
    with pytest.raises(_lib.OmError, match="no CUDA device"):
        task.autoreset(f(25, 4), f(24, 4), torch.zeros(4, dtype=torch.uint8), torch.zeros(4, dtype=torch.int32), f(41, 4),
                       f(41, 4), torch.zeros(4, dtype=torch.uint8), torch.zeros(4, dtype=torch.uint8))
    lib = _lib.load()
    assert lib.om_a3_autoreset(None, None, 0, 0, None, 4, 4, None) != 0
    assert b"null argument" in lib.om_last_error()
    assert "om_a3_autoreset" in _lib.PROTOTYPES and ctypes.sizeof(_lib.OmA3AutoResetArgs) > 0
