"""CPU: the per-env reset and auto-reset of the batched UnitreeH1 step -- the oracle's mushroom_rl Core loop on hand-built
episodes, the partial-reset model draw against Philox4x32-10, the argument checks of ``reset(mask=...)`` and the loud failure
of the new entry point without a GPU."""
import numpy as np
import pytest

from conftest import GOLDEN


def _model():
    from olympics_mujoco_b200 import mjcf
    return mjcf.load_builtin("unitree_h1")


def _table(model):
    from oracle import h1 as OH
    full = ["q_" + j for j in OH._SPEC_JOINTS] + ["dq_" + j for j in OH._SPEC_JOINTS]
    full = [k for k in full if not any(a in k for a in OH.ARM_JOINTS)]
    tab = np.load(GOLDEN / "trajectory_ref.npz")["table"].copy()[[full.index(k) for k in OH.keys(model)]]
    tab[2:] = tab[2:].astype(np.float32).astype(np.float64)
    return tab


def _states(model, table, n_steps, fall_at=()):
    """Scripted post-physics states: trajectory rows; at the steps of ``fall_at`` pelvis_ty is pushed below -0.3."""
    from oracle import h1 as OH
    out = []
    for t in range(n_steps):
        s = table[:, 0, 5 + t].copy()
        if t in fall_at:
            s[2] = -0.5                                   # q_pelvis_ty: UnitreeH1.py:173 pelvis_y_condition
        out.append(OH.set_sim_state(model, s))
    return out


def _run(fall_at, horizon, n_steps=7, **kw):
    from oracle import h1_autoreset as OA
    m = _model()
    tab = _table(m)
    return OA.core_rollout(m, tab, _states(m, tab, n_steps, fall_at), horizon, seed=4, env_id=3, **kw), m, tab


def test_core_loop_horizon_cut():
    r, m, tab = _run((), horizon=3)
    assert r["last"].tolist() == [False, False, True, False, False, True, False]
    assert r["episode_step"].tolist() == [1, 2, 0, 1, 2, 0, 1]
    assert not r["absorbing"].any()
    assert r["reset_count"].tolist() == [1, 1, 2, 2, 2, 3, 3]           # the first reset, then one per ended episode
    for t in range(7):
        if r["last"][t]:                                                    # the new episode's first observation
            assert np.array_equal(r["obs"][t], tab[2:, r["traj_no"][t], r["step_no"][t]])
            assert not np.array_equal(r["obs"][t], r["final_obs"][t])
        else:
            assert np.array_equal(r["obs"][t], r["final_obs"][t])


def test_core_loop_absorbing_before_horizon():
    r, _, _ = _run((1,), horizon=5)
    assert r["absorbing"].tolist() == [False, True, False, False, False, False, False]
    assert r["last"].tolist() == [False, True, False, False, False, False, True]
    assert r["episode_step"].tolist() == [1, 0, 1, 2, 3, 4, 0]
    assert r["final_obs"][1][0] == -0.5                                    # next_state keeps the fallen observation
    assert r["obs"][1][0] != -0.5


def test_core_loop_absorbing_exactly_at_horizon():
    r, _, _ = _run((2,), horizon=3)
    assert r["absorbing"][2] and r["last"][2]
    assert r["last"].tolist() == [False, False, True, False, False, True, False]
    assert r["reset_count"][-1] == 3                                       # one reset, not two, at step 2


def test_core_loop_without_absorbing_states():
    r, _, _ = _run((1, 4), horizon=3, use_absorbing_states=False)
    assert not r["absorbing"].any()
    assert r["last"].tolist() == [False, False, True, False, False, True, False]


def test_core_loop_reward_reads_the_observation_after_the_reset():
    from oracle import h1 as OH
    r, m, _ = _run((1,), horizon=5)
    xv = OH.x_vel_idx(m)
    for t in range(1, 7):
        assert r["reward"][t] == float(np.exp(-np.square(r["obs"][t - 1][xv] - OH.TARGET_VELOCITY_WALK)))


def test_reset_env_forcing_rules():
    from oracle import h1_autoreset as OA
    from oracle.trajectory import TrajectoryState
    m = _model()
    tab = _table(m)
    T = tab.shape[2]
    a = OA.reset_env(m, TrajectoryState(tab, seed=1, env_id=2), random_start=False, init_step_no=T + 7)
    assert (a["traj_no"], a["step_no"], a["reset_count"]) == (1, 7, 1)
    b = OA.reset_env(m, TrajectoryState(tab, seed=1, env_id=2), random_start=False)
    assert b["step_no"] == 0
    assert np.array_equal(b["qpos"][OA.OH.perm(m)][:2], [0.0, 0.0])       # root x, z re-centred
    assert a["prev_x_vel"] == a["obs"][OA.OH.x_vel_idx(m)]
    with pytest.raises(ValueError):
        OA.reset_env(m, TrajectoryState(tab), random_start=True, init_step_no=3)
    g = OA.reset_env(m, TrajectoryState(tab), grf_size=6)
    assert g["obs"].shape == (2 * len(OA.OH.perm(m)) - 2 + 6,) and not g["obs"][-6:].any()


def test_partial_reset_draws_follow_philox():
    from olympics_mujoco_b200.utils import philox as HP
    from oracle import h1_autoreset as OA
    from oracle import philox
    seed = (5 << 32) | 123
    assert HP.STREAM_PARTIAL_MODEL_RESET == OA.STREAM_PARTIAL_MODEL_RESET == 33
    assert HP.STREAM_MODEL_RESET == OA.STREAM_MODEL_RESET == 32
    for env in (0, 1, 17, 2 ** 31 + 5):
        for j in (0, 1, 2, 99):
            w = philox.philox4x32_10((env, j, 33, 0), (seed & 0xFFFFFFFF, seed >> 32))
            want = int((int(w[0]) * 4) >> 32)
            assert HP.env_partial_model_draw(seed, env, j, 4, 0) == want == OA.partial_model_draw(seed, env, j, 4, 0)
            assert HP.env_partial_model_draw(seed, env, j, 4, 2, random=False) == 3 == OA.partial_model_draw(seed, env, j, 4, 2,
                                                                                                           random=False)
    # stream 33 is not the whole-reset stream: over many (env, count) pairs the two draws are not the same sequence
    a = [HP.env_partial_model_draw(seed, e, 0, 4, 0) for e in range(256)]
    b = [HP.env_model_draw(seed, e, 0, 4) for e in range(256)]
    assert a != b and set(a) == {0, 1, 2, 3}


def test_masked_reset_argument_checks():
    import torch
    from olympics_mujoco_b200.environments.unitree_h1 import UnitreeH1
    env = object.__new__(UnitreeH1)               # the checks come before any device work
    env.n_envs, env._device = 4, "cuda"
    with pytest.raises(ValueError, match="obs"):
        UnitreeH1.reset(env, obs=np.zeros((4, 32)), mask=torch.ones(4, dtype=torch.bool))
    for bad in (torch.ones(3, dtype=torch.bool), torch.ones(4, dtype=torch.float32), torch.ones((4, 1), dtype=torch.uint8),
                np.ones(4, dtype=bool), torch.ones(4, dtype=torch.bool)):          # the last one: on the CPU, not the device
        with pytest.raises(ValueError, match="mask"):
            UnitreeH1.reset(env, mask=bad)


def test_reset_entry_point_fails_loudly_without_gpu():
    import ctypes
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from olympics_mujoco_b200 import _lib
    from olympics_mujoco_b200 import kernels as Kn
    with pytest.raises(_lib.OmError, match="no CUDA device"):
        Kn.h1_reset_envs(None, None, None, torch.zeros((17, 4)), torch.zeros((17, 4)), mask=torch.ones(4, dtype=torch.bool))
    lib = _lib.load()
    assert lib.om_h1_reset_envs(None, None, None, 0, 0, None, 4, 4, None) != 0
    assert b"null argument" in lib.om_last_error()
    assert "om_h1_reset_envs" in _lib.PROTOTYPES and ctypes.sizeof(_lib.OmH1ResetArgs) > 0
