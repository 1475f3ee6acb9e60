"""CPU: the plain-C oracle (oracle/c, engine-style formulation) against the NumPy oracle -- two independently
written restatements of the same third-party arithmetic must agree to float64 round-off."""
import numpy as np

from conftest import GOLDEN, a3_random_states, assert_close
from oracle import c_oracle
from oracle import h1 as OH
from oracle import kinematics as K
from oracle import learner as L


def test_forward_matches_numpy_oracle(h1_model, a3_model, h1_states):
    for model, (q, v) in ((h1_model, h1_states), (a3_model, a3_random_states(a3_model, 200, seed=4))):
        a = c_oracle.forward(c_oracle.CModel(model), q, v)
        b = K.forward(model, q, v)
        for k in ("xpos", "xquat", "site_xpos", "site_xmat", "cvel", "subtree_com"):
            assert_close(a[k], b[k], k, rtol=1e-12, atol=1e-12)


def test_h1_playback_matches_numpy_oracle(h1_model):
    tab = np.load(GOLDEN / "trajectory_ref.npz")["table"]
    n_env, n_steps, seed = 5, 130, 4242
    o = c_oracle.h1_play(c_oracle.CModel(h1_model), OH.perm(h1_model), tab, seed, 3, n_env, n_steps)
    for e in range(n_env):
        ref = OH.play_trajectory_from_velocity(h1_model, tab, 1, n_steps, seed=seed, env_id=3 + e)
        assert np.array_equal(o["traj_no"][e], ref["traj_no"]) and np.array_equal(o["step_no"][e], ref["step_no"])
        assert np.array_equal(o["fallen"][e].astype(bool), ref["fallen"])
        assert np.array_equal(o["obs"][e], ref["obs"])
        assert_close(o["reward"][e], ref["reward"], "reward", rtol=1e-13, atol=1e-13)
        for k, w in (("xpos", 63), ("xquat", 84), ("site_xpos", 3), ("cvel", 126)):
            assert_close(o[k][e], ref[k].reshape(n_steps, w), k, rtol=1e-12, atol=1e-12)


_FK_WIDTH = (("xpos", 63), ("xquat", 84), ("site_xpos", 3), ("cvel", 126))


def _assert_call_matches(o, lo, hi, e, ref):
    """Slots lo:hi of env e of a C oracle call against one call of the NumPy oracle."""
    assert np.array_equal(o["traj_no"][e, lo:hi], ref["traj_no"]) and np.array_equal(o["step_no"][e, lo:hi], ref["step_no"])
    assert np.array_equal(o["fallen"][e, lo:hi].astype(bool), ref["fallen"])
    assert np.array_equal(o["obs"][e, lo:hi], ref["obs"])
    assert_close(o["reward"][e, lo:hi], ref["reward"], "reward", rtol=1e-13, atol=1e-13)
    for k, w in _FK_WIDTH:
        assert_close(o[k][e, lo:hi], ref[k].reshape(hi - lo, w), k, rtol=1e-12, atol=1e-12)


def _assert_state_matches(state, e, fin, tab):
    """The C oracle's carried state of env e against the NumPy oracle's ``final`` (taken right after its call: the
    trajectory object inside it goes on with the next call)."""
    nj = tab.shape[0] // 2
    tr, st = fin["traj_no"], fin["step_no"]
    assert (state["traj_no"][e], state["step_no"][e], state["reset_count"][e]) == (tr, st, fin["reset_count"])
    assert np.array_equal(state["xy_off"][e], tab[:2, tr, st])
    assert_close(state["curr_qpos"][e], fin["curr_qpos"], "curr_qpos", rtol=1e-12, atol=1e-12)
    assert np.array_equal(state["pending"][e], fin["pending_sample"])
    assert state["prev_x_vel"][e] == fin["traj_state"].get_current_sample()[nj]


def test_h1_playback_chained_calls_match_numpy_oracle(h1_model):
    """Two calls on one carried state (what the environment does when it plays again: the second call begins with its
    own reset(), reset_count goes on) at a nonzero env_id0, every output and the state after each call."""
    tab = np.load(GOLDEN / "trajectory_ref.npz")["table"]
    n_env, env_id0, seed = 4, 11, 4242
    cm, perm = c_oracle.CModel(h1_model), OH.perm(h1_model)
    state = c_oracle.play_state(tab.shape[0], n_env)
    first = c_oracle.h1_play(cm, perm, tab, seed, env_id0, n_env, 37, n_episodes=2, state=state)
    s1 = {k: v.copy() for k, v in state.items()}
    second = c_oracle.h1_play(cm, perm, tab, seed, env_id0, n_env, 60, state=state)
    for e in range(n_env):
        ref = OH.play_trajectory_from_velocity(h1_model, tab, 2, 37, seed=seed, env_id=env_id0 + e)
        _assert_call_matches(first, 0, 74, e, ref)
        _assert_state_matches(s1, e, ref["final"], tab)
        ref = OH.play_trajectory_from_velocity(h1_model, tab, 1, 60, seed=seed, env_id=env_id0 + e,
                                               traj_state=ref["final"]["traj_state"])
        _assert_call_matches(second, 0, 60, e, ref)
        _assert_state_matches(state, e, ref["final"], tab)
    assert (state["reset_count"] >= 5).all()           # 2 + 1 end resets, 2 start resets, wraps of the 50-sample table


def test_h1_playback_continued_call_equals_one_multi_episode_call(h1_model):
    """A call with start_reset=False after one that ended with its reset continues exactly where a single two-episode
    call goes on (the first step integrates the stale sample's velocities from the reset's positions, :555-557), bit
    for bit; without outputs (NULL pointers) the same state and checksum come out."""
    tab = np.load(GOLDEN / "trajectory_ref.npz")["table"]
    n_env, env_id0, seed, n = 6, 917, 77, 45
    cm, perm = c_oracle.CModel(h1_model), OH.perm(h1_model)
    whole_state = c_oracle.play_state(tab.shape[0], n_env)
    whole = c_oracle.h1_play(cm, perm, tab, seed, env_id0, n_env, n, n_episodes=2, state=whole_state)
    state = c_oracle.play_state(tab.shape[0], n_env)
    a = c_oracle.h1_play(cm, perm, tab, seed, env_id0, n_env, n, state=state)
    b = c_oracle.h1_play(cm, perm, tab, seed, env_id0, n_env, n, state=state, start_reset=False)
    for k in ("xpos", "xquat", "site_xpos", "cvel", "obs", "reward", "fallen", "traj_no", "step_no"):
        assert np.array_equal(np.concatenate([a[k], b[k]], axis=1), whole[k]), k
    for k in whole_state:
        assert np.array_equal(state[k], whole_state[k]), k
    ref = OH.play_trajectory_from_velocity(h1_model, tab, 2, n, seed=seed, env_id=env_id0 + 2)
    _assert_call_matches(whole, 0, 2 * n, 2, ref)
    _assert_state_matches(whole_state, 2, ref["final"], tab)
    # NULL output pointers skip those outputs, nothing else
    bare_state = c_oracle.play_state(tab.shape[0], n_env)
    bare = c_oracle.h1_play(cm, perm, tab, seed, env_id0, n_env, n, n_episodes=2, state=bare_state, record=False)
    assert set(bare) == {"checksum"} and np.array_equal(bare["checksum"], whole["checksum"])
    for k in whole_state:
        assert np.array_equal(bare_state[k], whole_state[k]), k


def test_gae_matches_numpy_oracle():
    rng = np.random.default_rng(2)
    n, T = 6, 80
    r, v, vn = rng.normal(0, 1, (3, n, T))
    last = rng.random((n, T)) < 0.1
    ab = last & (rng.random((n, T)) < 0.5)
    vt, adv = c_oracle.gae(r, v, vn, ab, last, 0.99, 0.97)
    for e in range(n):
        f_vt, f_adv = L.compute_gae(v[e], vn[e], r[e], ab[e], last[e], 0.99, 0.97)
        assert_close(adv[e], f_adv, "adv", rtol=1e-13, atol=1e-13)
        assert_close(vt[e], f_vt, "vt", rtol=1e-13, atol=1e-13)
