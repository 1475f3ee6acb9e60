"""Oracle: per-env reset and mushroom_rl Core's episode loop for one UnitreeH1 env, float64 NumPy (TEST INFRASTRUCTURE).

Restates
* ``LocoEnvBase.reset``                 ``environments/loco_env_base.py:568-604`` (imitation-learning branch) with
  ``setup`` ``:606-657``: ``mj_resetData`` (qpos = qpos0, qvel = 0), ``mean_grf.reset()`` (:584), the trajectory reset under
  the ``random_start`` / ``init_step_no`` rules, ``set_sim_state`` of its sample, ``_create_observation(_build_obs(data))``;
* mushroom_rl ``Core`` (``core.py``, ``Core._step`` / ``_reset``; mushroom_rl is not installed here, as SURVEY.md A.2 restates
  its other pieces): after every step ``last = absorbing or episode_steps >= info.horizon``, and an env whose episode ended is
  reset alone; the recorded sample keeps the step's own observation as ``next_state``;
* the model an env draws at its own partial reset with a per-env carried weight (the Philox contract, stream 33).
"""
import numpy as np

from . import h1 as OH
from . import philox
from .trajectory import TrajectoryState

STREAM_MODEL_RESET = 32            # the model switch of a whole reset() (MultiMuJoCo, om_h1_draw_models)
STREAM_PARTIAL_MODEL_RESET = 33    # the model one env draws at its own partial reset (om_h1_reset_envs)


def partial_model_draw(seed, env_id, j, n_models, prev_index, random=True):
    """Model of env ``env_id`` (global id) after its ``j``-th partial reset (0-based): Philox(seed; env_id, j, 33) word 0 by
    multiply-shift, or the next model after ``prev_index`` in round robin."""
    if random:
        w = philox.draw(seed, np.uint32(env_id), np.uint32(j), STREAM_PARTIAL_MODEL_RESET)
        return int(philox.to_int(w[0], n_models))
    return (int(prev_index) + 1) % int(n_models)


def setup_forcing(random_start=True, init_step_no=None, traj_len=None):
    """(substep_no, traj_no) that setup() passes to reset_trajectory (None = drawn), loco_env_base.py:640-657."""
    if init_step_no is not None and random_start:
        raise ValueError("Either use a random start or set an initial step, not both.")
    if random_start:
        return None, None
    if init_step_no:
        return int(init_step_no % traj_len), int(init_step_no / traj_len)
    return 0, None


def reset_env(model, traj_state, random_start=True, init_step_no=None, grf_size=0):
    """The reset of ONE env (LocoEnvBase.reset for that env alone).  Advances ``traj_state`` (its reset_count included) and
    returns dict(qpos, qvel, obs, prev_x_vel, traj_no, step_no, reset_count); ``obs`` ends with ``grf_size`` zeros."""
    substep, traj_no = setup_forcing(random_start, init_step_no, traj_state.T)
    sample = traj_state.reset_trajectory(substep_no=substep, traj_no=traj_no)
    P = OH.perm(model)
    nj = len(P)
    qpos = np.asarray(model.qpos0, dtype=np.float64).copy()            # mj_resetData
    qvel = np.zeros(model.nv)
    qpos[P] = sample[:nj]                                               # set_sim_state :659-684
    qvel[P] = sample[nj:2 * nj]
    obs = np.concatenate([OH.create_observation(OH.build_obs(model, qpos, qvel)), np.zeros(grf_size)])
    return dict(qpos=qpos, qvel=qvel, obs=obs, prev_x_vel=obs[OH.x_vel_idx(model)], traj_no=traj_state.traj_no,
                step_no=traj_state.step_no, reset_count=traj_state.reset_count)


def step_obs(model, qpos, qvel, prev_obs, use_absorbing_states=True, target=OH.TARGET_VELOCITY_WALK, grf=None):
    """The step tail without FK: observation (+ GRF / 1000), absorbing, TargetVelocityReward on the previous observation."""
    obs = OH.create_observation(OH.build_obs(model, qpos, qvel))
    absorbing = bool(OH.has_fallen(obs)) and bool(use_absorbing_states)
    reward = float(OH.target_velocity_reward(prev_obs, OH.x_vel_idx(model), target))
    if grf is not None:
        obs = np.concatenate([obs, np.asarray(grf, dtype=np.float64) / 1000.0])
    return obs, absorbing, reward


def core_rollout(model, table, states, horizon, seed=0, env_id=0, use_absorbing_states=True, random_start=True,
                 init_step_no=None, target=OH.TARGET_VELOCITY_WALK, grfs=None, reset_count0=0):
    """mushroom_rl Core driving one env: the env is reset, then for each scripted post-physics ``(qpos, qvel)`` of
    ``states`` the step runs, ``episode_steps += 1``, ``last = absorbing or episode_steps >= horizon``, and the env is reset
    if ``last``.  ``grfs`` ([T, 6] or None): the contact forces of each step (use_foot_forces); ``reset_count0``: the env's
    trajectory resets before this rollout.

    Returns dict of arrays indexed by step: obs (after the reset, the input to the next action), final_obs (the step's own
    observation, the transition's next_state), reward, absorbing, last, episode_step, traj_no, step_no, reset_count;
    ``initial`` = the first reset's record."""
    grf_size = 0 if grfs is None else np.asarray(grfs).shape[-1]
    tr = TrajectoryState(table, seed=seed, env_id=env_id)
    tr.reset_count = int(reset_count0)
    first = reset_env(model, tr, random_start, init_step_no, grf_size)
    obs, episode_steps = first["obs"], 0
    rec = {k: [] for k in ("obs", "final_obs", "reward", "absorbing", "last", "episode_step", "traj_no", "step_no",
                           "reset_count")}
    for t, (qpos, qvel) in enumerate(states):
        final, absorbing, reward = step_obs(model, qpos, qvel, obs, use_absorbing_states, target,
                                            None if grfs is None else grfs[t])
        episode_steps += 1
        last = absorbing or episode_steps >= horizon
        obs = final
        if last:
            obs = reset_env(model, tr, random_start, init_step_no, grf_size)["obs"]
            episode_steps = 0
        for k, v in (("obs", obs), ("final_obs", final), ("reward", reward), ("absorbing", absorbing), ("last", last),
                     ("episode_step", episode_steps), ("traj_no", tr.traj_no), ("step_no", tr.step_no),
                     ("reset_count", tr.reset_count)):
            rec[k].append(v)
    out = {k: np.asarray(v) for k, v in rec.items()}
    out["initial"] = first
    return out
