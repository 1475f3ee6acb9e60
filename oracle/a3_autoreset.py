"""Oracle: the PPO sampler's loop for one StickFigureA3 env, float64 NumPy (TEST INFRASTRUCTURE).

Restates the per-worker loop of ``PPO.sample`` (reference ``rl/algos/ppo.py:150-198``)::

    state = env.reset(); done = False; traj_len = 0
    while not done and traj_len < max_traj_len:
        action = policy(state); value = critic(state)
        next_state, reward, done, _ = env.step(action)
        memory.store(state, action, reward, value)
        state = next_state; traj_len += 1
    memory.finish_path(last_val=(not done) * critic(state))

run back to back over a fixed number of steps, as the batched buffer does: when a path ends the env is reset
(``oracle.a3.reset`` with the env's next reset counter) and a new path starts.  The physics between two observations is
scripted: the post-physics ``(qpos, qvel, Contact)`` of every step is given.  A path still running at the end of the
script is cut there and finished with ``last_val = critic(state)``, the bootstrap the reference uses at ``max_traj_len``.
"""
import numpy as np

from . import a3 as OA
from . import learner as L

ENDED, TRUNCATED = 1, 2          # path_end codes (om_ppo_returns)


def ints_of(ts):
    """The device's ``ints`` row of a task state: phase, t1, t2, target_reached_frames, mode, seq_len, target_reached."""
    return [ts.phase, ts.t1, ts.t2, ts.target_reached_frames, ts.mode, ts.seq_len, int(ts.target_reached)]


def sample(model, states, clock_lut, max_traj_len=None, seed=0, env_id=0, iteration_count=np.inf, reset_count0=0):
    """One env through ``len(states)`` steps of the sampler loop.  ``states[t] = (qpos [25], qvel [24], OA.Contact)``;
    ``max_traj_len`` None = only ``done`` ends a path; ``reset_count0`` = the env's reset counter of its first reset.

    Returns dict of arrays indexed by step: ``obs`` (the state the step's action is taken in), ``final_obs`` (the step's
    own observation, ``next_state``), ``reward``, ``done``, ``trunc`` (``traj_len`` reached ``max_traj_len``), ``last``,
    ``path_end`` (1 done, 2 truncated, 0 the path goes on), and after the step's reset, if any: ``traj_len``,
    ``reset_count``, ``ints`` [T, 7], ``sequence`` [T, 20, 4], ``next_obs`` (the next step's ``obs``);  ``initial`` = the
    first reset's (qpos, qvel, ts, obs)."""
    rc = int(reset_count0)
    first = OA.reset(model, seed, env_id, rc, iteration_count)
    rc += 1
    ts, obs, traj_len = first[2], first[3], 0
    keys = ("obs", "final_obs", "reward", "done", "trunc", "last", "path_end", "traj_len", "reset_count", "ints", "sequence",
            "next_obs")
    rec = {k: [] for k in keys}
    for qpos, qvel, con in states:
        pre = obs
        final, reward, done, _ = OA.step_tail(model, np.asarray(qpos, np.float64), np.asarray(qvel, np.float64), ts, con,
                                              clock_lut)
        traj_len += 1
        trunc = max_traj_len is not None and traj_len >= max_traj_len
        last = done or trunc
        obs = final
        if last:
            _, _, ts, obs = OA.reset(model, seed, env_id, rc, iteration_count)
            rc += 1
            traj_len = 0
        for k, v in (("obs", pre), ("final_obs", final), ("reward", reward), ("done", done), ("trunc", trunc),
                     ("last", last), ("path_end", ENDED if done else (TRUNCATED if trunc else 0)), ("traj_len", traj_len),
                     ("reset_count", rc), ("ints", ints_of(ts)), ("sequence", np.array(ts.sequence, np.float64)),
                     ("next_obs", obs)):
            rec[k].append(v)
    out = {k: np.asarray(v) for k, v in rec.items()}
    out["initial"] = first
    return out


def paths(rec):
    """[(start, stop)] step ranges of the paths of a ``sample`` record; the last one may be cut by the end of the script."""
    out, start = [], 0
    for t, last in enumerate(rec["last"]):
        if last:
            out.append((start, t + 1))
            start = t + 1
    if start < len(rec["last"]):
        out.append((start, len(rec["last"])))
    return out


def path_returns(rec, critic, gamma):
    """PPOBuffer.finish_path of every path of ``rec`` with the reference's bootstrap ``(not done) * critic(state)``, ``state``
    the step's own observation after the path's last step.  ``critic(obs [41]) -> float``.  Returns (returns [T],
    advantages [T]) with ``advantage = return - critic(obs)``."""
    T = len(rec["reward"])
    ret, adv = np.empty(T), np.empty(T)
    for a, b in paths(rec):
        values = np.array([critic(o) for o in rec["obs"][a:b]])
        r, d = L.ppo_returns(rec["reward"][a:b, None], values[:, None], bool(rec["done"][b - 1]),
                             critic(rec["final_obs"][b - 1]), gamma)
        ret[a:b], adv[a:b] = r[:, 0], d[:, 0]
    return ret, adv
