"""Batched ``StickFigureA3`` in reinforcement-learning mode (reference
``real_humanoid_robots/StickFigureA3.py``: ``_initialize_observation_space`` :69-141, ``get_obs`` :144-181, ``step``
:187-202, ``reset_model`` :205-235; PD stepper ``environments/robot.py``).

``step(a)`` keeps the reference's contract ``(obs, total_reward, done, rewards_dict)`` for n envs.  The physics
between two observations (``robot.step`` -> frame_skip x [PD law -> ``mj_step``]) is NOT part of this path: it is an
attached callable returning the post-physics ``qpos``, ``qvel`` and the four contact-solver summaries the task reads;
everything after it runs in one fused CUDA kernel (``om_a3_task_step``).

``step(a, autoreset=True, max_traj_len=L)`` adds the path bookkeeping of the reference's PPO sampler
(``rl/algos/ppo.py:150-198``) in one more kernel (``om_a3_autoreset``) on the same stream: each env counts the steps of its
path (``traj_len``), a path ends on ``done`` or after ``L`` steps, and an env whose path ended is reset alone."""
from __future__ import annotations

import numpy as np
import torch

from .. import kernels as Kn
from .. import mjcf
from ..tasks.walking_task import REWARD_KEYS, WalkingTask

HALF_SITTING_DEG = [-30, 0, 0, 50, 0, -24, -30, 0, 0, 50, 0, -24, -3, -9.74, -30, -3, 9.74, -30]   # robot.py:61-66


class JVRC:
    """environments/robot.py: nominal pose, motor offsets, PD gains and the symmetry tables; ``step`` forwards the
    offset action to the attached physics."""

    def __init__(self, pdgains, dt, active, model, sim_dt):
        self.control_dt, self.actuators = dt, list(active)
        self.kp, self.kd = np.asarray(pdgains[0]), np.asarray(pdgains[1])
        assert self.kp.shape == self.kd.shape == (len(model.actuator_names),)                 # robot.py:44
        if np.around(dt % sim_dt, 6):
            raise Exception("Control dt should be an integer multiple of Simulation dt.")     # robot.py:56-57
        self.frame_skip = int(dt / sim_dt)
        self.iteration_count = np.inf
        pose = [0, 0, 0.81] + [1, 0, 0, 0] + [q * np.pi / 180.0 for q in HALF_SITTING_DEG]
        assert len(pose) == model.nq
        self.init_qpos_, self.init_qvel_ = list(pose), [0] * model.nv
        adr = [int(model.jnt_qposadr[model.jnt_names.index(j)]) for j in model.actuator_joint]
        self.motor_offset = np.array([self.init_qpos_[i] for i in adr])
        self.prev_action = None
        dadr = [int(model.jnt_dofadr[model.jnt_names.index(j)]) for j in model.actuator_joint]
        gear = np.asarray(model.actuator_gear, dtype=np.float64).reshape(len(adr), -1)[:, 0]
        self._pd_spec = Kn.make_pd_spec(adr, dadr, self.kp, self.kd, gear, np.zeros(len(adr)))

    def pd_ctrl(self, target, qpos, qvel):
        """One PD evaluation of do_simulation (robot.py:109-115 around step_pd): ``ctrl = (kp (target - q) - kd dq) / gear``
        for target [12, n], qpos [25, n], qvel [24, n]; the physics callable runs it once per simulation sub-step."""
        return Kn.pd_torque(self._pd_spec, target, qpos, qvel, add_offset=False)


class StickFigureA3:
    def __init__(self, n_envs=None, device="cuda", seed=0, env_id0=0, algorithm_type="reinforcement_learning", **_ignored):
        if str(algorithm_type).lower().split(".")[-1] != "reinforcement_learning":
            raise NotImplementedError("StickFigureA3: only the reinforcement-learning mode is on this path "
                                      "(the reference's imitation-learning branch is a stub that prints a message)")
        self._single = n_envs is None
        self.n_envs = 1 if n_envs is None else int(n_envs)
        self._device = device
        self._model = mjcf.load_builtin("stick_figure_a3")
        self._dm = Kn.DeviceModel(self._model)
        sim_dt, control_dt = 0.0025, 0.025                                                    # StickFigureA3.py:72-74
        coeff = 0.5
        kp = coeff * np.array([200, 200, 200, 250, 80, 80, 200, 200, 200, 250, 80, 80], dtype=np.float64)
        kd = coeff * np.array([20, 20, 20, 25, 8, 8, 20, 20, 20, 25, 8, 8], dtype=np.float64)
        self.actuators = list(range(12))
        self.task = WalkingTask(dt=control_dt, root_body="torso", lfoot_body="left_foot", rfoot_body="right_foot",
                                head_body="head")
        self.robot = JVRC((kp, kd), control_dt, self.actuators, self._model, sim_dt)
        base_mir_obs = [0.1, -1, 2, -3, -4, 5, -6, 13, -14, -15, 16, -17, 18, 7, -8, -9, 10, -11, 12,
                        25, -26, -27, 28, -29, 30, 19, -20, -21, 22, -23, 24]                 # :118-125
        append_obs = [len(base_mir_obs) + i for i in range(10)]
        self.robot.clock_inds = append_obs[0:2]
        self.robot.mirrored_obs = base_mir_obs + append_obs
        self.robot.mirrored_acts = [6, -7, -8, 9, -10, 11, 0.1, -1, -2, 3, -4, 5]
        self.action_space = np.zeros(len(self.actuators))
        self.base_obs_len = 41
        self.observation_space = np.zeros(self.base_obs_len)
        self._dev = Kn.A3Task(self._dm, self.n_envs, self.task.clock_lut, self.robot.init_qpos_, period=self.task._period,
                              delay_frames=self.task.delay_frames, target_radius=self.task.target_radius,
                              goal_height_ref=self.task._goal_height_ref, goal_speed_ref=self.task._goal_speed_ref,
                              seed=seed, env_id0=env_id0, device=device)
        self.task.bind(self._dev)
        self.qpos = Kn.soa(self._model.nq, self.n_envs, device=device)
        self.qvel = Kn.soa(self._model.nv, self.n_envs, device=device)
        self._obs = Kn.soa(41, self.n_envs, device=device)
        # steps of each env's current path (the sampler's traj_len); advanced by step(autoreset=True)
        self.traj_len = torch.zeros(self.n_envs, dtype=torch.int32, device=device)
        self._dynamics = None

    # ------------------------------------------------------------------ helpers
    def _out(self, x):
        return x[0] if self._single else x

    def attach_dynamics(self, fn):
        """``fn(env, target [n, 12]) -> (qpos [25, n], qvel [24, n], contact [4, n])`` (float32 CUDA, SoA): the
        reference's ``robot.step`` physics (robot.py:88-115) plus the contact summaries the task reads."""
        self._dynamics = fn

    def get_obs(self):
        return self._out(self._obs.t())

    # ------------------------------------------------------------------ reset / step
    def reset_model(self, mask=None):
        """StickFigureA3.py:205-235 (+ WalkingTask.reset) for every env, or the envs selected by ``mask``; their
        ``traj_len`` restarts at 0."""
        if mask is not None:
            mask = torch.as_tensor(mask, device=self._device).to(torch.uint8)
        self._dev.reset(self.qpos, self.qvel, mask=mask, iteration_count=self.robot.iteration_count, obs=self._obs)
        if mask is None:
            self.traj_len.zero_()
        else:
            self.traj_len.masked_fill_(mask.bool(), 0)
        return self.get_obs()

    def reset(self, obs=None):
        """loco_env_base.py:577-579 -> test_reset :220-223 -> reset_model."""
        return self.reset_model()

    def step(self, a, autoreset=False, max_traj_len=None):
        """StickFigureA3.py:187-202 -> (obs, reward, done, rewards dict).

        ``autoreset=True`` runs the reference's PPO sampler loop (rl/algos/ppo.py:150-198) on the device, after the step
        kernel and without a host synchronisation: ``traj_len += 1``; a path ends on ``done`` or when ``traj_len`` reaches
        ``max_traj_len`` (None: only ``done`` ends it); every env whose path ended is reset exactly as
        ``reset_model(mask=last)`` resets it.  ``obs`` is then the observation after those resets (the next action's
        input); ``reward`` and ``done`` are the step's own.  The dict gains ``last`` ([n] bool), ``path_end`` ([n] uint8: 1
        done -- bootstrap 0, it wins over a truncation on the same step; 2 truncated -- bootstrap V(final_obs); 0 the path
        goes on: the codes of ``learners.finish_path``), ``final_obs`` ([n, 41], the step's observation of every env: the
        ``next_state`` V is evaluated on at a truncation) and ``traj_len`` ([n] int32, after the update)."""
        if max_traj_len is not None and int(max_traj_len) < 1:
            raise ValueError(f"max_traj_len must be None or >= 1, got {max_traj_len}")
        if self._dynamics is None:
            raise RuntimeError("StickFigureA3.step needs the physics: call attach_dynamics(fn) first "
                               "(contact dynamics are outside this package)")
        a = torch.as_tensor(a, device=self._device, dtype=torch.float32)
        a = a.unsqueeze(0) if a.dim() == 1 else a
        target = torch.zeros((self.n_envs, len(self.robot.motor_offset)), device=self._device)
        target[:, self.actuators] = a                                                         # robot.py:89-93
        target += torch.as_tensor(self.robot.motor_offset, device=self._device, dtype=torch.float32)
        qpos, qvel, contact = self._dynamics(self, target)
        self.qpos.copy_(qpos)
        self.qvel.copy_(qvel)
        self.robot.prev_action = target
        if autoreset:
            return self._step_autoreset(contact.contiguous(), max_traj_len)
        out = self._dev.step(self.qpos, self.qvel, contact.contiguous(), out=dict(obs=self._obs))
        rewards = {k: self._out(out["terms"][i]) for i, k in enumerate(REWARD_KEYS)}
        return self.get_obs(), self._out(out["reward"]), self._out(out["done"].bool()), rewards

    def _step_autoreset(self, contact, max_traj_len):
        """step(autoreset=True) after the physics: the step kernel writes the step's observation (final_obs), then
        om_a3_autoreset writes the returned observation, traj_len, last and path_end and resets the envs whose path ended."""
        final = Kn.soa(41, self.n_envs, device=self._device)
        out = self._dev.step(self.qpos, self.qvel, contact, out=dict(obs=final))
        new = torch.empty_like(final)
        last = torch.empty(self.n_envs, dtype=torch.uint8, device=self._device)
        path_end = torch.empty_like(last)
        self._dev.autoreset(self.qpos, self.qvel, out["done"], self.traj_len, final, new, last, path_end,
                            max_traj_len=max_traj_len, iteration_count=self.robot.iteration_count)
        self._obs = new
        rewards = {k: self._out(out["terms"][i]) for i, k in enumerate(REWARD_KEYS)}
        rewards.update(last=self._out(last.view(torch.bool)), path_end=self._out(path_end), final_obs=self._out(final.t()),
                       traj_len=self._out(self.traj_len.clone()))
        return self.get_obs(), self._out(out["reward"]), self._out(out["done"].bool()), rewards

    def _has_fallen(self, obs, return_err_msg=False):
        """StickFigureA3.py:376-389: always False."""
        return (False, "") if return_err_msg else False
