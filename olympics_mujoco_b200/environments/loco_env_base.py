"""Batched ``LocoEnvBase``: the reference's environment API over n parallel environments on one B200.

Mirrors ``olympic_mujoco/environments/loco_env_base.py`` (``make`` via mushroom ``Environment.make``,
``reset`` :568-604, ``setup`` :606-657, ``set_sim_state`` :659-684, ``play_trajectory`` :338-442,
``play_trajectory_from_velocity`` :444-560, ``_create_observation`` :737-767, ``reward`` :776-781,
``_get_reward_function`` :783-825, ``create_dataset`` :926-968, ``get_obs_idx`` :1195-1205,
``_get_from_obs`` :1207-1232, ``_len_qpos_qvel`` :1261-1273, ``register`` :1337-1350, ``ValidTaskConf``
:1381-1455) and the pieces of mushroom_rl's ``MuJoCo`` / ``MultiMuJoCo`` it inherits (SURVEY.md A.2).

What differs by design:
* every per-env quantity is a CUDA tensor; observations come back as ``[n_envs, D]`` (``[D]`` when the env
  was made without ``n_envs``, the reference's single-env shape);
* contact dynamics (``mj_step``) are NOT part of this path: ``step`` gets the post-physics state from an
  attached dynamics callable (``attach_dynamics``) and runs the fused FK + observation + absorbing + reward
  kernel on it;
* resets draw from the Philox contract, not NumPy's global stream;
* no viewer: ``render=True`` / ``record=True`` raise NotImplementedError.
"""
from __future__ import annotations

import warnings
from copy import deepcopy
from itertools import product

import numpy as np
import torch

from .. import kernels as Kn
from ..observation_helper import BatchedData, ObservationHelper, ObservationType
from ..utils import CustomReward, NoReward, PosReward, TargetVelocityReward, Trajectory


class Box:
    """mushroom_rl.utils.spaces.Box (low/high/shape only)."""

    def __init__(self, low, high):
        self.low, self.high = np.array(low, dtype=np.float64), np.array(high, dtype=np.float64)

    @property
    def shape(self):
        return self.low.shape


class MDPInfo:
    def __init__(self, observation_space, action_space, gamma, horizon):
        self.observation_space, self.action_space = observation_space, action_space
        self.gamma, self.horizon = gamma, horizon


class LocoEnvBase:
    _registered_envs = dict()

    def __init__(self, model, action_spec, observation_spec, collision_groups=None, gamma=0.99, horizon=1000,
                 n_substeps=10, reward_type=None, reward_params=None, traj_params=None, random_start=True,
                 init_step_no=None, timestep=0.001, use_foot_forces=False, use_absorbing_states=True,
                 n_envs=None, device="cuda", seed=0, env_id0=0, random_env_reset=True, per_env_model=False,
                 **_ignored_viewer_params):
        self._single = n_envs is None
        self.n_envs = 1 if n_envs is None else int(n_envs)
        self._device, self._seed, self._env_id0 = device, int(seed), int(env_id0)
        # mushroom_rl MultiMuJoCo (loco_env_base.py:143-155, reset :586-599): a LIST of models -- the reference passes one
        # xml handle per carried weight -- with one MjData / ObservationHelper each; every reset() switches the env object
        # to the next model, or to a random one.  All n envs of this object share the current model, as the reference's
        # single env does.
        # per_env_model=True (a subclass's opt-in, e.g. UnitreeH1 per_env_weight): the models differ only in quantities the
        # kernels read per env at run time, and every reset() draws a model for EACH env (_draw_env_models); one MjData
        # mirror, device model and observation helper then serve all of them.
        models = list(model) if isinstance(model, (list, tuple)) else [model]
        self._models = models
        self._per_env_model = bool(per_env_model) and len(models) > 1
        self._timestep, self._n_substeps, self._n_intermediate_steps = timestep, n_substeps, 1
        if self._per_env_model:
            data = BatchedData(models[0], self.n_envs, device=device)
            self._datas, self._dms = [data] * len(models), [Kn.DeviceModel(models[0])] * len(models)
            self.obs_helpers = [ObservationHelper(observation_spec, models[0], data, max_joint_velocity=None)] * len(models)
        else:
            self._datas = [BatchedData(m, self.n_envs, device=device) for m in models]
            self._dms = [Kn.DeviceModel(m) for m in models]
            self.obs_helpers = [ObservationHelper(observation_spec, m, d, max_joint_velocity=None)
                                for m, d in zip(models, self._datas)]
        self._current_model_idx, self._random_env_reset, self._model_resets = 0, bool(random_env_reset), 0
        model = models[0]
        self._model, self._data, self._dm, self.obs_helper = model, self._datas[0], self._dms[0], self.obs_helpers[0]
        # mean ground reaction forces (RunningAveragedWindow over the n_intermediate_steps = 1 of a step, :1160-1174):
        # what the contact solver measured enters through set_ground_forces / the dynamics callable
        self._grf = torch.zeros((self._get_grf_size(), self.n_envs), dtype=torch.float32, device=device) \
            if use_foot_forces else None
        self._action_spec = list(action_spec) if action_spec else list(model.actuator_names)
        a_idx = [model.actuator_names.index(a) for a in self._action_spec]
        low = np.where(model.actuator_ctrllimited[a_idx], model.actuator_ctrlrange[a_idx, 0], -np.inf)
        high = np.where(model.actuator_ctrllimited[a_idx], model.actuator_ctrlrange[a_idx, 1], np.inf)
        self.info = MDPInfo(Box(*self.obs_helper.get_obs_limits()), Box(low, high), gamma, horizon)
        self._use_foot_forces = use_foot_forces
        self._reward_function = self._get_reward_function(reward_type, reward_params)
        self.info.observation_space = Box(*self._get_observation_space())
        self.norm_act_mean = (high + low) / 2.0                                  # :165-175
        self.norm_act_delta = (high - low) / 2.0
        self.info.action_space.low[:] = -1.0
        self.info.action_space.high[:] = 1.0
        self._dataset = None
        self.trajectories = None
        if traj_params:
            self.load_trajectory(traj_params)
        self._random_start, self._init_step_no = random_start, init_step_no
        self._use_absorbing_states = use_absorbing_states
        self._dynamics = None
        self._dynamics_soa = False
        self._action_kernel_spec = None
        self._obs = None
        self._play_state = None
        self._live = None

    # the current observation (mushroom's ``self._obs``); a fused playback call leaves it to be derived on first use
    @property
    def _obs(self):
        lazy = self.__dict__.get("_obs_lazy")
        if lazy is not None:
            self.__dict__["_obs_value"] = lazy()
            self.__dict__["_obs_lazy"] = None
        return self.__dict__.get("_obs_value")

    @_obs.setter
    def _obs(self, value):
        self.__dict__["_obs_value"] = value
        self.__dict__["_obs_lazy"] = None

    # ------------------------------------------------------------------ registry / factory
    @classmethod
    def register(cls):
        LocoEnvBase._registered_envs.setdefault(cls.__name__, cls)

    @staticmethod
    def list_registered_loco_mujoco():
        return list(LocoEnvBase._registered_envs.keys())

    @staticmethod
    def make(env_name, *args, **kwargs):
        """mushroom_rl ``Environment.make``: ``"Env.task.dataset"`` -> ``Env.generate(task, dataset, **kw)``."""
        if "." in env_name:
            parts = env_name.split(".")
            env_name, args = parts[0], parts[1:] + list(args)
        if env_name not in LocoEnvBase._registered_envs:
            raise KeyError(f"environment {env_name!r} is not registered "
                           f"(registered: {LocoEnvBase.list_registered_loco_mujoco()})")
        env = LocoEnvBase._registered_envs[env_name]
        if hasattr(env, "generate"):
            return env.generate(*args, **kwargs)
        return env(*args, **kwargs)

    @classmethod
    def get_all_task_names(cls):
        names = []
        for e in cls.list_registered_loco_mujoco():
            env = cls._registered_envs[e]
            for conf in env.valid_task_confs.get_all_combinations():
                names.append(".".join([env.__name__] + list(conf.values())))
        return names

    # ------------------------------------------------------------------ shapes
    @property
    def dt(self):
        return self._timestep * self._n_intermediate_steps * self._n_substeps

    def _out(self, x):
        """[n, ...] -> the reference's single-env shape when the env was made without n_envs."""
        return x[0] if self._single else x

    def _batched(self, x):
        x = torch.as_tensor(x, device=self._device)
        return x.unsqueeze(0) if (self._single and x.dim() == 1) else x

    # ------------------------------------------------------------------ trajectories
    def load_trajectory(self, traj_params, warn=True):
        if self.trajectories is not None:
            warnings.warn("New trajectories loaded, which overrides the old ones.", RuntimeWarning)
        self.trajectories = Trajectory(keys=self.get_all_observation_keys(), low=self.info.observation_space.low,
                                       high=self.info.observation_space.high, joint_pos_idx=self.obs_helper.joint_pos_idx,
                                       interpolate_map=self._interpolate_map, interpolate_remap=self._interpolate_remap,
                                       interpolate_map_params=self._get_interpolate_map_params(),
                                       interpolate_remap_params=self._get_interpolate_remap_params(), warn=warn,
                                       n_envs=self.n_envs, seed=self._seed, env_id0=self._env_id0, device=self._device,
                                       **traj_params)

    def get_all_observation_keys(self):
        return self.obs_helper.get_all_observation_keys()

    # ------------------------------------------------------------------ state
    def set_sim_state(self, sample):
        """:659-684: named scatter of spec-ordered samples [n, len(spec)] into qpos/qvel."""
        sample = self._batched(sample).to(torch.float32)
        spec = self.obs_helper.observation_spec
        assert sample.shape[-1] == len(spec)
        if getattr(self, "_scatter_idx", None) is None:         # spec column -> qpos / qvel row, built once
            cq, rq, cv, rv = [], [], [], []
            for i, (key, name, ot) in enumerate(spec):
                if ot == ObservationType.JOINT_POS:
                    rows = self._data.joint_rows(name)[0]
                    assert rows.stop - rows.start == 1, "set_sim_state handles single-dof joints (as the reference's specs do)"
                    cq.append(i); rq.append(rows.start)
                elif ot == ObservationType.JOINT_VEL:
                    rows = self._data.joint_rows(name)[1]
                    assert rows.stop - rows.start == 1
                    cv.append(i); rv.append(rows.start)
            t = lambda a: torch.as_tensor(a, dtype=torch.long, device=self._device)
            self._scatter_idx = (t(cq), t(rq), t(cv), t(rv))
        cq, rq, cv, rv = self._scatter_idx
        st = sample.t()
        self._data.qpos.index_copy_(0, rq, st.index_select(0, cq))       # two scatters instead of one per key
        self._data.qvel.index_copy_(0, rv, st.index_select(0, cv))

    def set_state(self, qpos, qvel):
        """:1155-1160: write qpos/qvel ([n, nq], [n, nv]) and run the forward pass (K1)."""
        qpos, qvel = self._batched(qpos), self._batched(qvel)
        assert qpos.shape == (self.n_envs, self._model.nq) and qvel.shape == (self.n_envs, self._model.nv)
        self._data.qpos.copy_(qpos.t())
        self._data.qvel.copy_(qvel.t())
        self.forward()

    def forward(self):
        """The hot-path subset of ``mujoco.mj_forward``: kinematics, COM, COM velocity (K1)."""
        d = self._data
        Kn.fk(self._dm, d.qpos, d.qvel, out=dict(xpos=d.xpos, xquat=d.xquat, site_xpos=d.site_xpos,
                                                 site_xmat=d.site_xmat, cvel=d.cvel, subtree_com=d.subtree_com))

    @property
    def data(self):
        return self._data

    def _init_sim_from_obs(self, obs):
        obs = self._batched(obs)
        obs = torch.cat([torch.zeros((obs.shape[0], 2), device=obs.device, dtype=obs.dtype), obs], dim=1)   # :697
        spec = self.obs_helper.observation_spec
        assert obs.shape[1] >= len(spec)
        self.set_sim_state(obs[:, :len(spec)])

    def reset(self, obs=None):
        """:568-604 (imitation-learning branch)."""
        self._data.qpos[:] = torch.as_tensor(self._model.qpos0, dtype=torch.float32, device=self._device)[:, None]
        self._data.qvel.zero_()                                                              # mj_resetData
        if self._grf is not None:
            self._grf.zero_()                                                                # mean_grf.reset() :584
        self._next_model()
        self.setup(obs)
        self._obs = self._create_observation(self.obs_helper._build_obs(self._data))
        return self._out(self._modify_observation(self._obs))

    def _next_model(self):
        """The model switch of reset() (MultiMuJoCo :586-599); nothing with a single model.  Decided on the host; with
        per_env_model every env also draws its own model on the device (the host's pick is env 0's)."""
        if len(self._models) > 1:
            if self._per_env_model:
                self._draw_env_models(self._model_resets)
            if self._random_env_reset:
                # np.random.randint in the reference; here the Philox contract (stream 32, counter = number of resets)
                from ..utils.philox import STREAM_MODEL_RESET, philox_randint
                self._current_model_idx = philox_randint(self._seed, self._env_id0, self._model_resets, STREAM_MODEL_RESET,
                                                         len(self._models))
            else:
                self._current_model_idx = self._current_model_idx + 1 if self._current_model_idx < len(self._models) - 1 else 0
            self._model_resets += 1
            self._select_model(self._current_model_idx)

    def _draw_env_models(self, count):
        raise NotImplementedError

    def _select_model(self, idx):
        if self._per_env_model:               # the one data / device model / helper serve every env's model
            self._model = self._models[idx]
            return
        prev = self._data
        self._model, self._data = self._models[idx], self._datas[idx]
        self._dm, self.obs_helper = self._dms[idx], self.obs_helpers[idx]
        if prev is not self._data:
            self._scatter_idx = None
            self._live = None

    def setup(self, obs):
        """:606-657."""
        self._reward_function.reset_state()
        if obs is not None:
            self._init_sim_from_obs(obs)
            return
        if not self.trajectories and self._random_start:
            raise ValueError("Random start not possible without trajectory data.")
        elif not self.trajectories and self._init_step_no is not None:
            raise ValueError("Setting an initial step is not possible without trajectory data.")
        elif self._init_step_no is not None and self._random_start:
            raise ValueError("Either use a random start or set an initial step, not both.")
        if self.trajectories is not None:
            if self._random_start:
                sample = self.trajectories.reset_trajectory()
            elif self._init_step_no:
                traj_len = self.trajectories.trajectory_length
                n_traj = self.trajectories.number_of_trajectories
                assert self._init_step_no <= traj_len * n_traj
                sample = self.trajectories.reset_trajectory(int(self._init_step_no % traj_len),
                                                            int(self._init_step_no / traj_len))
            else:
                sample = self.trajectories.reset_trajectory(substep_no=0)
            self.set_sim_state(sample)

    # ------------------------------------------------------------------ observations
    @staticmethod
    def _get_grf_size():
        """:1087-1103: four force sensors x 3 by default; UnitreeH1 overrides it (two feet, 6)."""
        return 12

    def set_ground_forces(self, grf):
        """The contact solver's output for the step just simulated: ``_get_ground_forces()`` ([n, grf_size], newtons;
        UnitreeH1.py:113-121 = floor-foot_r[:3], floor-foot_l[:3]).  The solver is outside this package (north star), so
        the forces are an INPUT -- pushed here, or returned as a third value by the dynamics callable.  With one
        intermediate step the running-average window (:1160-1174) holds exactly this sample."""
        if self._grf is None:
            raise RuntimeError("the environment was made without use_foot_forces=True")
        g = self._batched(torch.as_tensor(grf, device=self._device, dtype=torch.float32))
        assert g.shape == (self.n_envs, self._get_grf_size())
        self._grf.copy_(g.t())

    def _get_observation_space(self):
        """:712-735."""
        low, high = self.info.observation_space.low[2:], self.info.observation_space.high[2:]
        if self._use_foot_forces:
            inf = np.ones(self._get_grf_size()) * np.inf
            return np.concatenate([low, -inf]), np.concatenate([high, inf])
        return low, high

    def _create_observation(self, obs):
        """:737-767: drop the root x and y entries; with use_foot_forces append mean_grf / 1000."""
        obs = obs[..., 2:]
        if self._use_foot_forces:
            return torch.cat([obs, self._grf.t().to(obs.dtype).expand(*obs.shape[:-1], -1) / 1000.0], dim=-1).contiguous()
        return obs.contiguous()

    def _modify_observation(self, obs):
        return obs

    def _get_joint_pos(self):
        return self.obs_helper.get_joint_pos_from_obs(self.obs_helper._build_obs(self._data))

    def _get_joint_vel(self):
        return self.obs_helper.get_joint_vel_from_obs(self.obs_helper._build_obs(self._data))

    def get_obs_idx(self, key):
        return [i - 2 for i in self.obs_helper.obs_idx_map[key]]

    def _get_idx(self, keys):
        if type(keys) != list:
            assert type(keys) == str
            keys = [keys]
        return np.concatenate([self.obs_helper.obs_idx_map[k] for k in keys]) - 2

    def _get_from_obs(self, obs, keys):
        """:1207-1232."""
        obs = torch.as_tensor(obs)
        pad = torch.zeros(obs.shape[:-1] + (2,), dtype=obs.dtype, device=obs.device)
        obs = torch.cat([pad, obs], dim=-1)
        if type(keys) != list:
            assert type(keys) == str
            keys = [keys]
        return torch.cat([self.obs_helper.get_from_obs(obs, k) for k in keys], dim=-1)

    def get_kinematic_obs_mask(self):
        return np.arange(len(self.obs_helper.observation_spec) - 2)

    def _len_qpos_qvel(self):
        keys = self.get_all_observation_keys()
        return len([k for k in keys if k.startswith("q_")]), len([k for k in keys if k.startswith("dq_")])

    # ------------------------------------------------------------------ reward / termination
    def reward(self, state, action, next_state, absorbing):
        return self._reward_function(state, action, next_state, absorbing)

    def _get_reward_function(self, reward_type, reward_params):
        """:783-825."""
        if reward_type == "custom":
            return CustomReward(**reward_params)
        elif reward_type == "target_velocity":
            x_vel_idx = self.get_obs_idx("dq_pelvis_tx")
            assert len(x_vel_idx) == 1
            return TargetVelocityReward(x_vel_idx=x_vel_idx[0], **reward_params)
        elif reward_type == "x_pos":
            x_idx = self.get_obs_idx("q_pelvis_tx")
            assert len(x_idx) == 1
            return PosReward(pos_idx=x_idx[0])
        elif reward_type is None:
            return NoReward()
        raise NotImplementedError("The specified reward has not been implemented: %s" % reward_type)

    def _has_fallen(self, obs, return_err_msg=False):
        raise NotImplementedError

    def is_absorbing(self, obs):
        return self._has_fallen(obs) if self._use_absorbing_states else self._out(
            torch.zeros(self.n_envs, dtype=torch.bool, device=self._device))

    # ------------------------------------------------------------------ actions (N1: the step before the path)
    def _preprocess_action(self, action):
        """:1050-1069."""
        a = torch.as_tensor(action, device=self._device, dtype=torch.float32)
        single = a.dim() == 1
        a = a.unsqueeze(0) if single else a
        if getattr(self, "_action_kernel_spec", None) is None:
            self._action_kernel_spec = Kn.make_action_spec(self.norm_act_delta, self.norm_act_mean)
        ctrl = Kn.action_affine(self._action_kernel_spec, a.t().contiguous()).t()      # kernel works on [nu, n] SoA
        return ctrl[0] if single else ctrl

    def attach_dynamics(self, fn):
        """``fn(env, ctrl [n, nu]) -> (qpos [n, nq], qvel [n, nv])``: the physics between two observations
        (``mj_step`` x n_substeps in the reference).  Contact dynamics stay outside this package."""
        self._dynamics = fn

    def step(self, action):
        raise NotImplementedError

    # ------------------------------------------------------------------ dataset
    def create_dataset(self, ignore_keys=None):
        """:926-968 (the terminal-state check runs on the GPU)."""
        if self._dataset is None:
            if self.trajectories is None:
                raise ValueError("No trajectory was passed to the environment. "
                                 "To create a dataset pass a trajectory first.")
            dataset = self.trajectories.create_dataset(ignore_keys=ignore_keys)
            fallen, msg = self._has_fallen(torch.as_tensor(dataset["states"], dtype=torch.float32, device=self._device),
                                           return_err_msg=True, batched=True)
            if bool(fallen.any()):
                raise ValueError("Some of the states in the created dataset are terminal states. "
                                 "This should not happen.\n\nViolations:\n" + msg)
            self._dataset = deepcopy(dataset)
            return dataset
        return deepcopy(self._dataset)

    def load_dataset_and_get_traj_files(self, dataset_path, freq=None):
        """:970-1044 (N4: the "perfect"-dataset format): a dataset ``{states [N, D], last [N], ...}`` (npz path or
        dict) -> per-key trajectory dict for ``load_trajectory(dict(traj_files=...))``.  The two spec keys a dataset
        does not carry (root x and z) are zeros, or -- with ``freq`` -- the running integral of their velocities,
        restarted after every ``last == 1`` (vectorised: a segmented cumulative sum)."""
        dataset = np.load(str(dataset_path), allow_pickle=True) if not isinstance(dataset_path, dict) else dataset_path
        self._dataset = deepcopy({k: d for k, d in dataset.items()})
        states = np.atleast_2d(np.asarray(dataset["states"], dtype=np.float64))
        last = np.asarray(dataset["last"])
        rel_keys = [spec[0] for spec in self.obs_helper.observation_spec]
        num = len(states)
        assert states.shape[1] == len(rel_keys) - 2, "a dataset state is the observation without the first two keys"
        trajectories = dict()
        for i, key in enumerate(rel_keys):
            if i >= 2:
                trajectories[key] = states[:, i - 2]
            elif freq is None:
                trajectories[key] = np.zeros(num)
            else:
                assert num > 2
                inc = states[:-1, rel_keys.index("d" + key) - 2] / float(freq)
                start = np.flatnonzero(last[:num - 1] == 1) + 1                 # samples that restart at 0
                cs = np.concatenate([[0.0], np.cumsum(inc)])
                seg = np.zeros(num, dtype=np.int64)
                seg[start] = 1
                base = np.concatenate([[0.0], cs[start]])[np.cumsum(seg)]        # running sum at the segment start
                # sample j of a segment = sum of that segment's increments before j (the increment INTO a restart is dropped)
                trajectories[key] = cs - base
        if num > 2:
            trajectories["split_points"] = np.concatenate([[0], np.squeeze(np.argwhere(last == 1) + 1, axis=-1)])
        return trajectories

    # ------------------------------------------------------------------ playback
    def play_trajectory(self, n_episodes=None, n_steps_per_episode=None, render=False, record=False,
                        recorder_params=None):
        """:338-442: force the model to the trajectory samples step by step (per-step kernels K3 + K1)."""
        assert self.trajectories is not None
        if render or record:
            raise NotImplementedError("rendering is outside the hot path; call with render=False")
        assert n_episodes is not None and n_steps_per_episode is not None, "unbounded playback needs a viewer"
        self.reset()
        sample = self.trajectories.get_current_sample()
        self.set_sim_state(sample)
        dev = self.trajectories.device_state
        fallen_any = torch.zeros(self.n_envs, dtype=torch.bool, device=self._device)
        obs = None
        for _ in range(n_episodes):
            for _ in range(n_steps_per_episode):
                self.set_sim_state(sample)
                self.forward()
                dev.next(sample=self.trajectories._sample, auto_reset=True)          # :414-418
                sample = self.trajectories._sample.t()
                obs = self._create_observation(sample)
                fallen_any |= self._has_fallen(obs, batched=True)
            self.reset()
        return dict(obs=self._out(obs), has_fallen=self._out(fallen_any))

    def play_trajectory_from_velocity(self, n_episodes=None, n_steps_per_episode=None, render=False, record=False,
                                      recorder_params=None, **_fused_only):
        """:444-560 with per-step kernels (K3 + A7 + K1), for any model / observation spec of joint entries: the Euler step
        of the joint positions runs in float64 like the reference's.  (The default UnitreeH1 overrides this with ONE fused
        kernel per episode.)  Returns the last observation and whether any step had fallen."""
        assert self.trajectories is not None
        if render or record:
            raise NotImplementedError("rendering is outside the hot path; call with render=False")
        assert n_episodes is not None and n_steps_per_episode is not None, "unbounded playback needs a viewer"
        self.reset()                                                             # :481
        sample = self.trajectories.get_current_sample().clone()                  # :483   [n, K]
        len_qpos, len_qvel = self._len_qpos_qvel()
        curr_qpos = sample[:, :len_qpos].double()
        dev = self.trajectories.device_state
        fallen_any = torch.zeros(self.n_envs, dtype=torch.bool, device=self._device)
        obs = None
        for _ in range(n_episodes):
            for _ in range(n_steps_per_episode):
                qvel = sample[:, len_qpos:len_qpos + len_qvel].double()
                qpos = curr_qpos + self.dt * qvel                                # :515-517
                sample = sample.clone()
                sample[:, :len_qpos] = qpos.to(sample.dtype)                     # :519
                self.set_sim_state(sample)                                       # :521
                self.forward()                                                   # :525
                curr_qpos = qpos                                                 # :529 (_get_joint_pos reads it back)
                wrapped = torch.zeros(self.n_envs, dtype=torch.uint8, device=self._device)
                dev.next(sample=self.trajectories._sample, wrapped=wrapped, auto_reset=True)   # :532-537
                sample = self.trajectories._sample.t().clone()
                w = wrapped.bool()
                if bool(w.any()):
                    curr_qpos = torch.where(w[:, None], sample[:, :len_qpos].double(), curr_qpos)
                obs = self._create_observation(sample)                           # :539
                fallen_any |= self._has_fallen(obs, batched=True)                # :541
            self.reset()                                                         # :555
            curr_qpos = self._get_joint_pos().double()                           # :557
        return dict(obs=self._out(obs), has_fallen=self._out(fallen_any))

    def stop(self):
        pass

    # ------------------------------------------------------------------ interpolation hooks (:1275-1335)
    @staticmethod
    def _interpolate_map(traj, **interpolate_map_params):
        return np.array(traj)

    @staticmethod
    def _interpolate_remap(traj, **interpolate_remap_params):
        return [obs for obs in traj]

    def _get_interpolate_map_params(self):
        pass

    def _get_interpolate_remap_params(self):
        pass


class ValidTaskConf:
    """The valid (task, mode, data_type) settings of an environment (reference ``loco_env_base.py:1381-1455``): same
    constructor, ``get_all`` and ``get_all_combinations`` results.  A forbidden triple may hold ``None`` wildcards."""

    _FIELDS = ("task", "mode", "data_type")

    def __init__(self, tasks=None, modes=None, data_types=None, non_combinable=None):
        if non_combinable is not None and any(len(triple) != 3 for triple in non_combinable):
            raise AssertionError("non_combinable entries are (task, mode, data_type) triples")
        self.tasks, self.modes, self.data_types, self.non_combinable = tasks, modes, data_types, non_combinable

    def get_all(self):
        return tuple(deepcopy(x) for x in (self.tasks, self.modes, self.data_types, self.non_combinable))

    @staticmethod
    def _hits(choice, forbidden):
        return all(f is None or f == c for c, f in zip(choice, forbidden))

    def get_all_combinations(self):
        axes = [values if values is not None else [None] for values in (self.tasks, self.modes, self.data_types)]
        out = []
        for choice in product(*axes):
            conf = {k: v for k, v in zip(self._FIELDS, choice) if v is not None}
            if self.non_combinable is None:
                out.append(conf)
            else:
                # the reference appends the combination once per forbidden triple it does NOT match (so a list of several
                # triples repeats entries); every environment in the tree declares at most one triple
                out.extend(conf for forbidden in self.non_combinable if not self._hits(choice, forbidden))
        return out
