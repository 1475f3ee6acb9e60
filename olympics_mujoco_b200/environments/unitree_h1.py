"""Batched ``UnitreeH1`` environment (reference ``real_humanoid_robots/UnitreeH1.py`` and
``base_robot/base_humanoid_robot.py``): same constructor switches, observation/action specs, ``generate``,
``_has_fallen`` and ``is_absorbing``; ``step`` and ``play_trajectory_from_velocity`` run the fused CUDA kernels (the
playback and live-step kernels exist for every constructor variant built from the shipped tables).
"""
from __future__ import annotations

import warnings
from pathlib import Path

import numpy as np
import torch

from .. import kernels as Kn
from .. import mjcf, synthetic
from ..observation_helper import ObservationType
from ..utils import check_validity_task_mode_dataset
from .loco_env_base import LocoEnvBase, ValidTaskConf


class BaseHumanoidRobot(LocoEnvBase):
    """base_robot/base_humanoid_robot.py: dataset defaults, ``generate`` timing logic, ``is_absorbing``."""

    def create_dataset(self, ignore_keys=None):
        if ignore_keys is None:
            ignore_keys = ["q_pelvis_tx", "q_pelvis_tz"]                      # base_humanoid_robot.py:33-34
        return super().create_dataset(ignore_keys)

    @staticmethod
    def generate(env, path, task="walk", dataset_type="real", debug=False, clip_trajectory_to_joint_ranges=False,
                 traj_params=None, **kwargs):
        """base_humanoid_robot.py:124-234.  ``traj_params`` (extension) overrides the dataset lookup: pass
        ``dict(traj_path=...)``, ``dict(traj_files=...)`` or ``dict(table=...)``.  When the reference's dataset
        file is absent (they are not redistributable / not available offline) a synthetic dataset-shaped
        trajectory is used, with the same warning the reference gives before falling back to its mini datasets."""
        if task in ("walk", "carry"):
            mdp = env(reward_type="target_velocity", reward_params=dict(target_velocity=1.25), **kwargs)
        elif task == "run":
            mdp = env(reward_type="target_velocity", reward_params=dict(target_velocity=2.5), **kwargs)
        else:
            raise ValueError(f"unsupported task {task!r}")
        desired_contr_freq = 1 / mdp.dt
        if traj_params is None:
            if dataset_type != "real":
                raise NotImplementedError("perfect datasets need the reference's dataset files")
            traj_data_freq = 500
            full = Path(__file__).resolve().parent.parent / path
            if full.exists():
                traj_params = dict(traj_path=str(full))
            else:
                warnings.warn("Datasets not found, falling back to a synthetic dataset-shaped trajectory. Please "
                              "install the datasets to use this environment for imitation learning!")
                traj_params = dict(traj_files=synthetic.h1_walk_dataset(model=mdp._model,
                                                                         speed=1.25 if task == "walk" else 2.5))
            traj_params.update(traj_dt=1 / traj_data_freq, control_dt=1 / desired_contr_freq,
                               clip_trajectory_to_joint_ranges=clip_trajectory_to_joint_ranges)
        mdp.load_trajectory(traj_params, warn=False)
        return mdp

    def is_absorbing(self, obs):
        """base_humanoid_robot.py:246-260 (imitation-learning branch)."""
        if self._use_absorbing_states:
            return self._has_fallen(obs)
        return self._out(torch.zeros(self.n_envs, dtype=torch.bool, device=self._device))


class UnitreeH1(BaseHumanoidRobot):
    valid_task_confs = ValidTaskConf(tasks=["walk", "run", "carry"], data_types=["real", "perfect"],
                                     non_combinable=[("carry", None, "perfect")])

    def __init__(self, disable_arms=True, disable_back_joint=False, hold_weight=False, weight_mass=None, xml_path=None,
                 per_env_weight=False, **kwargs):
        """UnitreeH1.py:38-111.  ``hold_weight``: a jointless "weight" body under torso_link (arms fixed in their MJCF
        orientation); ``weight_mass=None`` builds one model per valid weight (0.1, 1, 5, 10 kg) and every reset() switches
        the env object to one of them (MultiMuJoCo).

        ``per_env_weight=True`` (extension; needs ``hold_weight`` and no fixed ``weight_mass``): every reset() draws a
        weight for EACH env, as n reference env objects would -- env ``env_id0 + e`` after the object's reset number k
        holds model ``philox_randint(seed, env_id0 + e, k, 32, 4)`` (``random_env_reset``) or ``(env_id0 + e + k + 1) mod
        4`` (round robin); env 0 of the first shard follows the shared pick.  ``model_index`` (int32 [n], into
        ``mjcf.H1_VALID_WEIGHTS``) and ``weight_body_mass`` (float32 [n], 2 x the weight in kg) hold the draw on the device
        and every kernel of the env reads the mass per env.  Trajectory wrap resets inside an episode keep the weight."""
        if per_env_weight and (not hold_weight or weight_mass is not None):
            raise ValueError("per_env_weight draws one of the valid weights per env: it needs hold_weight=True and "
                             "weight_mass=None")
        if hold_weight:
            assert disable_arms is True, ("If you want Unitree H1 to carry a weight, please disable the arms. "
                                          "They will be kept fixed.")
        action_spec = self._get_action_specification()
        observation_spec = self._get_observation_specification()
        self._hidable_obs = ("positions", "velocities", "foot_forces", "weight")
        self._disable_arms, self._disable_back_joint = disable_arms, disable_back_joint
        self._hold_weight, self._weight_mass = hold_weight, weight_mass
        self._valid_weights = list(mjcf.H1_VALID_WEIGHTS)
        joints_to_remove, motors_to_remove, _ = self._get_xml_modifications()
        obs_to_remove = ["q_" + j for j in joints_to_remove] + ["dq_" + j for j in joints_to_remove]
        observation_spec = [e for e in observation_spec if e[0] not in obs_to_remove]
        action_spec = [a for a in action_spec if a not in motors_to_remove]
        base = mjcf.compile_mjcf(xml_path, name="UnitreeH1") if xml_path is not None else None   # the user's h1.xml
        weights = [None] if not hold_weight else ([weight_mass] if weight_mass is not None else self._valid_weights)
        models = [mjcf.unitree_h1_variant(disable_arms, disable_back_joint, hold_weight, w, base=base) for w in weights]
        super().__init__(models if len(models) > 1 else models[0], action_spec, observation_spec,
                         per_env_model=per_env_weight, **kwargs)
        model = self._model
        if per_env_weight:
            self._bind_env_weights()
        js = [e[1] for e in observation_spec if e[2] == ObservationType.JOINT_POS]
        perm = [int(model.jnt_qposadr[model.jnt_names.index(j)]) for j in js]
        rf = self._reward_function
        self._spec = Kn.make_h1_spec(perm, self.get_obs_idx("dq_pelvis_tx")[0],
                                     target_velocity=getattr(rf, "_target_vel", 0.0),
                                     use_absorbing_states=kwargs.get("use_absorbing_states", True))
        self._fused_reward = hasattr(rf, "_target_vel")
        self._prev_x_vel = torch.zeros(self.n_envs, device=self._device)
        # steps since each env's last reset (mushroom Core's episode_steps); advanced by step(autoreset=True)
        self.episode_step = torch.zeros(self.n_envs, dtype=torch.int32, device=self._device)

    # ------------------------------------------------------------------ per-env carried weight
    def _bind_env_weights(self):
        """One device model for the four carry models, its weight body's mass read per env from ``weight_body_mass``.
        Before the first reset every env holds model 0, as the shared env object does."""
        if not self._dm.h1_variant:
            raise NotImplementedError("per_env_weight needs the carry models of the shipped tables (no xml_path)")
        self._weight_body = self._models[0].body_id("weight")
        self._weight_masses = [float(m.body_mass[self._weight_body]) for m in self._models]
        self.model_index = torch.zeros(self.n_envs, dtype=torch.int32, device=self._device)
        self.weight_body_mass = torch.full((self.n_envs,), self._weight_masses[0], dtype=torch.float32, device=self._device)
        # each env's number of partial resets (reset(mask=...), step(autoreset=True)): the counter of its own model draw
        self.partial_resets = torch.zeros(self.n_envs, dtype=torch.int32, device=self._device)
        Kn.bind_env_body_mass(self._dm, self._weight_body, self.weight_body_mass)

    def _draw_env_models(self, count):
        Kn.h1_draw_models(self._seed, self._env_id0, count, self._weight_masses, self.model_index, self.weight_body_mass,
                          random=self._random_env_reset)

    # ------------------------------------------------------------------ specs (UnitreeH1.py:134-160, 293-376)
    def _get_xml_modifications(self):
        joints, motors = [], []
        if self._disable_arms:
            joints += list(mjcf.H1_ARM_JOINTS)
            motors += [j + "_actuator" for j in mjcf.H1_ARM_JOINTS]
        if self._disable_back_joint:
            joints += ["back_bkz"]
            motors += ["back_bkz_actuator"]
        return joints, motors, []

    @staticmethod
    def _get_observation_specification():
        joints = synthetic.H1_SPEC_JOINTS
        return [("q_" + j, j, ObservationType.JOINT_POS) for j in joints] + \
               [("dq_" + j, j, ObservationType.JOINT_VEL) for j in joints]

    @staticmethod
    def _get_action_specification():
        order = ["back_bkz", "l_arm_shy", "l_arm_shx", "l_arm_shz", "left_elbow", "r_arm_shy", "r_arm_shx", "r_arm_shz",
                 "right_elbow", "hip_flexion_r", "hip_adduction_r", "hip_rotation_r", "knee_angle_r", "ankle_angle_r",
                 "hip_flexion_l", "hip_adduction_l", "hip_rotation_l", "knee_angle_l", "ankle_angle_l"]
        return [j + "_actuator" for j in order]

    @staticmethod
    def _get_grf_size():
        return 6

    # ------------------------------------------------------------------ termination (UnitreeH1.py:162-203)
    def _has_fallen(self, obs, return_err_msg=False, batched=False):
        obs = torch.as_tensor(obs, device=self._device, dtype=torch.float32)
        single = obs.dim() == 1
        o = obs.unsqueeze(0) if single else obs
        fallen = Kn.h1_has_fallen(o[:, :4].t().contiguous()).bool()
        res = fallen[0] if (single and not batched) else fallen
        if not return_err_msg:
            return res
        msg = ""
        if bool(fallen.any()):
            row = o[int(torch.nonzero(fallen)[0])].double().cpu().numpy()
            if row[0] < -0.3 or row[0] > 0.1:
                msg += "pelvis_y_condition violated.\n"
            elif row[1] < -np.pi / 4.5 or row[1] > np.pi / 12:
                msg += "pelvis_tilt_condition violated.\n"
            elif row[2] < -np.pi / 12 or row[2] > np.pi / 8:
                msg += "pelvis_list_condition violated.\n"
            else:
                msg += "pelvis_rotation_condition violated.\n"
        return res, msg

    # ------------------------------------------------------------------ factory (UnitreeH1.py:205-242)
    @staticmethod
    def generate(task="walk", dataset_type="real", **kwargs):
        check_validity_task_mode_dataset(UnitreeH1.__name__, task, None, dataset_type,
                                         *UnitreeH1.valid_task_confs.get_all())
        if task == "carry":
            # The reference's BaseHumanoidRobot.generate leaves `mdp` unbound for "carry" (base_humanoid_robot.py:143-150
            # handles only "walk" and "run"), although its docstring describes the task: "walking while carrying an unknown
            # weight".  That is what is built here: the walk MDP (target 1.25 m/s, the walk dataset) holding a weight.
            kwargs.setdefault("hold_weight", True)
        if dataset_type == "real":
            path = "datasets/humanoids/real/05-run_UnitreeH1.npz" if task == "run" else \
                "datasets/humanoids/real/02-constspeed_UnitreeH1.npz"
        else:                                                                   # UnitreeH1.py:226-238
            assert kwargs.get("use_foot_forces", False) is False and kwargs.get("disable_arms", True) is True
            assert kwargs.get("disable_back_joint", False) is False and kwargs.get("hold_weight", False) is False
            path = "datasets/humanoids/perfect/unitreeh1_%s/perfect_expert_dataset_det.npz" % ("run" if task == "run" else "walk")
        return BaseHumanoidRobot.generate(UnitreeH1, path, task, dataset_type, clip_trajectory_to_joint_ranges=True,
                                          **kwargs)

    # ------------------------------------------------------------------ step (mushroom MuJoCo.step, SURVEY.md A.2)
    def reset(self, obs=None, mask=None):
        """``mask=None``: reset every env (loco_env_base.py:568-604).  ``mask`` ([n] bool or uint8 tensor on the env's
        device): reset only the envs it selects, each exactly as reset() resets it, in one kernel (``om_h1_reset_envs``)
        and without a host synchronisation -- qpos = qpos0 and qvel = 0, the GRF row zeroed (use_foot_forces), the
        trajectory reset under the random_start / init_step_no rules of setup() (the om_traj_reset draw contract;
        reset_count += 1), set_sim_state of its sample, the observation of that state, prev_x_vel and episode_step = 0.
        Every state tensor of the other envs stays as it was; the FK mirrors (data.xpos, ...) are not written, as reset()
        leaves them.  Returns the full [n, D] observation: the new rows of the reset envs, the current ones of the others.

        Model switch of a masked reset: with ``per_env_weight`` env e draws its own model at its own partial resets --
        ``philox_randint(seed, env_id0 + e, j, 33, 4)`` with j = ``partial_resets[e]`` (then incremented), or
        ``(model_index[e] + 1) mod 4`` in round robin; the full reset() keeps its own contract (stream 32, the object's
        reset count).  With a shared MultiMuJoCo (a carried weight of every valid mass without ``per_env_weight``) all envs
        hold the object's one model, so only a reset of the whole object switches it: a masked reset neither switches the
        model nor advances the object's reset count.  ``mask`` together with ``obs`` raises ValueError."""
        if mask is None:
            out = super().reset(obs)
            self._prev_x_vel.copy_(self._obs[:, self._spec.x_vel_idx])
            self.episode_step.zero_()
            self._play_state = None
            return out
        if obs is not None:
            raise ValueError("reset(obs=..., mask=...) is not supported: a masked reset draws from the trajectory")
        if not torch.is_tensor(mask) or mask.dtype not in (torch.bool, torch.uint8) or tuple(mask.shape) != (self.n_envs,) \
                or mask.device.type != torch.device(self._device).type:
            raise ValueError(f"mask must be a [{self.n_envs}] bool or uint8 tensor on the env's device")
        cur = self._obs
        if cur is None:                              # never reset: the other envs keep the observation of their state
            cur = self._create_observation(self.obs_helper._build_obs(self._data))
        obs_in = cur.t().contiguous()
        new = torch.empty_like(obs_in)
        self._reset_envs(mask=mask, obs_in=obs_in, obs=new)
        self._obs = new.t()
        self._play_state = None
        return self._out(self._modify_observation(self._obs))

    def _reset_envs(self, obs_in, obs, mask=None, absorbing=None):
        """om_h1_reset_envs with this env's state: the envs of ``mask``, or (mask=None) the auto-reset after a step."""
        if self.trajectories is None:
            raise ValueError("a per-env reset draws from the trajectory: load one first")
        if self._init_step_no is not None and self._random_start:
            raise ValueError("Either use a random start or set an initial step, not both.")
        forced_traj, forced_step = -1, -1                                # setup() :640-657
        if not self._random_start:
            if self._init_step_no:
                traj_len = self.trajectories.trajectory_length
                assert self._init_step_no <= traj_len * self.trajectories.number_of_trajectories
                forced_traj, forced_step = int(self._init_step_no / traj_len), int(self._init_step_no % traj_len)
            else:
                forced_step = 0
        d = self._data
        draw = {}
        if self._per_env_model:
            draw = dict(partial_resets=self.partial_resets, model_index=self.model_index, mass=self.weight_body_mass,
                        masses=self._weight_masses, random=self._random_env_reset)
        last = None if mask is not None else torch.empty(self.n_envs, dtype=torch.uint8, device=self._device)
        Kn.h1_reset_envs(self._dm, self._spec, self.trajectories.device_state, d.qpos, d.qvel, mask=mask, absorbing=absorbing,
                         horizon=self.info.horizon, forced_traj=forced_traj, forced_step=forced_step, obs_in=obs_in, obs=obs,
                         prev_x_vel=self._prev_x_vel, episode_step=self.episode_step, last=last, grf=self._grf, **draw)
        return last

    def attach_dynamics(self, fn, soa=False):
        """``soa=True``: ``fn(env, ctrl [nu, n]) -> (qpos [nq, n], qvel [nv, n])`` float32 CUDA tensors in the kernels' own
        layout (component-major, env index contiguous) -- ``step`` then runs without a single transposing copy."""
        super().attach_dynamics(fn)
        self._dynamics_soa = bool(soa)

    def _take_dynamics(self, res):
        """(qpos, qvel) or (qpos, qvel, ground_forces [n, 6]): the third value is what the contact solver measured
        (``_get_ground_forces``, UnitreeH1.py:113-121) and feeds the GRF part of the observation."""
        if len(res) == 3:
            self.set_ground_forces(res[2])
            return res[0], res[1]
        return res

    def step(self, action, autoreset=False):
        """action [n, nu] in [-1, 1] ([nu, n] with SoA dynamics) -> (obs, reward, absorbing, info).  The physics between
        observations comes from the attached dynamics; everything after it is one fused kernel (K1 + K2).

        ``autoreset=True`` adds mushroom_rl Core's bookkeeping on the device, in one more kernel on the same stream and
        without a host synchronisation: ``episode_step += 1``, ``last = absorbing | (episode_step >= info.horizon)``, and
        every env with ``last`` set gets the masked reset of ``reset(mask=last)``.  ``obs`` is then the observation after
        those resets (the input to the next action); ``reward`` and ``absorbing`` are the step's own; ``info["last"]`` ([n]
        bool) and ``info["final_obs"]`` -- the step's own observation of EVERY env, the ``next_state`` of the transition
        (with use_foot_forces it carries the step's GRF / 1000, the reset rows of ``obs`` zeros)."""
        if self._dynamics is None:
            raise RuntimeError("step() needs a dynamics backend: env.attach_dynamics(fn).  Contact dynamics "
                               "(mj_step) are outside this package's hot path.")
        d = self._data
        if getattr(self, "_dynamics_soa", False):
            if getattr(self, "_action_kernel_spec", None) is None:
                self._action_kernel_spec = Kn.make_action_spec(self.norm_act_delta, self.norm_act_mean)
            ctrl = Kn.action_affine(self._action_kernel_spec, action)               # [nu, n], no transposes
            qpos, qvel = self._take_dynamics(self._dynamics(self, ctrl))
            assert qpos.shape == d.qpos.shape and qvel.shape == d.qvel.shape, "SoA dynamics return [nq, n], [nv, n]"
            if qpos is not d.qpos:                            # a dynamics that writes env.data.qpos / qvel in place and
                d.qpos.copy_(qpos)                            # returns them costs no copy at all
            if qvel is not d.qvel:
                d.qvel.copy_(qvel)
            qpos, qvel = d.qpos, d.qvel
        else:
            ctrl = self._preprocess_action(self._batched(action))
            qpos, qvel = self._take_dynamics(self._dynamics(self, ctrl))
            d.qpos.copy_(torch.as_tensor(qpos, device=self._device, dtype=torch.float32).reshape(self.n_envs, -1).t())
            d.qvel.copy_(torch.as_tensor(qvel, device=self._device, dtype=torch.float32).reshape(self.n_envs, -1).t())
            qpos, qvel = d.qpos, d.qvel
        prev_obs = self._obs
        if autoreset:
            return self._step_autoreset(prev_obs, ctrl, qpos, qvel)
        out = Kn.h1_step(self._dm, self._spec, qpos, qvel, self._prev_x_vel,
                         out=dict(xpos=d.xpos, xquat=d.xquat, site_xpos=d.site_xpos, cvel=d.cvel))
        cur_obs = out["obs"].t()
        if self._use_foot_forces:                                # _create_observation :737-767: append mean_grf / 1000
            cur_obs = torch.cat([cur_obs, self._grf.t() / 1000.0], dim=1)
        absorbing = out["absorbing"].bool()
        reward = out["reward"] if self._fused_reward else self.reward(prev_obs, ctrl, cur_obs, absorbing)
        self._obs = cur_obs
        self._prev_x_vel.copy_(out["obs"][self._spec.x_vel_idx])
        return self._out(self._modify_observation(cur_obs)), self._out(reward), self._out(absorbing), {}

    def _step_autoreset(self, prev_obs, ctrl, qpos, qvel):
        """step(autoreset=True) after the dynamics: the step kernel writes the step's observation (the transition's
        final_obs, [D, n] SoA with the GRF rows appended), then om_h1_reset_envs in auto-reset mode writes the returned
        observation, last, episode_step and prev_x_vel and resets the envs whose episode ended."""
        d = self._data
        nobs = 2 * self._spec.n_obs_q - 2
        final = torch.empty((nobs + (0 if self._grf is None else self._grf.shape[0]), self.n_envs), device=self._device)
        out = Kn.h1_step(self._dm, self._spec, qpos, qvel, self._prev_x_vel,
                         out=dict(xpos=d.xpos, xquat=d.xquat, site_xpos=d.site_xpos, cvel=d.cvel, obs=final[:nobs]))
        if self._grf is not None:                                  # _create_observation: append mean_grf / 1000
            torch.div(self._grf, 1000.0, out=final[nobs:])
        final_obs = final.t()
        absorbing = out["absorbing"].view(torch.bool)                # 0 / 1 bytes: a view, no copy
        reward = out["reward"] if self._fused_reward else self.reward(prev_obs, ctrl, final_obs, absorbing)
        new = torch.empty_like(final)
        last = self._reset_envs(obs_in=final, obs=new, absorbing=out["absorbing"])
        self._obs = new.t()
        self._play_state = None
        info = dict(last=self._out(last.view(torch.bool)), final_obs=self._out(self._modify_observation(final_obs)))
        return self._out(self._modify_observation(self._obs)), self._out(reward), self._out(absorbing), info

    # ------------------------------------------------------------------ fused live step / graph
    def _has_fused_kernels(self):
        """Every model of this env (one per carried weight with MultiMuJoCo) has generated playback / live-step kernels."""
        return all(dm.h1_variant for dm in self._dms)

    def _live_stepper(self):
        if not self._has_fused_kernels() or not self._fused_reward or self._use_foot_forces:
            raise NotImplementedError("the fused live step is generated for the UnitreeH1 models of the shipped tables with "
                                      "the target-velocity reward")
        if getattr(self, "_live", None) is None:
            if self._obs is None:
                self.reset()
            d = self._data
            self._live = Kn.H1LiveStep(self._dm, self._spec, self.trajectories.device_state, self._prev_x_vel,
                                       out=dict(qpos=d.qpos, qvel=d.qvel, xpos=d.xpos, xquat=d.xquat, site_xpos=d.site_xpos,
                                                cvel=d.cvel))
        return self._live

    def step_trajectory(self):
        """One env step driven by the loaded trajectory instead of physics -- what ``play_trajectory`` does per step
        (loco_env_base.py:404-422): next sample (wrap -> reset), ``set_sim_state``, the forward pass, observation,
        ``has_fallen``, reward on the previous observation -- as ONE kernel and one C call (``om_h1_live_step``).
        Returns ``(obs, reward, absorbing, info)`` like ``step``; the tensors are views of buffers that the next call
        overwrites."""
        live = self._live_stepper()
        out = live()
        self._obs = out["obs"].t()
        return (self._out(self._modify_observation(self._obs)), self._out(out["reward"]), self._out(out["absorbing"].bool()),
                {})

    def step_graph(self, n_steps, want=("obs", "reward", "absorbing")):
        """Capture ``n_steps`` consecutive fused live steps into ONE CUDA graph.  Returns ``(replay, buffers)``: every
        ``replay()`` advances all envs by ``n_steps`` and fills the time-major buffers ``[n_steps, C, n]`` (``want`` may
        also name xpos, xquat, site_xpos, cvel, wrapped).  A launch-bound inner loop belongs in a graph: at 131 072 envs a
        replayed step costs what the kernel costs."""
        live = self._live_stepper()
        n, dev = self.n_envs, self._device
        bufs = {}
        for k in want:
            c, dt_ = live.keys[k]
            bufs[k] = torch.empty((n_steps, n) if c is None else (n_steps, c, n), dtype=dt_, device=dev)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        base = dict(live.out)
        graph = torch.cuda.CUDAGraph()
        tr = self.trajectories.device_state
        carried = [tr.traj_no, tr.step_no, tr.reset_count, tr.xy_off, self._prev_x_vel]
        with torch.cuda.stream(side):
            saved = [t.clone() for t in carried]
            live.rebind(out={k: v[0] for k, v in bufs.items()}, stream=side.cuda_stream)()      # warm-up outside the capture
            for t, s0 in zip(carried, saved):                                                   # ... that leaves no trace
                t.copy_(s0)
            side.synchronize()
            with torch.cuda.graph(graph, stream=side):
                for t in range(n_steps):
                    live.rebind(out={k: v[t] for k, v in bufs.items()}, stream=torch.cuda.current_stream().cuda_stream)()
        torch.cuda.current_stream().wait_stream(side)
        live.out = base
        live.rebind()

        def replay():
            graph.replay()
            self._obs = bufs["obs"][-1].t() if "obs" in bufs else self._obs
            return bufs
        return replay, bufs

    # ------------------------------------------------------------------ fused playback (loco_env_base.py:444-560)
    def set_sim_state(self, sample):
        """loco_env_base.py:659-684 as one kernel (the spec is joint positions then joint velocities)."""
        sample = self._batched(sample).to(torch.float32)
        if sample.shape[-1] != 2 * self._spec.n_obs_q:
            return super().set_sim_state(sample)
        Kn.set_sim_state(self._dm, self._spec, sample.t().contiguous(), self._data.qpos, self._data.qvel)

    def make_rollout_buffers(self, n_steps, want=("xpos", "xquat", "site_xpos", "cvel", "obs", "reward", "fallen",
                                                  "traj_no_t", "step_no_t")):
        m, n, dev = self._model, self.n_envs, self._device
        spec = dict(xpos=(m.nbody * 3, torch.float32), xquat=(m.nbody * 4, torch.float32),
                    site_xpos=(m.nsite * 3, torch.float32), cvel=(m.nbody * 6, torch.float32),
                    obs=(2 * self._spec.n_obs_q - 2, torch.float32),
                    reward=(None, torch.float32), fallen=(None, torch.uint8), traj_no_t=(None, torch.int32),
                    step_no_t=(None, torch.int32))
        return {k: torch.empty((n_steps, n) if spec[k][0] is None else (n_steps, spec[k][0], n), dtype=spec[k][1],
                               device=dev) for k in want}

    def _play(self, forced, n_episodes, n_steps_per_episode, render, record, out, want, continue_episode, obs_moments):
        """Both playback calls: every call of the reference begins with ``reset()`` (:377 / :481) and ends every episode
        with one (:432 / :555).  The first call resets through the Python API (it also allocates the carried state);
        later calls perform the same reset INSIDE the first kernel of the call.  ``continue_episode=True`` (extension)
        skips the reset at the start and carries the state of the previous call on.

        With MultiMuJoCo (a carried weight of every valid mass) each reset() performed inside a kernel switches the model on
        the host exactly as reset() does, so each episode runs on the model the preceding reset chose.  A variant model
        called with none of ``out`` / ``want`` / ``obs_moments`` returns what the base class returns, ``dict(obs=[n, nobs]
        last observation, has_fallen=[n])``, from the kernel's carried sample and its per-step fallen flags."""
        assert self.trajectories is not None
        if render or record:
            raise NotImplementedError("rendering is outside the hot path; call with render=False")
        assert n_episodes is not None and n_steps_per_episode is not None, "unbounded playback needs a viewer"
        dev = self.trajectories.device_state
        start_reset = not continue_episode
        if self._play_state is None:
            self.reset()                                                             # :377 / :481
            sample = self.trajectories.get_current_sample().t().contiguous()         # :379 / :483
            self._play_state = dict(curr_qpos=sample[:self._spec.n_obs_q].double().contiguous(), pending=sample.clone(),
                                    prev_x_vel=self._prev_x_vel)
            start_reset = False
        res = None
        summary = not self._dm.specialised and out is None and want is None and obs_moments is None
        kw = dict(want=("fallen",)) if summary else ({} if want is None else dict(want=want))
        fallen_any = torch.zeros(self.n_envs, dtype=torch.bool, device=self._device) if summary else None
        for ep in range(n_episodes):
            if start_reset and ep == 0:
                self._next_model()                                                   # the in-kernel reset() at :377 / :481
            res = Kn.h1_play_from_velocity(self._dm, self._spec, dev, self._play_state, n_steps_per_episode, dt=self.dt,
                                           end_episode_reset=True, out=out, forced=forced, obs_moments=obs_moments,
                                           start_reset=start_reset and ep == 0, **kw)
            if summary:
                fallen_any |= res["fallen"].any(dim=0).bool()
            self._next_model()                                                       # the in-kernel reset() at :432 / :555
        # the env is left in the state of the final reset() (:432 / :555): its observation is that sample's, fetched on
        # first use (the loop's `sample` variable -- our `pending` -- stays the stale one, as in the reference)
        self.__dict__["_obs_lazy"] = lambda: self._create_observation(self.trajectories.get_current_sample())
        if summary:
            obs = self._play_state["pending"][2:].t().clone() if n_episodes and n_steps_per_episode else None
            return dict(obs=None if obs is None else self._out(obs), has_fallen=self._out(fallen_any))
        return res

    def play_trajectory(self, n_episodes=None, n_steps_per_episode=None, render=False, record=False, recorder_params=None,
                        out=None, want=None, continue_episode=False, obs_moments=None):
        """loco_env_base.py:338-442 as one fused kernel per episode (``om_h1_play_trajectory``): the model is forced to
        every trajectory sample, FK runs on it, the next sample gives the observation and the has_fallen flag.
        Returns the last episode's time-major rollout buffers (the reference only renders); see ``_play`` for the other
        variants' return value."""
        if not self._has_fused_kernels() or (self._use_foot_forces and not self._dm.specialised):
            return super().play_trajectory(n_episodes, n_steps_per_episode, render, record, recorder_params)
        return self._play(True, n_episodes, n_steps_per_episode, render, record, out, want, continue_episode, obs_moments)

    def play_trajectory_from_velocity(self, n_episodes=None, n_steps_per_episode=None, render=False, record=False,
                                      recorder_params=None, out=None, want=None, continue_episode=False, obs_moments=None):
        """Replays the loaded trajectory by integrating its joint velocities (reference semantics -- a ``reset()`` at the
        start of EVERY call and after every episode -- one fused kernel per episode).  Returns the last episode's
        time-major rollout buffers ([T, C, n] SoA; use ``kernels.env_major`` for [T, n, ...] views) -- the reference
        returns nothing and only renders.  ``obs_moments``: float64 [65] buffer that receives the moment sums of the
        emitted observations (S1 fused into the kernel); ``2 nobs + 1`` values for a model with nobs observations.  See
        ``_play`` for the return value of the other variants."""
        if not self._has_fused_kernels() or self._use_foot_forces:
            # a model without generated kernels (user XML, an unlisted weight) or foot forces: per-step kernels of the base class
            return super().play_trajectory_from_velocity(n_episodes, n_steps_per_episode, render, record, recorder_params)
        return self._play(False, n_episodes, n_steps_per_episode, render, record, out, want, continue_episode, obs_moments)
