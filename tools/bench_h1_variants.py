"""Timing of the fused playback and live step of every UnitreeH1 variant, with the default model measured in the same
process, alternating: fused play_trajectory_from_velocity at 4096 envs x 500 steps with the configs[1] result set (FK, obs,
reward, fallen, trajectory state), one call of the base class's per-step path at the same size, and step_graph replay time
per step at 131 072 envs.  One JSON line (measurement aid).

``carry_per_env`` is the carry task with a weight drawn per env (``per_env_weight=True``: every env of the batch carries its
own of the four weights, the kernels read its mass at run time); it alternates with the fixed 1 kg carry kernels
(``carry_1``) like every other row.  Its call time includes the two model draws of the call (start and end reset).

Algorithmic bytes per env-step, from shapes: 2 NQ * 4 sample in + nbody * 13 * 4 FK out (xpos, xquat, cvel) + nsite * 12
+ (2 NQ - 2) * 4 obs + 13 (reward, fallen, traj_no, step_no) + 2 NQ * 4 (the carried / reset sample)."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
WANT = ("xpos", "xquat", "site_xpos", "cvel", "obs", "reward", "fallen", "traj_no_t", "step_no_t")
VARIANTS = dict(default={}, noback=dict(disable_back_joint=True), arms=dict(disable_arms=False),
                arms_noback=dict(disable_arms=False, disable_back_joint=True),
                carry_0p1=dict(hold_weight=True, weight_mass=0.1), carry_1=dict(hold_weight=True, weight_mass=1.0),
                carry_5=dict(hold_weight=True, weight_mass=5.0), carry_10=dict(hold_weight=True, weight_mass=10.0),
                carry_per_env=dict(hold_weight=True, per_env_weight=True))


def bytes_per_env_step(m):
    nq = m.nq
    return 2 * nq * 4 + m.nbody * 13 * 4 + m.nsite * 12 + (2 * nq - 2) * 4 + 13 + 2 * nq * 4


def make_env(kw, n):
    import olympics_mujoco_b200 as om
    from olympics_mujoco_b200 import mjcf, synthetic
    model = mjcf.unitree_h1_variant(**{k: v for k, v in kw.items() if k != "per_env_weight"},
                                    **({"weight_mass": 1.0} if kw.get("per_env_weight") else {}))
    data = synthetic.h1_walk_dataset(n_traj=4, t_raw=2500, seed=1, model=model)
    return om.LocoEnvBase.make("UnitreeH1.walk.real", n_envs=n, seed=3, **kw,
                               traj_params=dict(traj_files=data, traj_dt=1 / 500, control_dt=0.01))


def time_calls(fn, calls):
    fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(calls):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / calls


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name()


def measure(envs=4096, steps=500, calls=20, rounds=3, graph_envs=131072, graph_steps=16):
    from olympics_mujoco_b200.environments.loco_env_base import LocoEnvBase as Base
    peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()) if (ROOT / "MEASURED_PEAKS.json").exists() else {"hbm_gbs": 6650.0}
    envs_by = {k: make_env(kw, envs) for k, kw in VARIANTS.items()}
    bufs = {k: e.make_rollout_buffers(steps, want=WANT) for k, e in envs_by.items()}
    play = {k: (lambda e=e, b=bufs[k]: e.play_trajectory_from_velocity(1, steps, out=b, want=WANT)) for k, e in envs_by.items()}
    ms = {k: [] for k in VARIANTS}
    for _ in range(rounds):                                   # alternate the models so that drift hits all alike
        for k in VARIANTS:
            ms[k].append(time_calls(play[k], calls))
    res = {}
    for k, e in envs_by.items():
        b = bytes_per_env_step(e._model)
        best = min(ms[k])
        ach = b * envs * steps / (best * 1e-3) / 1e9
        base_env = make_env(VARIANTS[k], envs)
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        Base.play_trajectory_from_velocity(base_env, 1, steps)
        t1.record()
        torch.cuda.synchronize()
        base_ms = t0.elapsed_time(t1)
        del base_env
        g = make_env(VARIANTS[k], graph_envs)
        g.reset()
        replay, _ = g.step_graph(graph_steps, want=("obs", "reward", "absorbing", "xpos", "xquat", "site_xpos", "cvel"))
        graph_ms = time_calls(replay, 10) / graph_steps
        del g, replay
        torch.cuda.empty_cache()
        res[k] = dict(nq=e._model.nq, nbody=e._model.nbody, play_ms=best, play_ms_all=ms[k], bytes_per_env_step=b,
                      achieved_gbs=ach, frac=ach / peaks["hbm_gbs"], base_class_ms=base_ms, speedup=base_ms / best,
                      step_graph_ms_per_step=graph_ms)
    return {"workload": f"UnitreeH1 variants: fused play_trajectory_from_velocity {envs} envs x {steps} steps (configs[1] "
                        f"result set), step_graph at {graph_envs} envs", "gpu": gpu_info(), "peak_hbm_gbs": peaks["hbm_gbs"],
            "timing": f"CUDA events, best of {rounds} alternating rounds of {calls} calls after warm-up", "variants": res}


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--graph-envs", type=int, default=131072)
    a = ap.parse_args()
    print(json.dumps(measure(a.envs, a.steps, a.calls, graph_envs=a.graph_envs)))
