"""Cost of the on-device auto-reset of the UnitreeH1 step (``step(autoreset=True)``: ``om_h1_reset_envs`` after
``om_h1_step``).  For each env count, on CUDA-graph replays of consecutive steps:
  * ``h1_step`` alone (FK outputs written, as ``UnitreeH1.step`` does);
  * ``h1_step`` + the auto-reset kernel, with ``episode_step`` staggered so that 1/H of the envs reset per step, H in
    ``--horizons``;
  * the auto-reset kernel alone (same staggering), whose algorithmic bytes over its time give its share of the HBM
    bandwidth measured on this card (6454.6 GB/s, DESIGN.md section 3).
Prints one JSON line, with the card's name and power limit read in the same run.

    python tools/bench_h1_autoreset.py [--envs 131072,1048576] [--horizons 1000,50,1] [--steps 10] [--reps 20]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

HBM_GBPS = 6454.6          # measured copy bandwidth of a B200 (DESIGN.md section 3)
NQ, K, D = 17, 34, 32      # the default UnitreeH1 model: observation-spec joints, trajectory keys, observation width


def algorithmic_bytes(n, horizon):
    """Bytes the auto-reset kernel must move per call: every env reads absorbing (1), episode_step (4) and its final
    observation (4 D) and writes the returned observation (4 D), last (1), episode_step (4) and prev_x_vel (4); each of the
    n / H envs that resets also reads its table row (4 K), writes qpos / qvel (8 NQ) and its trajectory state (20).  This
    configuration has no GRF rows and no per-env model draw (24 + 8 more bytes per reset env when it has)."""
    per_env = 1 + 4 + 4 * D + 4 * D + 1 + 4 + 4
    per_reset = 4 * K + 8 * NQ + 20
    return n * per_env + (n / horizon) * per_reset


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def measure(n, horizons, steps, reps):
    import numpy as np
    import torch
    import bench
    from olympics_mujoco_b200 import kernels as Kn
    from olympics_mujoco_b200.build import H1_SPEC_JOINTS
    model, table = bench.build_table()
    dm = Kn.DeviceModel(model)
    perm = [int(model.jnt_qposadr[model.jnt_names.index(j)]) for j in H1_SPEC_JOINTS]
    spec = Kn.make_h1_spec(perm, NQ - 2, use_absorbing_states=False)      # only the horizon ends an episode
    traj = Kn.DeviceTrajectory(table, n, seed=5)
    sample = traj.reset()
    qpos, qvel = torch.empty((NQ, n), device="cuda"), torch.empty((NQ, n), device="cuda")
    Kn.set_sim_state(dm, spec, sample, qpos, qvel)
    pxv = sample[NQ].clone()
    es = torch.zeros(n, dtype=torch.int32, device="cuda")
    out = dict(obs=torch.empty((D, n), device="cuda"), reward=torch.empty(n, device="cuda"),
               absorbing=torch.zeros(n, dtype=torch.uint8, device="cuda"))
    out = Kn.h1_step(dm, spec, qpos, qvel, pxv, want_fk=True, out=out)
    new, last = torch.empty((D, n), device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda")

    def step_only():
        Kn.h1_step(dm, spec, qpos, qvel, pxv, want_fk=True, out=out)

    def reset(h):
        Kn.h1_reset_envs(dm, spec, traj, qpos, qvel, absorbing=out["absorbing"], horizon=h, obs_in=out["obs"], obs=new,
                         prev_x_vel=pxv, episode_step=es, last=last)

    def graph(body):
        body()                                             # warm-up (module load) outside the capture
        torch.cuda.synchronize()
        g, side = torch.cuda.CUDAGraph(), torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.cuda.graph(g, stream=side):
            for _ in range(steps):
                body()
        torch.cuda.current_stream().wait_stream(side)
        return g

    def time_us(g, stagger=None):
        if stagger is not None:
            es.copy_(torch.arange(n, device="cuda", dtype=torch.int32) % stagger)
        g.replay()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(reps):
            g.replay()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) * 1e3 / (reps * steps)

    g_step = graph(step_only)
    res = dict(envs=n, step_us=round(time_us(g_step), 2), horizons=[])
    for h in horizons:
        g_both = graph(lambda: (step_only(), reset(h)))
        g_reset = graph(lambda: reset(h))
        # stagger so that 1/H of the envs reach the horizon at every step (H = 1: every env, every step)
        both, alone = time_us(g_both, h), time_us(g_reset, h)
        base = time_us(g_step)
        nbytes = algorithmic_bytes(n, h)
        res["horizons"].append(dict(H=h, step_plus_reset_us=round(both, 2), step_us=round(base, 2),
                                    added_us=round(both - base, 2), reset_kernel_us=round(alone, 2),
                                    reset_bytes=int(nbytes), reset_gbps=round(nbytes / alone / 1e3, 1),
                                    reset_frac_hbm=round(nbytes / alone / 1e3 / HBM_GBPS, 3),
                                    resets_per_step=float(np.round(n / h, 1))))
    return res


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--envs", default="131072,1048576")
    ap.add_argument("--horizons", default="1000,50,1")
    ap.add_argument("--steps", type=int, default=10, help="consecutive steps per captured graph")
    ap.add_argument("--reps", type=int, default=20, help="timed graph replays")
    a = ap.parse_args(argv)
    envs = [int(x) for x in a.envs.split(",")]
    horizons = [int(x) for x in a.horizons.split(",")]
    if a.steps < 1 or a.reps < 1 or min(envs) < 1 or min(horizons) < 1:
        ap.error("--envs, --horizons, --steps and --reps must be positive")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_h1_autoreset: no CUDA device -- the timings exist only on the GPU")
    name, pl = card()
    out = dict(tool="bench_h1_autoreset", card=name, power_limit=pl, hbm_gbps=HBM_GBPS,
               note="reset_frac_hbm: algorithmic bytes of the auto-reset kernel alone over its time; at 131072 envs its "
                    "~35 MB stay in the 126 MB L2 between graph replays",
               results=[measure(n, horizons, a.steps, a.reps) for n in envs])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
