"""Cost of the on-device auto-reset of the StickFigureA3 step (``step(autoreset=True)``: ``om_a3_autoreset`` after the
one-step ``om_a3_task_step``).  For each env count, on CUDA-graph replays of 10 consecutive steps:
  * the one-step A3 kernel alone (``a3_task_kernel``, observation / terms / reward / done written);
  * step + auto-reset, with ``done`` forced (contact flag bit 2) on 1/L of the envs per step, L in ``--rates``;
  * the auto-reset kernel alone on the same ``done`` pattern.
Each kernel's algorithmic bytes (below) over its time, divided by the HBM copy bandwidth measured on this card
(6454.6 GB/s, DESIGN.md section 3), give its share of HBM.  Prints one JSON line with the card's name and power limit read
in the same run; ``--out`` also writes it to a file.

    python tools/bench_a3_autoreset.py [--envs 16384,262144,1048576] [--rates 1,50,400] [--steps 10] [--reps 20] [--out F]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

HBM_GBPS = 6454.6          # measured copy bandwidth of a B200 (DESIGN.md section 3)
NQ, NV, NOBS, NINT, NSEQ = 25, 24, 41, 7, 80


def step_bytes(n):
    """The one-step kernel per env: qpos / qvel / contact in (4 (25 + 24 + 4)), task ints in (28) and out (20), the two
    targets' rows (32), obs / terms / reward out (4 (41 + 6 + 1)) and done (1) = 485 B."""
    return n * (4 * (NQ + NV + 4) + 4 * NINT + 4 * 5 + 32 + 4 * (NOBS + 6 + 1) + 1)


def reset_bytes(n, rate):
    """The auto-reset kernel: every env reads done (1) and traj_len (4) and writes traj_len (4), last (1) and path_end (1);
    an env that goes on copies its step observation (4 * 41 in and out); each of the n / L envs that resets reads and writes
    reset_count (8) and writes qpos / qvel (4 * 49), the task ints (28), the footstep plan (4 * 80) and its observation
    (4 * 41).  The task's constants (nominal pose, phase table) are a few hundred bytes, read from L2."""
    resets = n / rate
    return n * 11 + (n - resets) * 8 * NOBS + resets * (8 + 4 * (NQ + NV) + 4 * NINT + 4 * NSEQ + 4 * NOBS)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def measure(n, rates, steps, reps):
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    from olympics_mujoco_b200 import mjcf
    from olympics_mujoco_b200.tasks.phase_clock import phase_clock_lut
    from oracle import a3 as OA
    task = Kn.A3Task(Kn.DeviceModel(mjcf.load_builtin("stick_figure_a3")), n, phase_clock_lut(), OA.init_qpos(), seed=5)
    dev = "cuda"
    qpos, qvel = torch.empty((NQ, n), device=dev), torch.empty((NV, n), device=dev)
    new = torch.empty((NOBS, n), device=dev)
    task.reset(qpos, qvel, iteration_count=5000.0, obs=new)
    out = dict(obs=torch.empty((NOBS, n), device=dev), terms=torch.empty((6, n), device=dev),
               reward=torch.empty(n, device=dev), done=torch.zeros(n, dtype=torch.uint8, device=dev))
    tl = torch.zeros(n, dtype=torch.int32, device=dev)
    last, pe = torch.empty(n, dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.uint8, device=dev)
    env = torch.arange(n, device=dev)
    # per step s of a graph: its own contact record (flags bit 2 on the envs with (e + s) % L == 0) and done pattern
    con = torch.empty((steps, 4, n), device=dev)
    done = torch.empty((steps, n), dtype=torch.uint8, device=dev)

    def pattern(rate):
        for s in range(steps):
            bad = ((env + s) % rate == 0)
            con[s, 0].fill_(150.0)
            con[s, 1].fill_(250.0)
            con[s, 2].fill_(0.002)
            con[s, 3] = 1.0 + 2.0 * bad.float()
            done[s] = bad.to(torch.uint8)

    def step_only(s):
        task.step(qpos, qvel, con[s], out=out)

    def reset_only(s):
        task.autoreset(qpos, qvel, done[s], tl, out["obs"], new, last, pe, iteration_count=5000.0)

    def graph(body):
        for s in range(steps):                                   # warm-up (module load) outside the capture
            body(s)
        torch.cuda.synchronize()
        g, side = torch.cuda.CUDAGraph(), torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.cuda.graph(g, stream=side):
            for s in range(steps):
                body(s)
        torch.cuda.current_stream().wait_stream(side)
        return g

    def time_us(g):
        g.replay()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(reps):
            g.replay()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) * 1e3 / (reps * steps)

    pattern(rates[0])
    g_step = graph(step_only)
    base = time_us(g_step)
    sb = step_bytes(n)
    res = dict(envs=n, step_us=round(base, 2), step_bytes=int(sb), step_frac_hbm=round(sb / base / 1e3 / HBM_GBPS, 3),
               rates=[])
    for rate in rates:
        pattern(rate)
        g_both = graph(lambda s: (step_only(s), reset_only(s)))
        g_reset = graph(reset_only)
        both, alone, base = time_us(g_both), time_us(g_reset), time_us(g_step)
        rb = reset_bytes(n, rate)
        res["rates"].append(dict(L=rate, resets_per_step=round(n / rate, 1), step_us=round(base, 2),
                                 step_plus_reset_us=round(both, 2), added_us=round(both - base, 2),
                                 reset_kernel_us=round(alone, 2), reset_bytes=int(rb), reset_gbps=round(rb / alone / 1e3, 1),
                                 reset_frac_hbm=round(rb / alone / 1e3 / HBM_GBPS, 3)))
    return res


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--envs", default="16384,262144,1048576")
    ap.add_argument("--rates", default="1,50,400", help="forced done rate 1/L per step, L in this list")
    ap.add_argument("--steps", type=int, default=10, help="consecutive steps per captured graph")
    ap.add_argument("--reps", type=int, default=20, help="timed graph replays")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args(argv)
    envs = [int(x) for x in a.envs.split(",")]
    rates = [int(x) for x in a.rates.split(",")]
    if a.steps < 1 or a.reps < 1 or min(envs) < 1 or min(rates) < 1:
        ap.error("--envs, --rates, --steps and --reps must be positive")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_a3_autoreset: no CUDA device -- the timings exist only on the GPU")
    name, pl = card()
    out = dict(tool="bench_a3_autoreset", card=name, power_limit=pl, hbm_gbps=HBM_GBPS,
               note="frac_hbm: algorithmic bytes of one kernel over its time (CUDA events on graph replays); at 16384 envs "
                    "the working set stays in the 126 MB L2 between replays",
               results=[measure(n, rates, a.steps, a.reps) for n in envs])
    line = json.dumps(out)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
