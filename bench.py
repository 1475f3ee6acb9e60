"""Headline benchmark: env-steps/sec of the H1 hot path (FK + obs + reward + GAE), BASELINE.json configs[1].

One "step" = one pass of the hot path over one batch: a 4096-env x 500-step
``play_trajectory_from_velocity`` rollout per GPU (Euler step, set_sim_state, FK, next sample / wrap reset,
observation, has_fallen, TargetVelocityReward) followed by GAE(lambda) + advantage normalisation over the
[500, 4096] rollout buffer.  Every rank owns its own 4096 envs (weak scaling); the only exchange is one
NCCL all-reduce of the float64 moment sums (advantage + observation statistics) per rollout.

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference ...                     # CPU oracle port on the host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results as DIR/*.npy
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
# stdout carries exactly one JSON line: NCCL's banner ("NCCL version ..." under NCCL_DEBUG=VERSION/INFO) goes to stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

BYTES_PER_ENV_STEP = 1517          # SURVEY.md section 8(d), config 2 (algorithmic HBM bytes of the playback step)
# dram__bytes_read.sum + dram__bytes_write.sum of play_h1_tp_kernel at 4096 envs x 500 steps come from the newest committed
# `ncu --set full` capture of that launch shape (first file that exists); the line names the file and its hash
TRAFFIC_PROFILES = ("profiles/r02_play_h1_tp_raw.csv", "profiles/r01d_play_h1_tp_raw.csv")
N_ENVS = 4096
HORIZON = 500
GAMMA, LAM = 0.99, 0.97
DUMP_BYTES = 60_000_000            # --dump-outputs: the sampled arrays; with the .npy headers well below 64 MB


def workload_config(n, T):
    """`config` of BOTH arms, key for key (the reference arm's bounded sample is in its `cpu_baseline.sample`)."""
    return {"workload": f"UnitreeH1 walk playback rollout {n} envs x {T} steps per GPU + GAE (configs[1])",
            "envs_per_gpu": n, "horizon": T, "l2": "rollout outputs (2.5 GB/step) exceed the 126 MB L2",
            "gamma": GAMMA, "lam": LAM}


def ncu_traffic(kernel_substr="play_h1_tp_kernel"):
    """(bytes per launch, "file@sha16") of the playback kernel from the committed ncu summary, or (None, None)."""
    import csv
    import hashlib
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for rel in TRAFFIC_PROFILES:
        f = ROOT / rel
        if not f.exists():
            continue
        rows = list(csv.reader(open(f)))
        hdr, units = rows[0], rows[1]
        try:
            ir, iw = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
            row = next(r for r in rows[2:] if kernel_substr in r[0])
            total = float(row[ir]) * scale[units[ir]] + float(row[iw]) * scale[units[iw]]
        except (ValueError, StopIteration, KeyError):
            continue
        return total, f"{rel}@{hashlib.sha256(f.read_bytes()).hexdigest()[:16]}"
    return None, None


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text()), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler(threading.Thread):
    """SM clocks / throttle reasons sampled DURING the timed region (NVML in-process; nvidia-smi if NVML is unavailable)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def _nvml_row(self):
        """The same fields through NVML in this process: a query costs well under a millisecond, where every nvidia-smi
        spawn initialises the driver API again and was seen to stall the end-to-end leg's copies for tens of ms."""
        import pynvml as nv
        if not hasattr(self, "_h"):
            nv.nvmlInit()
            self._h = nv.nvmlDeviceGetHandleByIndex(self.index)
        h = self._h
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = int(get_reasons(h))
        flag = lambda m: "Active" if bits & m else "Not Active"
        return [str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)),
                str(nv.nvmlDeviceGetPowerUsage(h) / 1000.0), flag(0x8), flag(0x40), flag(0x20), flag(0x4)]

    def run(self):
        use_nvml = True
        while not self._stop_evt.is_set():
            try:
                if use_nvml:
                    try:
                        self.rows.append(self._nvml_row())
                    except Exception:
                        use_nvml = False
                if not use_nvml:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                    self.rows.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.1)       # NOT faster: at 100 Hz per rank the NVML queries of 4 ranks cost the step 9 % (driver lock)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def build_table():
    """Dataset-shaped synthetic trajectory -> the reference's resampled table [34, 4, 500] (100 Hz)."""
    from olympics_mujoco_b200 import mjcf, synthetic
    from olympics_mujoco_b200.utils.trajectory import resample_table
    model = mjcf.load_builtin("unitree_h1")
    data = synthetic.h1_walk_dataset(n_traj=4, t_raw=2500, seed=0, model=model)
    return model, resample_table(data, model)


# ------------------------------------------------------------------------------------------- reference arm
def run_reference(args):
    """The reference's CPU path for the same workload, restated (oracle port; the reference's own MuJoCo /
    mushroom_rl stack cannot be installed here).  Rank 0 only; bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cpu_baseline
    model, table = build_table()
    res = cpu_baseline.run(model, table, steps=args.steps, warmup=args.warmup, horizon=args.horizon)
    line = {"impl": "reference", "metric": "env-steps/sec (FK+obs+reward+GAE)", "value": res["value"],
            "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.envs, args.horizon),
            "cpu_baseline": {"value": res["value"], "unit": "env-steps/s", "cores": res["cores"], "kind": res["kind"],
                             "sample": res["sample"]},
            "e2e": {"value": res["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ------------------------------------------------------------------------------------------- configs[4]
def sharded_1m(rank, world, local, table, rollouts=4, warmup=2):
    """BASELINE.json configs[4]: 1 048 576 UnitreeH1 envs sharded by contiguous index range over the ranks, 64-step
    rollouts (two 32-step playback calls into the same device buffers) and ONE all-reduce of the float64 observation
    moments per rollout.  Every rank runs it; returns the aggregate (max-over-ranks time) on every rank."""
    import torch
    import torch.distributed as dist
    from olympics_mujoco_b200 import distributed as D
    from olympics_mujoco_b200 import kernels as Kn
    from olympics_mujoco_b200.environments import LocoEnvBase
    total, t_call, calls = 1 << 20, 32, 2
    env_id0, n_local = D.env_shard(total, rank, world)
    env = LocoEnvBase.make("UnitreeH1.walk.real", n_envs=n_local, traj_params=dict(table=table), seed=1234,
                           env_id0=env_id0, device=f"cuda:{local}")
    roll = env.make_rollout_buffers(t_call)
    mom = torch.zeros(65, dtype=torch.float64, device="cuda")

    def rollout():
        mom.zero_()
        for c in range(calls):                                 # one 64-step rollout = two calls into the same buffers; the
            env.play_trajectory_from_velocity(n_episodes=1, n_steps_per_episode=t_call, render=False, out=roll,
                                              continue_episode=c > 0, obs_moments=mom)   # moments: fused into the kernel
        D.all_reduce_moments(mom)                              # NVLink mailbox kernel (or NCCL), no-op at world 1
        return Kn.moment_stats(mom, "ppo_obs")                 # one kernel

    for _ in range(warmup):
        rollout()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(rollouts):
        rollout()
    t1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = torch.tensor([t0.elapsed_time(t1) / rollouts], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    del roll, env
    torch.cuda.empty_cache()
    ms = float(ms)
    peaks, _ = measured_peaks()
    per_gpu = BYTES_PER_ENV_STEP * (total / world) * t_call * calls / (ms * 1e-3) / 1e9
    return {"workload": f"UnitreeH1 walk, 1048576 envs sharded over {world} GPU(s) (configs[4]): 64-step rollouts, one "
                        "all-reduce of the observation moments per rollout", "envs_per_gpu": n_local, "value": total * t_call * calls / (ms * 1e-3),
            "unit": "env-steps/s", "ms_per_rollout": ms, "scaling": "strong",
            "roofline": {"bound": "hbm", "achieved_per_gpu": per_gpu, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": per_gpu / peaks["hbm_gbs"], "bytes_per_env_step": BYTES_PER_ENV_STEP,
                         "note": "whole rollout incl. the moments pass and the all-reduce, not the kernel alone"}}


def collective_check(rank, world, use_mailbox):
    """Once per run at N > 1: a known per-rank vector (small integers and dyadic fractions: every partial sum is exact in
    float64, so the order of the additions cannot matter) is all-reduced through the route the bench uses (the NVLink
    mailbox kernel) AND through NCCL; both must be bit-equal to each other and to the closed form, on every rank."""
    import torch
    import torch.distributed as dist
    from olympics_mujoco_b200 import distributed as D
    k = torch.arange(68, dtype=torch.float64, device="cuda")
    x = (rank + 1) * (k + 1) + (rank % 4) * 0.25 + k * 2.0 ** -20
    expect = (world * (world + 1) / 2) * (k + 1) + sum((r % 4) * 0.25 for r in range(world)) + world * k * 2.0 ** -20
    via_nccl = x.clone()
    dist.all_reduce(via_nccl, op=dist.ReduceOp.SUM)
    ok = torch.equal(via_nccl, expect)
    if use_mailbox:
        for _ in range(3):                                     # both parity slots
            via_mailbox = D.all_reduce_moments(x.clone())
            ok = ok and torch.equal(via_mailbox, via_nccl)
        torch.cuda.synchronize()
        ok = ok and not D._mailbox.timed_out()
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return "ok" if int(flag) == 1 else "MISMATCH"


def compact(d):
    """One side measurement -> the few numbers the record needs (the whole JSON line must stay short enough to survive a
    truncated stdout tail)."""
    if isinstance(d, list):
        return [compact(x) for x in d]
    if not isinstance(d, dict) or "error" in d:
        return d
    keep = {}
    for k in ("value", "unit", "ms", "ms_per_step", "ms_per_rollout", "task_kernel_ms", "h1_step_kernel_ms", "live_step_ms", "live_step_eager_ms", "live_step_frac",
              "eager_python_loop_ms_per_step", "envs_per_gpu", "scaling", "net"):
        if k in d:
            keep[k] = round(d[k], 5) if isinstance(d[k], float) and abs(d[k]) < 1e6 else d[k]
    if "timing" in d:                                   # how the device time was taken: "eager" launches or "graph" replay
        keep["timing"] = "graph" if d["timing"].startswith("CUDA-graph") else "eager"
    r = d.get("roofline")
    if r:
        for k in ("frac", "frac_executed", "frac_dram", "peak", "bound"):
            if k in r:
                keep[k] = round(r[k], 4) if isinstance(r[k], float) else r[k]
    return keep


def dump_sample(out, vt, adv, mom, budget=DUMP_BYTES):
    """What one step of the timed path hands its caller, gathered on the device: the rollout buffers ([T, C, n] or
    [T, n]) and the value targets and normalised advantages ([T, n]) of a fixed, seeded sample of envs (``env_index``)
    and steps (``step_index``), and copies of the float64 moment sums over all envs (``adv_moments`` [3], ``obs_moments``
    [65]).  As many envs as fit in ``budget`` bytes keep every step; only when one env's steps alone exceed it are the
    steps sampled as well."""
    import torch
    arrays = dict(out, v_target=vt, adv=adv)
    T, n = adv.shape
    per_cell = sum((v[0].numel() // n) * (4 if v.dtype == torch.float32 else 8) for v in arrays.values())  # one (step, env)
    cells = max(1, (budget - 8 * (mom.numel() + n + T)) // per_cell)
    n_env = min(n, max(1, cells // T))
    n_t = min(T, cells // n_env)
    rng = np.random.default_rng(0)
    envs = np.sort(rng.choice(n, size=n_env, replace=False))
    steps = np.arange(T) if n_t == T else np.sort(rng.choice(T, size=n_t, replace=False))
    e_sel, t_sel = (torch.as_tensor(i, device=adv.device) for i in (envs, steps))
    sample = {k: v.index_select(0, t_sel).index_select(v.dim() - 1, e_sel) for k, v in arrays.items()}
    sample.update(adv_moments=mom[:3].clone(), obs_moments=mom[3:].clone(), env_index=envs, step_index=steps)
    return sample


def write_dump(path, sample):
    """``dump_sample``'s arrays as ``path/<name>.npy``: float32 results stay float32, integer and flag buffers and the
    indices are written as float64."""
    path = Path(path)
    path.mkdir(parents=True, exist_ok=True)
    for k, v in sample.items():
        v = v if isinstance(v, np.ndarray) else v.cpu().numpy()
        np.save(path / f"{k}.npy", v if v.dtype in (np.float32, np.float64) else v.astype(np.float64))


# ------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from olympics_mujoco_b200 import kernels as Kn
    from olympics_mujoco_b200.environments import LocoEnvBase

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    # Pin this rank to the CPUs next to its GPU BEFORE any pinned host buffer exists: the end-to-end leg moves 289 MB
    # per step over PCIe into host memory, and with 8 ranks a remote NUMA node halves that bandwidth.
    full_affinity = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
    except Exception:
        pass
    from olympics_mujoco_b200 import distributed as D
    collective, coll_check = "none", None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        # the path's only exchange: 68 float64 per rollout.  One small kernel over NVLink peer memory (csrc/om_mailbox.cu);
        # NCCL if the mailboxes cannot be mapped (decided collectively, so every rank takes the same route)
        collective = "nvlink_mailbox" if (not args.nccl and D.enable_mailbox(True)) else "nccl"
        coll_check = collective_check(rank, world, collective == "nvlink_mailbox")
    n, T = args.envs, args.horizon

    model, table = build_table()
    env = LocoEnvBase.make("UnitreeH1.walk.real", n_envs=n, traj_params=dict(table=table), seed=1234,
                           env_id0=rank * n, device=f"cuda:{local}")
    rolls = [env.make_rollout_buffers(T) for _ in range(2)]    # device-resident [T, C, n] outputs, double-buffered for e2e
    roll = rolls[0]
    g = torch.Generator(device="cuda").manual_seed(7 + rank)
    values = torch.randn((T + 1, n), device="cuda", generator=g)
    values_host = values.cpu().pin_memory()
    last = torch.zeros((T, n), dtype=torch.uint8, device="cuda")
    mom = torch.zeros(3 + 65, dtype=torch.float64, device="cuda")    # advantage [3] + observation [2*32+1]
    ev_k0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ev_k1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]

    mom_adv, mom_obs = mom[:3], mom[3:]

    def hot_step(i=None, vals=values, roll=roll):
        mom.zero_()
        if i is not None:
            ev_k0[i].record()
        # one call = the reference's call: reset() at its start (inside the kernel), 500 steps, end-of-episode reset; the
        # observation moments (S1) are accumulated by the playback kernel itself
        out = env.play_trajectory_from_velocity(n_episodes=1, n_steps_per_episode=T, render=False, out=roll,
                                                obs_moments=mom_obs)
        if i is not None:
            ev_k1[i].record()
        vt, adv = Kn.gae(out["reward"], vals[:-1], vals[1:], out["fallen"], last, GAMMA, LAM)
        Kn.moments_scalar(adv, out=mom_adv)
        D.all_reduce_moments(mom)                              # the path's only exchange (520 B + 24 B, float64)
        stats = Kn.adv_stats(mom_adv, unbiased=False, eps=1e-8)
        Kn.normalize(adv, stats, out=adv)
        return out, vt, adv

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ("value")
    for _ in range(args.warmup):
        hot_step()
    sync_all()
    Kn.reset_launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    # only the last step's results are held: holding each step's while the next one allocates its own would make the
    # caching allocator grow inside the timed region
    for i in range(args.steps - 1):
        hot_step(i)
    last_step = hot_step(args.steps - 1)
    t1.record()
    sync_all()
    launches = Kn.launch_count()
    # gathered on the device before the end-to-end leg reuses the buffers; copied and written once the clocks are sampled
    dump = dump_sample(*last_step, mom) if args.dump_outputs and rank == 0 else None
    del last_step                                              # the end-to-end leg starts from the same allocator state
    ms = torch.tensor([t0.elapsed_time(t1)], device="cuda", dtype=torch.float64)
    kms = torch.tensor([sum(a.elapsed_time(b) for a, b in zip(ev_k0, ev_k1)) / args.steps], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(kms, op=dist.ReduceOp.MAX)
    ms_per_step = float(ms) / args.steps
    value = world * n * T / (ms_per_step * 1e-3)

    # ---- end to end through the public API with host buffers: every step copies its inputs from pinned host memory
    # and its results (observations, rewards, flags, advantages, value targets) back to pinned host memory.  The
    # device->host copy of step i runs on a copy stream while step i+1 computes (two buffer sets); everything,
    # including the last copy, is inside the timed region.
    def host_set():
        h = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in
             dict(obs=roll["obs"], reward=roll["reward"], fallen=roll["fallen"]).items()}
        h["adv"] = torch.empty((T, n)).pin_memory()
        h["v_target"] = torch.empty((T, n)).pin_memory()
        return h
    hosts = [host_set(), host_set()]
    copy_stream = torch.cuda.Stream()
    main = torch.cuda.current_stream()
    copied = [None, None]

    def e2e_step(i):
        b = i % 2
        if copied[b] is not None:
            main.wait_event(copied[b])                         # buffer set b is free again
        vals = values_host.to("cuda", non_blocking=True)
        out, vt, adv = hot_step(vals=vals, roll=rolls[b])
        done = torch.cuda.Event()
        done.record(main)
        copy_stream.wait_event(done)
        with torch.cuda.stream(copy_stream):
            for k, src in (("obs", out["obs"]), ("reward", out["reward"]), ("fallen", out["fallen"]), ("adv", adv),
                           ("v_target", vt)):
                hosts[b][k].copy_(src, non_blocking=True)
                src.record_stream(copy_stream)
            vals.record_stream(copy_stream)
            copied[b] = torch.cuda.Event()
            copied[b].record(copy_stream)
    e2e_steps = args.steps
    for i in range(2):
        e2e_step(i)
    # The end-to-end leg is bound by the HOST path (PCIe + host memory of a shared machine: profiles/r02d_probe_d2h.json),
    # which is noisy from run to run -- one run in five or so reads 2-3x (once 7x) slower than the others, at N = 1 and
    # at N = 2, with or without the clock sampler.  The timed region is therefore measured three times; every reading is
    # reported and the best one is the value.
    e2e_runs = []
    for rep_ in range(3):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main)
        for i in range(e2e_steps):
            e2e_step(i)
        for ev in copied:
            main.wait_event(ev)                                # the last device->host copies are inside the region
        e1.record(main)
        sync_all()
        t = torch.tensor([e0.elapsed_time(e1) / e2e_steps], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_runs.append(float(t))
    clocks = sampler.stop()                                    # sampled across the timed regions (device-resident + e2e)
    if dump is not None:
        write_dump(args.dump_outputs, dump)
        del dump
    e2e_ms = min(e2e_runs)
    host = hosts[0]
    h2d = values_host.numel() * 4
    d2h = sum(v.numel() * v.element_size() for v in host.values())

    sharded = None
    if not args.no_other_configs:
        try:
            sharded = sharded_1m(rank, world, local, table)
        except Exception as e:                                  # never lose the headline line to a side measurement
            sharded = {"error": repr(e)}

    if collective == "nvlink_mailbox":
        bad = torch.tensor([1.0 if D._mailbox.timed_out() else 0.0], device="cuda")
        dist.all_reduce(bad, op=dist.ReduceOp.MAX)
        if float(bad) > 0:                                      # a peer never delivered: that round's sums are NaN there
            collective = "nvlink_mailbox (a round timed out)"
            coll_check = "TIMEOUT"
            sys.stderr.write("bench: the mailbox all-reduce timed out on some rank\n")

    if rank == 0:
        peaks, which = measured_peaks()
        kernel_ms = float(kms)
        achieved = BYTES_PER_ENV_STEP * n * T / (kernel_ms * 1e-3) / 1e9
        traffic, traffic_src = ncu_traffic() if (n, T) == (4096, 500) else (None, None)
        line = {"metric": "env-steps/sec (FK+obs+reward+GAE)", "value": value, "unit": "env-steps/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(n, T), "collective": collective, "collective_check": coll_check,
                "clocks": clocks, "gpu_launches": launches,
                "e2e": {"value": world * n * T / (float(e2e_ms) * 1e-3), "unit": "env-steps/s",
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step_runs": [round(x, 4) for x in e2e_runs], "steps_per_run": e2e_steps},
                # frac: ALGORITHMIC bytes (SURVEY 8(d): 1517 B/env-step, of which the 280 B of trajectory-table and per-env
                # state reads are L2 hits) / kernel time / measured copy peak; frac_dram: the DRAM bytes ncu counted for this
                # launch shape / the same kernel time / the same peak -- the fraction of the HBM pins actually used
                "roofline": {"bound": "hbm", "kernel": "play_snapshot_kernel + play_h1_tp_kernel (one 500-step episode incl. its end-of-episode reset)", "achieved": achieved,
                             "peak": peaks["hbm_gbs"], "peak_source": which, "unit": "GB/s",
                             "frac": achieved / peaks["hbm_gbs"],
                             "frac_dram": (traffic / (kernel_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]) if traffic else None,
                             "traffic": traffic, "traffic_source": traffic_src,
                             "bytes_per_env_step": BYTES_PER_ENV_STEP, "kernel_ms": kernel_ms}}
        if sharded is not None:
            # configs[4] (strong scaling over the ranks), compact and EARLY in the line so that it survives a cut tail
            line["sharded_1m"] = compact(sharded)
        if not args.no_other_configs:
            # the other BASELINE.json configs on this GPU (parity cases; measured here so that one file carries them)
            sys.path.insert(0, str(ROOT / "tools"))
            other = {}
            try:
                import bench_a3
                other["a3_ppo_rollout_16384x64"] = bench_a3.measure(steps=10, warmup=3)
                other["a3_ppo_rollout_262144x64"] = bench_a3.measure(envs=262144, steps=5, warmup=2)
            except Exception as e:                              # never lose the headline line to a side measurement
                other["a3_error"] = repr(e)
            try:
                import bench_h1_step
                other["h1_single_step_1048576"] = bench_h1_step.measure(steps=10, warmup=3)
                other["h1_single_step_131072"] = bench_h1_step.measure(envs=131072, steps=10, warmup=3)
            except Exception as e:
                other["h1_step_error"] = repr(e)
            try:
                import bench_disc
                other["disc_reward_65536"] = bench_disc.measure(steps=20, warmup=3)
                other["disc_reward_1048576"] = bench_disc.measure(envs=1 << 20, steps=10, warmup=3)   # steady state
            except Exception as e:
                other["disc_error"] = repr(e)
            if args.verbose_other:
                sys.stderr.write(json.dumps(other) + "\n")      # the full dictionaries, for the profiles/ record
            line["other_configs"] = {k: compact(v) for k, v in other.items()}
        if not args.no_cpu_baseline:
            if full_affinity is not None:
                os.sched_setaffinity(0, full_affinity)          # the CPU baseline uses every host core
            from oracle import cpu_baseline
            res = cpu_baseline.run(model, table, steps=1, warmup=0, horizon=T, budget_s=args.cpu_budget)
            line["cpu_baseline"] = {"value": res["value"], "unit": "env-steps/s", "cores": res["cores"],
                                    "kind": res["kind"], "sample": res["sample"]}
            # SURVEY 8(d) (i) and (ii): the reference-shaped Python loop, one core and one process per core
            try:
                one = cpu_baseline.python_loop(model, table, horizon=T)
                many = cpu_baseline.python_multiproc(horizon=T)
                line["cpu_baseline"]["python_loop_1core"] = {"value": one["value"], "sample": one["sample"]}
                line["cpu_baseline"]["python_loop_multiproc"] = {"value": many["value"], "cores": many["cores"],
                                                                 "sample": many["sample"]}
            except Exception as e:
                line["cpu_baseline"]["python_loop_error"] = repr(e)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line, on the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=N_ENVS)
    ap.add_argument("--horizon", type=int, default=HORIZON)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--nccl", action="store_true", help="use NCCL for the moment all-reduce instead of the NVLink mailbox kernel")
    ap.add_argument("--cpu-budget", type=float, default=15.0)
    ap.add_argument("--verbose-other", action="store_true", help="full side-measurement dictionaries on stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results (a fixed sample, at most 64 MB) as "
                    "DIR/*.npy; --impl ours only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of --impl ours")
    # stdout carries exactly one JSON line: whatever libraries print at the C level (NCCL's version banner under
    # NCCL_DEBUG=VERSION/WARN ...) is sent to stderr for the duration of the run
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
