"""Timing of BASELINE.json configs[3]: VAIL / GAIL discriminator-reward rollout, 65536 envs (tcgen05 MLP).
Prints one JSON line per network (measurement aid; the driver-facing bench is bench.py).

``--n-in 32 30 48 --rounds 3`` times the networks at other input widths (the UnitreeH1 variants' kinematic
observations) in one process, alternating the widths round by round; a width other than 32 takes the reference weights
with a seeded first layer of that width."""
import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def flop(kind, n_in=32):
    """Useful FLOP per sample, the first layer at the width the kernels compute: n_in rounded up to 32."""
    k = 32 * -(-n_in // 32)
    return {"vail": 2 * (k * 256 + 256 * 128 + 2 * 128 * 128 + 128), "gail": 2 * (k * 512 + 512 * 256 + 256)}[kind]


_TF32_PEAK = None


def tf32_peak():
    """Dense TF32 tensor-pipe rate MEASURED on this GPU: cuBLAS fp32 matmul with TF32 allowed, 8192^3, best of 10 (CUDA
    events) -- the same recipe MEASURED_PEAKS.json uses for bf16.  A measuring stick only: no library GEMM is on the path."""
    global _TF32_PEAK
    if _TF32_PEAK is None:
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        try:
            m = 8192
            a = torch.randn((m, m), device="cuda")
            b = torch.randn((m, m), device="cuda")
            for _ in range(3):
                a @ b
            torch.cuda.synchronize()
            best = float("inf")
            for _ in range(10):
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                a @ b
                t1.record()
                torch.cuda.synchronize()
                best = min(best, t0.elapsed_time(t1))
            _TF32_PEAK = 2.0 * m ** 3 / (best * 1e-3) / 1e12
            del a, b
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev
    return _TF32_PEAK


def measure(envs=65536, steps=50, warmup=5, n_in=32):
    args = argparse.Namespace(envs=envs, steps=steps, warmup=warmup)
    res = []
    from olympics_mujoco_b200 import kernels as Kn
    g = np.load(ROOT / "tests/golden/discriminator_ref.npz")
    n = args.envs
    gen = torch.Generator(device="cuda").manual_seed(0)
    s = torch.randn((n_in, n), device="cuda", generator=gen)
    eps = torch.randn((128, n), device="cuda", generator=gen)
    mean, std = torch.zeros(n_in, device="cuda"), torch.ones(n_in, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()) if (ROOT / "MEASURED_PEAKS.json").exists() else {"bf16_tflops": 1590.0}
    for kind in ("vail", "gail"):
        pref = "v_" if kind == "vail" else "g_"
        names = ("w1", "b1", "w2", "b2", "wmu", "bmu", "wlv", "blv", "wd", "bd") if kind == "vail" else ("w1", "b1", "w2", "b2", "w3", "b3")
        params = {k: g[pref + k] for k in names}
        if n_in != 32:
            rng = np.random.default_rng(n_in)
            params["w1"] = (rng.uniform(-1, 1, (params["w1"].shape[0], n_in)) / np.sqrt(n_in)).astype(np.float32)
        disc = Kn.Discriminator(kind, params)
        e = eps if kind == "vail" else None
        for _ in range(args.warmup):
            disc.reward(s, mean, std, eps=e)
        torch.cuda.synchronize()
        tot = 0.0
        for _ in range(args.steps):
            flush.zero_()                                    # L2 flush between timed launches
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            disc.reward(s, mean, std, eps=e)
            t1.record()
            torch.cuda.synchronize()
            tot += t0.elapsed_time(t1)
        ms = tot / args.steps
        useful = flop(kind, n_in) * n / (ms * 1e-3) / 1e12
        peak_tf32 = tf32_peak()
        width = "" if n_in == 32 else f", {n_in} inputs"
        res.append({"workload": f"{kind.upper()} discriminator reward, {n} envs{width} (configs[3])", "net": kind, "ms": ms,
                    "value": n / (ms * 1e-3), "unit": "samples/s",
                    "roofline": {"bound": "tensor", "achieved": useful, "executed_3xtf32": 3 * useful, "unit": "TFLOP/s",
                                 "peak": peak_tf32, "peak_note": "TF32 matmul 8192^3 measured in this process (best of 10)",
                                 "bf16_burst_half": peaks["bf16_tflops"] / 2,
                                 "frac": useful / peak_tf32, "frac_executed": 3 * useful / peak_tf32,
                                 "flop_per_sample": flop(kind, n_in)}})
        if n_in != 32:
            res[-1]["n_in"] = n_in
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--n-in", type=int, nargs="+", default=[32], help="input widths (1..64), timed in this order")
    ap.add_argument("--rounds", type=int, default=1, help="repeat the sequence of widths, alternating them")
    a = ap.parse_args()
    for _ in range(a.rounds):
        for n_in in a.n_in:
            for r in measure(a.envs, a.steps, a.warmup, n_in):
                print(json.dumps(r))


if __name__ == "__main__":
    main()
