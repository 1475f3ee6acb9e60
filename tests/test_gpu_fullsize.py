"""GPU tests at BASELINE.json's FULL sizes through size-independent properties and kernel-against-kernel agreement:
configs[1] 4096 envs x 500 steps H1 playback, configs[2] 16384 envs x 64 steps A3 rollout, configs[4] 1 M sharded envs.
The time-parallel and sequential playback kernels compared here share their loop body, so a defect common to both
passes; test_gpu_fullsize_oracle.py compares the benchmarked configs[1] step and a configs[4] shard with the float64 C
oracle on every env and step.  (configs[3], the 65536-env discriminator, is covered against the oracle in
test_gpu_disc.py.)"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _h1_setup(n, seed, env_id0=0):
    import bench
    from olympics_mujoco_b200 import kernels as Kn
    from oracle import h1 as OH
    model, table = bench.build_table()                       # the bench's [34, 4, 500] table
    dm = Kn.DeviceModel(model)
    spec = Kn.make_h1_spec(OH.perm(model), OH.x_vel_idx(model))
    traj = Kn.DeviceTrajectory(table, n, seed=seed, env_id0=env_id0)
    sample = traj.reset()
    state = dict(curr_qpos=sample[:17].double().contiguous(), pending=sample.clone(), prev_x_vel=sample[17].clone())
    return model, table, dm, spec, traj, state


def test_h1_playback_full_size_properties(om_knob):
    """4096 envs x 500 steps: (1) the time-parallel kernel and the sequential-in-time kernel agree bit for bit on every
    integer / gathered output and within the path's 1e-5 tolerance on the FK outputs; (2) the observation is exactly the
    table row of the recorded (traj_no, step_no); (3) the index advances by one except at wrap resets, which happen exactly at step_no == T; (4) quaternions are unit; (5) the reward is
    exp(-(previous dq_pelvis_tx - 1.25)^2); (6) fallen is never raised on the non-terminal dataset."""
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    n, T, seed = 4096, 500, 4242
    outs = {}
    for chunk in ("7", "1000000"):
        om_knob("play_chunk", int(chunk))
        model, table, dm, spec, traj, state = _h1_setup(n, seed)
        out = Kn.h1_play_from_velocity(dm, spec, traj, state, T)
        torch.cuda.synchronize()
        outs[chunk] = (out, traj.traj_no.clone(), traj.step_no.clone(), traj.reset_count.clone(), state["curr_qpos"].clone())
    a, b = outs["7"], outs["1000000"]
    for k in a[0]:
        if k in ("xpos", "xquat", "site_xpos", "cvel"):
            # the Euler sum is re-associated through the float64 prefix table: q agrees to ~1e-15, its fp32 image and the
            # FK outputs to the last bit or two
            assert torch.allclose(a[0][k], b[0][k], rtol=1e-5, atol=1e-5), f"time-parallel vs sequential: {k}"
        else:
            assert torch.equal(a[0][k], b[0][k]), f"time-parallel and sequential kernels differ in {k}"
    for i in range(1, 4):
        assert torch.equal(a[i], b[i])
    assert torch.allclose(a[4], b[4], rtol=1e-13, atol=1e-13)
    out = a[0]
    tr, st = out["traj_no_t"].long(), out["step_no_t"].long()
    Tt = table.shape[2]
    tab32 = torch.as_tensor(table.astype(np.float32), device="cuda")                       # [34, n_traj, T]
    gathered = tab32[2:, tr, st]                                                            # [32, T, n]
    assert torch.equal(out["obs"], gathered.permute(1, 0, 2).contiguous()), "obs must be the exact table row"
    dstep = st[1:] - st[:-1]
    wrapped = dstep != 1
    assert torch.all(st < Tt) and torch.all(st >= 0) and torch.all((tr >= 0) & (tr < table.shape[1]))
    assert torch.all(st[:-1][wrapped] == Tt - 1), "a reset happens only after the last sample of a trajectory"
    assert int(wrapped.sum()) > n // 2                       # 500 steps of 500-sample trajectories: most envs wrap once
    q = out["xquat"].view(T, 21, 4, n)
    assert torch.allclose((q * q).sum(dim=2), torch.ones((), device="cuda"), atol=2e-6)
    prev = torch.cat([state["prev_x_vel"].new_zeros(1, n), out["obs"][:-1, 15]], dim=0)
    r_ref = torch.exp(-(prev[1:] - 1.25) ** 2)
    assert torch.allclose(out["reward"][1:], r_ref, rtol=1e-6, atol=1e-7)
    assert int(out["fallen"].sum()) == 0
    assert torch.isfinite(out["cvel"]).all() and torch.isfinite(out["xpos"]).all()


def test_a3_rollout_full_size_properties(a3_model, om_knob):
    """16384 envs x 64 steps: the fused kernel and the time-parallel pair agree (integers and flags bit for bit,
    floats to fp32 rounding); phase advances mod 88; done == (root z - lowest foot site z < 0.6) | bad collision as
    recomputed from the K1 kernel's outputs; observation rows that are pure copies are exact."""
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    from olympics_mujoco_b200.tasks.phase_clock import phase_clock_lut
    from oracle import a3 as OA
    n, T = 16384, 64
    dm = Kn.DeviceModel(a3_model)
    g = torch.Generator(device="cuda").manual_seed(3)
    res = {}
    for split in ("0", "1"):
        om_knob("a3_split", int(split))
        task = Kn.A3Task(dm, n, phase_clock_lut(), OA.init_qpos(), seed=11)
        q0, v0 = Kn.soa(25, n), Kn.soa(24, n)
        task.reset(q0, v0, iteration_count=6000.0)
        if split == "0":
            qpos = q0[None] + 0.01 * torch.randn((T, 25, n), device="cuda", generator=g).cumsum(0)
            # a tenth of the envs fold their legs (hip flexion, knee flexion) until the feet come up under the root
            fold = torch.linspace(0, 1, T, device="cuda")[:, None] * (torch.rand(n, device="cuda", generator=g) < 0.1)
            for hip, knee in ((7, 10), (13, 16)):
                qpos[:, hip] -= 1.3 * fold
                qpos[:, knee] -= 1.6 * fold
            qvel = torch.randn((T, 24, n), device="cuda", generator=g)
            con = torch.stack([torch.rand((T, n), device="cuda", generator=g) * 400, torch.rand((T, n), device="cuda", generator=g) * 400,
                               (torch.rand((T, n), device="cuda", generator=g) - 0.5) * 0.02,
                               (torch.rand((T, n), device="cuda", generator=g) < 0.7).float()
                               + 2 * (torch.rand((T, n), device="cuda", generator=g) < 0.01).float()], dim=1).contiguous()
            ints0 = task.ints.clone()
        out = task.step(qpos, qvel, con)
        torch.cuda.synchronize()
        res[split] = (out, task.ints.clone())
    (fa, ia), (sp, ib) = res["0"], res["1"]
    assert torch.equal(ia, ib) and torch.equal(fa["done"], sp["done"])
    for k in ("obs", "terms", "reward"):
        assert torch.allclose(fa[k], sp[k], rtol=1e-6, atol=1e-6), k
    out = sp
    assert torch.equal(ia[0], (ints0[0] + T) % 88)                                          # phase clock
    assert torch.equal(out["obs"][:, 7:19], qpos[:, 7:19]) and torch.equal(out["obs"][:, 19:31], qvel[:, 6:18])
    assert torch.equal(out["obs"][:, 4:7], qvel[:, 3:6])
    # done == the FLOAT64 oracle's decision on every one of the 1 048 576 env-steps (no tolerance on the flag: decisions
    # within 1e-5 m of the threshold are re-taken in float64 by the kernels)
    from oracle import kinematics as K
    q64 = qpos.permute(0, 2, 1).reshape(T * n, 25).double().cpu().numpy()
    ls, rs = a3_model.site_id("lf_force"), a3_model.site_id("rf_force")
    h = np.empty(T * n)
    for c0 in range(0, T * n, 1 << 17):
        ref = K.mj_kinematics(a3_model, q64[c0:c0 + (1 << 17)])
        h[c0:c0 + (1 << 17)] = ref["xpos"][:, 1, 2] - np.minimum(ref["site_xpos"][:, ls, 2], ref["site_xpos"][:, rs, 2])
    bad = (con[:, 3] >= 2)
    want_done = torch.as_tensor((h < 0.6).reshape(T, n), device="cuda") | bad
    assert torch.equal(out["done"].bool(), want_done)
    # (whether any of these env-steps needed the float64 re-decision depends on the draw; the adversarial inputs of
    # test_gpu_a3.py::test_a3_threshold_flags_equal_float64_oracle_on_adversarial_inputs always do)
    # full-size parity against the oracle: 24 envs stepped through all 64 steps by the float64 restatement of the task
    seq_dev = task.sequence.cpu().numpy().T.reshape(n, 20, 4).astype(np.float64)
    lut = phase_clock_lut()
    rng = np.random.default_rng(0)
    conh, qh, vh = con.cpu().numpy(), qpos.cpu().numpy(), qvel.cpu().numpy()
    obs_h, rew_h, done_h = out["obs"].cpu().numpy(), out["reward"].cpu().numpy(), out["done"].cpu().numpy()
    ints_end = ib.cpu().numpy()
    from conftest import assert_close
    for e in rng.choice(n, 24, replace=False):
        _, _, ts, _ = OA.reset(a3_model, 11, int(e), 0, iteration_count=6000.0)
        assert [ts.phase, ts.t1, ts.t2, ts.target_reached_frames, ts.mode, ts.seq_len, int(ts.target_reached)] == list(ints0[:, e].cpu().numpy())
        ts.sequence = [seq_dev[e, k].copy() if k < ts.seq_len else np.asarray(ts.sequence[k]).copy() for k in range(len(ts.sequence))]
        for t in range(T):
            c = conh[t, :, e].astype(np.float64)
            fl = int(c[3])
            cc = OA.Contact(l_grf=c[0], r_grf=c[1], min_z=c[2], foot_contact=bool(fl & 1), bad_collision=bool(fl & 2))
            obs, total, dn, _ = OA.step_tail(a3_model, qh[t, :, e].astype(np.float64), vh[t, :, e].astype(np.float64), ts, cc, lut)
            assert bool(done_h[t, e]) == dn
            assert_close(obs_h[t, :, e], obs, f"obs env {e} step {t}")
            assert_close(rew_h[t, e], total, f"reward env {e} step {t}")
        assert [ts.phase, ts.t1, ts.t2, ts.target_reached_frames, ts.mode, ts.seq_len, int(ts.target_reached)] == list(ints_end[:, e])
    assert bool((want_done & ~bad).any()) and bool(bad.any()) and 0.005 < float(out["done"].float().mean()) < 0.5
    assert torch.isfinite(out["obs"]).all() and torch.isfinite(out["reward"]).all()
    assert float(out["reward"].min()) > -0.31 and float(out["reward"].max()) < 1.0 + 1e-5   # 0.15*(2 tan terms in [-1,1]) + ...


def test_sharded_million_env_step_equals_single_process():
    """configs[4]: 1 048 576 H1 envs.  Two shards with env_id0 offsets (what ranks 0 and 1 of a 2-GPU job run) produce
    exactly the slices of the single-process run: resets (Philox contract), one fused step, and their float64 moment
    partial sums add up to the global ones (what the NCCL all-reduce delivers)."""
    import torch
    from olympics_mujoco_b200 import distributed as D
    from olympics_mujoco_b200 import kernels as Kn
    n = 1 << 20
    runs = {}
    for name, (e0, m) in dict(all=(0, n), lo=D.env_shard(n, 0, 2), hi=D.env_shard(n, 1, 2)).items():
        model, table, dm, spec, traj, state = _h1_setup(m, seed=77, env_id0=e0)
        sample = traj.current()
        qpos, qvel = torch.empty((17, m), device="cuda"), torch.empty((17, m), device="cuda")
        from oracle import h1 as OH
        perm = torch.as_tensor(OH.perm(model), device="cuda")
        qpos[perm] = sample[:17]
        qvel[perm] = sample[17:]
        out = Kn.h1_step(dm, spec, qpos, qvel, sample[17].clone(), want_fk=True)
        mom = Kn.moments(out["obs"])
        torch.cuda.synchronize()
        runs[name] = (traj.traj_no.clone(), traj.step_no.clone(), out["obs"].clone(), out["xpos"].clone(), out["reward"].clone(), mom)
        del out
    half = n // 2
    for i in range(2):
        assert torch.equal(runs["all"][i][:half], runs["lo"][i]) and torch.equal(runs["all"][i][half:], runs["hi"][i])
    for i in (2, 3):
        assert torch.equal(runs["all"][i][:, :half], runs["lo"][i]) and torch.equal(runs["all"][i][:, half:], runs["hi"][i])
    assert torch.equal(runs["all"][4][:half], runs["lo"][4])
    tot = runs["lo"][5] + runs["hi"][5]
    assert torch.allclose(tot, runs["all"][5], rtol=1e-12) and float(tot[-1]) == n
    counts = torch.bincount(runs["all"][1].long(), minlength=500).float()                   # uniform substep draw
    assert float(counts.min()) > 0.85 * n / 500 and float(counts.max()) < 1.15 * n / 500
