"""GPU: the auto-reset of the batched StickFigureA3 step (``step(autoreset=True, max_traj_len=L)``, ``om_a3_autoreset``)
against ``step`` + ``reset_model(mask=last)`` bit for bit, against the float64 oracle of the PPO sampler loop (flags, ints,
observations, rewards and per-path returns), under the reset curriculum, across shards, at edge and padded sizes, and
replayed from a CUDA graph."""
import ctypes as C

import numpy as np
import pytest

from conftest import assert_close

pytestmark = pytest.mark.gpu

SEED = 3


def _env(n, seed=SEED, env_id0=0):
    from olympics_mujoco_b200 import StickFigureA3
    return StickFigureA3(n_envs=n, seed=seed, env_id0=env_id0)


class Physics:
    """Scripted physics that continues from ``env.qpos`` / ``env.qvel`` (small noise per step) with random contact summaries;
    ``bad(t)`` -> [n] bool sets contact flag bit 2 (bad collision), which makes the step's ``done`` true.  Every step's
    inputs are recorded (float64 copies of the fp32 values the kernels read)."""

    def __init__(self, n, bad=None, seed=1):
        self.n, self.bad, self.rng, self.t, self.script = n, bad, np.random.default_rng(seed), 0, []

    def __call__(self, env, target):
        import torch
        n, rng = self.n, self.rng
        f32 = lambda a: torch.as_tensor(a, dtype=torch.float32, device="cuda")
        q = env.qpos + f32(rng.normal(0, 0.01, (25, n)))
        v = env.qvel + f32(rng.normal(0, 0.1, (24, n)))
        bad = np.zeros(n, bool) if self.bad is None else np.asarray(self.bad(self.t), bool)
        c = f32(np.stack([rng.uniform(0, 300, n), rng.uniform(0, 300, n), rng.uniform(-0.01, 0.01, n), 1.0 + 2.0 * bad]))
        self.script.append((q.cpu().numpy().T.astype(np.float64), v.cpu().numpy().T.astype(np.float64), c.cpu().numpy().T))
        self.t += 1
        return q, v, c


def _state(env):
    d = env._dev
    return dict(qpos=env.qpos.clone(), qvel=env.qvel.clone(), ints=d.ints.clone(), sequence=d.sequence.clone(),
                reset_count=d.reset_count.clone(), traj_len=env.traj_len.clone())


def test_autoreset_equals_step_then_masked_reset():
    """step(a, autoreset=True) == step(a) + reset_model(mask=last), bit for bit, on every state tensor and observation."""
    import torch
    n, L, T = 96, 7, 40
    bad = lambda t: (np.arange(n) * 3 + t) % 11 == 0
    A, B = _env(n), _env(n)
    A.attach_dynamics(Physics(n, bad))
    B.attach_dynamics(Physics(n, bad))
    A.reset()
    B.reset()
    tl = torch.zeros(n, dtype=torch.int32, device="cuda")
    n_reset = n_keep = 0
    codes = set()
    for t in range(T):
        act = np.zeros((n, 12), np.float32)
        oa, ra, da, ia = A.step(act, autoreset=True, max_traj_len=L)
        ob, rb, db, _ = B.step(act)
        final_b = ob.clone()
        tl += 1
        trunc = tl >= L
        last = db | trunc
        B.reset_model(mask=last)
        tl.masked_fill_(last, 0)
        assert torch.equal(ra, rb) and torch.equal(da, db)
        assert torch.equal(ia["final_obs"], final_b)
        assert torch.equal(ia["last"], last)
        want_pe = torch.where(db, 1, torch.where(trunc, 2, 0)).to(torch.uint8)
        assert torch.equal(ia["path_end"], want_pe)
        assert torch.equal(ia["traj_len"], tl)
        assert torch.equal(oa, B.get_obs())
        sa, sb = _state(A), _state(B)
        sb["traj_len"] = tl
        for k in sa:
            assert torch.equal(sa[k], sb[k]), (t, k)
        keep = ~last
        assert torch.equal(oa[keep], ia["final_obs"][keep])                # no reset: the step's observation stays
        n_reset += int(last.sum())
        n_keep += int(keep.sum())
        codes |= set(ia["path_end"].unique().tolist())
    assert codes == {0, 1, 2} and n_reset > 100 and n_keep > 1000


def _bad_table(n, T, seed=5):
    """Forced done (bad collision) per (t, env): env class e % 4 -- 0 never; 1 at t = 49 (where the first path's truncation
    falls: done and truncation together) and every 37 steps after; 2 at two fixed steps; 3 at random, rate 1/40."""
    rng = np.random.default_rng(seed)
    bad = np.zeros((T, n), bool)
    t = np.arange(T)
    for e in range(n):
        c = e % 4
        if c == 1:
            bad[:, e] = (t == 49) | ((t > 49) & ((t - 49) % 37 == 0))
        elif c == 2:
            bad[[10 + e % 30, 150], e] = True
        elif c == 3:
            bad[:, e] = rng.random(T) < 1 / 40
    return bad


def test_autoreset_rollout_against_the_sampler_oracle(a3_model):
    """64 envs x 300 steps, max_traj_len = 50, against oracle.a3_autoreset: integers, flags and path_end exact; obs and
    reward within the project tolerance; finish_path over the device buffer (path_end, v_next = V(final_obs), last_val =
    V(obs_T), a fixed linear critic) equal to the oracle's per-path returns."""
    import torch
    from olympics_mujoco_b200.learners import finish_path
    from olympics_mujoco_b200.tasks.phase_clock import phase_clock_lut
    from oracle import a3 as OA
    from oracle import a3_autoreset as OR
    n, T, L, gamma, it = 64, 300, 50, 0.99, 6000.0
    bad = _bad_table(n, T)
    env = _env(n, seed=11, env_id0=100)
    env.robot.iteration_count = it
    phys = Physics(n, lambda t: bad[t], seed=2)
    env.attach_dynamics(phys)
    obs = env.reset().clone()
    keys = ("obs", "final_obs", "reward", "done", "last", "path_end", "traj_len", "reset_count", "ints", "sequence")
    rec = {k: [] for k in keys}
    for t in range(T):
        rec["obs"].append(obs.cpu().numpy())
        obs, r, d, info = env.step(np.zeros((n, 12), np.float32), autoreset=True, max_traj_len=L)
        obs = obs.clone()
        for k, v in (("final_obs", info["final_obs"]), ("reward", r), ("done", d), ("last", info["last"]),
                     ("path_end", info["path_end"]), ("traj_len", info["traj_len"]), ("reset_count", env._dev.reset_count),
                     ("ints", env._dev.ints.t()), ("sequence", env._dev.sequence.t().reshape(n, 20, 4))):
            rec[k].append(v.cpu().numpy().copy())
    dev = {k: np.stack(v) for k, v in rec.items()}                         # [T, n, ...]
    w = np.random.default_rng(7).normal(0, 0.05, 41)
    b = 0.3
    critic64 = lambda o: float(w @ o) + b
    wt = torch.as_tensor(w, dtype=torch.float32, device="cuda")
    V = lambda o: torch.as_tensor(o, device="cuda") @ wt + b                # [T, n, 41] or [n, 41] -> values
    values, v_next = V(dev["obs"]).contiguous(), V(dev["final_obs"]).contiguous()
    ret, adv = finish_path(torch.as_tensor(dev["reward"], device="cuda"), values, gamma,
                           path_end=torch.as_tensor(dev["path_end"], device="cuda"), v_next=v_next, last_val=V(obs.cpu().numpy()))
    ret, adv = ret.cpu().numpy(), adv.cpu().numpy()
    lut = phase_clock_lut()
    seen = dict(ended=0, truncated=0, both=0)
    for e in range(n):
        states = [(q[e], v[e], OA.Contact(l_grf=c[e, 0], r_grf=c[e, 1], min_z=c[e, 2], foot_contact=bool(int(c[e, 3]) & 1),
                                          bad_collision=bool(int(c[e, 3]) & 2))) for q, v, c in phys.script]
        o = OR.sample(a3_model, states, lut, max_traj_len=L, seed=11, env_id=100 + e, iteration_count=it)
        for k in ("done", "last", "path_end", "traj_len", "reset_count"):
            np.testing.assert_array_equal(dev[k][:, e].astype(np.int64), o[k].astype(np.int64), err_msg=f"env {e} {k}")
        np.testing.assert_array_equal(dev["ints"][:, e], o["ints"], err_msg=f"env {e} ints")
        assert_close(dev["sequence"][:, e], o["sequence"], f"env {e} sequence")
        assert_close(dev["obs"][:, e], o["obs"], f"env {e} obs")
        assert_close(dev["final_obs"][:, e], o["final_obs"], f"env {e} final_obs")
        assert_close(dev["reward"][:, e], o["reward"], f"env {e} reward")
        r_ref, a_ref = OR.path_returns(o, critic64, gamma)
        # returns are discounted sums of up to 50 rewards (and a critic value): the tolerance of one reward times 10
        assert_close(ret[:, e], r_ref, f"env {e} returns", atol=1e-4)
        assert_close(adv[:, e], a_ref, f"env {e} advantages", atol=1e-4)
        seen["ended"] += int((o["path_end"] == 1).sum())
        seen["truncated"] += int((o["path_end"] == 2).sum())
        seen["both"] += int((o["done"] & o["trunc"]).sum())
    assert seen["ended"] > 50 and seen["truncated"] > 50 and seen["both"] >= 8, seen


@pytest.mark.parametrize("it", [0.0, 7000.0, np.inf])
def test_autoreset_curriculum_step_heights(a3_model, it):
    """iteration_count is read from env.robot at call time: the reset footstep plans climb 0, 0.05 or 0.1 per step, as
    oracle.a3.reset draws them."""
    from oracle import a3 as OA
    from oracle import a3_autoreset as OR
    n = 48
    env = _env(n, seed=21)
    env.attach_dynamics(Physics(n, lambda t: np.ones(n, bool)))
    env.reset()
    env.robot.iteration_count = it
    env.step(np.zeros((n, 12), np.float32), autoreset=True)
    seq = env._dev.sequence.t().reshape(n, 20, 4).cpu().numpy()
    ints = env._dev.ints.t().cpu().numpy()
    dz = set()
    for e in range(n):
        _, _, ts, _ = OA.reset(a3_model, 21, e, 1, iteration_count=it)
        assert ints[e].tolist() == OR.ints_of(ts)
        assert_close(seq[e], np.asarray(ts.sequence), f"env {e} sequence")
        if ts.mode == OA.FORWARD:
            dz.add(round(abs(float(ts.sequence[5][2] - ts.sequence[4][2])), 6))
    assert dz == {dict([(0.0, 0.0), (7000.0, 0.05), (np.inf, 0.1)])[it]}


def _task(n, seed=SEED, env_id0=0):
    from olympics_mujoco_b200 import kernels as Kn
    from olympics_mujoco_b200.tasks.phase_clock import phase_clock_lut
    from oracle import a3 as OA
    from olympics_mujoco_b200 import mjcf
    return Kn.A3Task(Kn.DeviceModel(mjcf.load_builtin("stick_figure_a3")), n, phase_clock_lut(), OA.init_qpos(), seed=seed,
                     env_id0=env_id0)


class Bufs:
    """The device buffers of one step + auto-reset at the Kn level."""

    def __init__(self, n):
        import torch
        z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device="cuda")
        self.qpos, self.qvel, self.con = z(25, n), z(24, n), z(4, n)
        self.out = dict(obs=z(41, n), terms=z(6, n), reward=z(n), done=z(n, dt=torch.uint8))
        self.obs, self.tl = z(41, n), z(n, dt=torch.int32)
        self.last, self.pe = z(n, dt=torch.uint8), z(n, dt=torch.uint8)

    def step(self, task, L, it=5000.0):
        task.step(self.qpos, self.qvel, self.con, out=self.out)
        task.autoreset(self.qpos, self.qvel, self.out["done"], self.tl, self.out["obs"], self.obs, self.last, self.pe,
                       max_traj_len=L, iteration_count=it)

    def all(self, task):
        return dict(qpos=self.qpos, qvel=self.qvel, final=self.out["obs"], reward=self.out["reward"], done=self.out["done"],
                    obs=self.obs, tl=self.tl, last=self.last, pe=self.pe, ints=task.ints, seq=task.sequence,
                    rc=task.reset_count)


def _inputs(n, T, seed=4):
    rng = np.random.default_rng(seed)
    noise = [(rng.normal(0, 0.01, (25, n)).astype(np.float32), rng.normal(0, 0.1, (24, n)).astype(np.float32)) for _ in range(T)]
    con = [np.stack([rng.uniform(0, 300, n), rng.uniform(0, 300, n), rng.uniform(-0.01, 0.01, n),
                     1.0 + 2.0 * (rng.random(n) < 0.15)]).astype(np.float32) for _ in range(T)]
    return noise, con


def test_autoreset_two_shards_equal_one_batch():
    import torch
    n, T, L = 130, 12, 4
    full, a, b = _task(n), _task(n // 2), _task(n // 2, env_id0=n // 2)
    bf, ba, bb = Bufs(n), Bufs(n // 2), Bufs(n // 2)
    for t_, bu in ((full, bf), (a, ba), (b, bb)):
        t_.reset(bu.qpos, bu.qvel, iteration_count=5000.0, obs=bu.obs)
    noise, con = _inputs(n, T)
    h = n // 2
    for t in range(T):
        for bu, sl in ((bf, slice(0, n)), (ba, slice(0, h)), (bb, slice(h, n))):
            bu.qpos += torch.as_tensor(noise[t][0][:, sl], device="cuda")
            bu.qvel += torch.as_tensor(noise[t][1][:, sl], device="cuda")
            bu.con.copy_(torch.as_tensor(con[t][:, sl].copy(), device="cuda"))
        bf.step(full, L)
        ba.step(a, L)
        bb.step(b, L)
        F, A, B = bf.all(full), ba.all(a), bb.all(b)
        for k in F:
            assert torch.equal(F[k][..., :h], A[k]) and torch.equal(F[k][..., h:], B[k]), (t, k)
    assert int(full.reset_count.sum()) > n + 20


@pytest.mark.parametrize("n", [0, 1, 63, 129])
def test_autoreset_sizes_through_the_env(n):
    import torch
    from olympics_mujoco_b200 import StickFigureA3
    env = _env(n)
    env.attach_dynamics(Physics(n))
    obs0 = env.reset()
    assert obs0.shape == (n, 41) and env.traj_len.shape == (n,)
    tl, rc = np.zeros(n, np.int64), np.ones(n, np.int64)
    for t in range(4):
        obs, r, d, info = env.step(np.zeros((n, 12), np.float32), autoreset=True, max_traj_len=2)
        assert obs.shape == (n, 41) and info["final_obs"].shape == (n, 41) and r.shape == d.shape == (n,)
        assert info["last"].dtype == torch.bool and info["path_end"].dtype == torch.uint8
        assert info["traj_len"].dtype == torch.int32 and info["traj_len"].shape == (n,)
        d = d.cpu().numpy()
        tl += 1
        pe = np.where(d, 1, np.where(tl >= 2, 2, 0))
        tl[pe > 0] = 0
        rc += pe > 0
        assert info["path_end"].cpu().numpy().tolist() == pe.tolist() and info["traj_len"].cpu().numpy().tolist() == tl.tolist()
        assert torch.isfinite(obs).all() and torch.isfinite(info["final_obs"]).all()
    assert env._dev.reset_count.cpu().numpy().tolist() == rc.tolist()
    single = StickFigureA3(seed=SEED)
    single.attach_dynamics(Physics(1))
    single.reset()
    obs, r, d, info = single.step(np.zeros(12, np.float32), autoreset=True, max_traj_len=1)
    assert obs.shape == (41,) and info["final_obs"].shape == (41,) and int(info["path_end"]) in (1, 2) and bool(info["last"])


def test_autoreset_padded_ld_leaves_the_padding_alone():
    """n envs of an ld = n + 63 wide state: columns n.. of every tensor the call may write keep their sentinel, and the
    n processed columns equal those of an unpadded batch."""
    import torch
    n, ld = 65, 128
    pad, ref = _task(ld), _task(n)
    bp, br = Bufs(ld), Bufs(n)
    pad.reset(bp.qpos, bp.qvel, obs=bp.obs)
    ref.reset(br.qpos, br.qvel, obs=br.obs)
    rng = np.random.default_rng(9)
    done = torch.as_tensor(rng.random(ld) < 0.4, device="cuda").to(torch.uint8)
    done[n:] = 1
    tl = torch.as_tensor(rng.integers(0, 6, ld), dtype=torch.int32, device="cuda")
    obs_in = torch.as_tensor(rng.normal(0, 1, (41, ld)), dtype=torch.float32, device="cuda")
    S = dict(qpos=bp.qpos, qvel=bp.qvel, ints=pad.ints, seq=pad.sequence, rc=pad.reset_count, tl=bp.tl, obs=bp.obs,
             last=bp.last, pe=bp.pe)
    bp.tl.copy_(tl)
    br.tl.copy_(tl[:n])
    for k, x in S.items():
        x[..., n:] = 77 if x.dtype != torch.float32 else float("nan")
    keep = {k: x[..., n:].clone() for k, x in S.items()}
    pad.autoreset(bp.qpos, bp.qvel, done, bp.tl, obs_in, bp.obs, bp.last, bp.pe, max_traj_len=5, n=n)
    ref.autoreset(br.qpos, br.qvel, done[:n].contiguous(), br.tl, obs_in[:, :n].contiguous(), br.obs, br.last, br.pe,
                  max_traj_len=5)
    R = dict(qpos=br.qpos, qvel=br.qvel, ints=ref.ints, seq=ref.sequence, rc=ref.reset_count, tl=br.tl, obs=br.obs,
             last=br.last, pe=br.pe)
    for k, x in S.items():
        assert torch.equal(x[..., n:], keep[k]) or (x.dtype == torch.float32 and torch.isnan(x[..., n:]).all()), k
        assert torch.equal(x[..., :n], R[k]), k
    assert 0 < int(br.last.sum()) < n


def test_autoreset_step_captured_in_a_cuda_graph_replays_like_eager():
    import torch
    n, T, L = 300, 8, 3
    te, tg = _task(n, seed=8), _task(n, seed=8)
    be, bg = Bufs(n), Bufs(n)
    te.reset(be.qpos, be.qvel, obs=be.obs)
    tg.reset(bg.qpos, bg.qvel, obs=bg.obs)
    noise, con = _inputs(n, T, seed=6)
    eager = []
    for t in range(T):                                       # eager first: it also loads every kernel before the capture
        be.qpos += torch.as_tensor(noise[t][0], device="cuda")
        be.qvel += torch.as_tensor(noise[t][1], device="cuda")
        be.con.copy_(torch.as_tensor(con[t], device="cuda"))
        be.step(te, L)
        eager.append({k: v.clone() for k, v in be.all(te).items()})
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        bg.step(tg, L)
    for t in range(T):
        bg.qpos += torch.as_tensor(noise[t][0], device="cuda")
        bg.qvel += torch.as_tensor(noise[t][1], device="cuda")
        bg.con.copy_(torch.as_tensor(con[t], device="cuda"))
        g.replay()
        got = bg.all(tg)
        for k in got:
            assert torch.equal(got[k], eager[t][k]), (t, k)
    assert int(tg.reset_count.sum()) > n + 100


def test_autoreset_refusals_launch_nothing(a3_model, h1_model):
    import torch
    from olympics_mujoco_b200 import _lib
    from olympics_mujoco_b200 import kernels as Kn
    n = 8
    task, bu = _task(n), Bufs(n)
    lib = _lib.load()
    v = lambda t: t.data_ptr()
    st = task._state()

    def args(**kw):
        a = dict(done=v(bu.out["done"]), max_traj_len=0, iteration_count=0.0, reset_count=v(task.reset_count), traj_len=v(bu.tl),
                 qpos=v(bu.qpos), qvel=v(bu.qvel), state=st, obs_in=v(bu.out["obs"]), obs=v(bu.obs), last=v(bu.last),
                 path_end=v(bu.pe))
        a.update(kw)
        return _lib.OmA3AutoResetArgs(**a)

    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    h1 = Kn.DeviceModel(h1_model)
    cases = [(h1.handle, args(), n, n, "not the StickFigureA3 model"), (task.dm.handle, args(), n, n - 1, "n <= ld"),
             (task.dm.handle, args(max_traj_len=-1), n, n, "max_traj_len"),
             (task.dm.handle, args(traj_len=None), n, n, "null input"), (task.dm.handle, args(obs_in=None), n, n, "null input")]
    for model, a, nn, ld, msg in cases:
        before = Kn.launch_count()
        assert lib.om_a3_autoreset(model, task.handle, 1, 0, C.byref(a), nn, ld, stream) != 0
        assert msg in lib.om_last_error().decode()
        assert Kn.launch_count() == before
    assert lib.om_a3_autoreset(task.dm.handle, task.handle, 1, 0, C.byref(args()), n, n, stream) == 0
