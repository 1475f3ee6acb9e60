"""GPU: the VAIL / GAIL discriminator (K4) at input widths other than 32 -- the kinematic observation of every UnitreeH1
variant (30 without the back joint, 48 with arms, 46 with arms and without the back joint) and the ends of the
supported range 1..64.  Kernels against the float64 oracle (oracle/learner.py) and a float64 torch restatement built
from nn.Linear, the over-read check with NaN padding, the refusals, and the learner hooks end to end on played
observations of each variant."""
import ctypes as C

import numpy as np
import pytest

from conftest import assert_close

pytestmark = pytest.mark.gpu

WIDTHS = (30, 46, 48, 64, 1)
KNOB_DEFAULTS = dict(disc_vail2=-1, disc_pg2=-1)


@pytest.fixture
def disc_knob():
    """Force a discriminator kernel variant for one test (om_debug_set); both knobs are back on automatic afterwards."""
    from olympics_mujoco_b200 import _lib
    lib = _lib.load()

    def set_knob(name, value):
        _lib.check(lib.om_debug_set(name.encode(), int(value)))
    yield set_knob
    for k, v in KNOB_DEFAULTS.items():
        lib.om_debug_set(k.encode(), v)


def _params(kind, n_in, seed=0):
    """Seeded weights in nn.Linear layout, scaled like nn.Linear's default initialisation."""
    rng = np.random.default_rng(seed)
    lin = lambda o, i: (rng.uniform(-1, 1, (o, i)) / np.sqrt(i), rng.uniform(-1, 1, o) / np.sqrt(i))
    p = {}
    if kind == "vail":
        p["w1"], p["b1"] = lin(256, n_in)
        p["w2"], p["b2"] = lin(128, 256)
        p["wmu"], p["bmu"] = lin(128, 128)
        p["wlv"], p["blv"] = lin(128, 128)
        p["wd"], p["bd"] = lin(1, 128)
    else:
        p["w1"], p["b1"] = lin(512, n_in)
        p["w2"], p["b2"] = lin(256, 512)
        p["w3"], p["b3"] = lin(1, 256)
    return {k: v.astype(np.float32) for k, v in p.items()}


def _torch_ref(kind, p, s, mean, std, eps):
    """float64 restatement with torch.nn.Linear on the device: s [n_in, n] -> (logit [n], kl [n] or None)."""
    import torch
    nn = torch.nn

    def linear(w, b):
        m = nn.Linear(w.shape[1], w.shape[0], dtype=torch.float64, device="cuda")
        with torch.no_grad():
            m.weight.copy_(torch.as_tensor(w, dtype=torch.float64))
            m.bias.copy_(torch.as_tensor(b, dtype=torch.float64))
        return m
    with torch.no_grad():
        x = (s.double().t() - mean.double()) / std.double()
        if kind == "vail":
            h = torch.relu(linear(p["w2"], p["b2"])(torch.relu(linear(p["w1"], p["b1"])(x))))
            mu, lv = linear(p["wmu"], p["bmu"])(h), linear(p["wlv"], p["blv"])(h)
            z = mu + torch.exp(lv / 2) * (eps.double().t() if eps is not None else 0.0)
            d = linear(p["wd"], p["bd"])(z)[:, 0]
            kl = 0.5 * (mu * mu + torch.exp(lv) - lv - 1).sum(dim=1)
            return d, kl
        h = torch.tanh(linear(p["w2"], p["b2"])(torch.tanh(linear(p["w1"], p["b1"])(x))))
        return linear(p["w3"], p["b3"])(h)[:, 0], None


def _reward(d):
    return -np.log(1.0 - 1.0 / (1.0 + np.exp(-np.asarray(d, np.float64))) + 1e-8)


def _inputs(n_in, n, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    scale = torch.rand(n_in, 1, device="cuda", generator=g) * 2.8 + 0.2
    s = torch.randn((n_in, n), device="cuda", generator=g) * scale + torch.randn((n_in, 1), device="cuda", generator=g)
    mean = torch.randn(n_in, device="cuda", generator=g) * 0.5
    std = torch.rand(n_in, device="cuda", generator=g) * 2 + 0.3
    eps = torch.randn((128, n), device="cuda", generator=g)
    return s, mean, std, eps


def _check_forward(kind, n_in, n, with_eps, seed):
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    from oracle import learner as L
    p = _params(kind, n_in, seed=n_in)
    disc = Kn.Discriminator(kind, p)
    assert disc.n_in == n_in
    s, mean, std, eps = _inputs(n_in, n, seed)
    e = eps if (kind == "vail" and with_eps) else None
    fw = disc.forward(s, mean, std, eps=e, want_reward=True)
    r, d = disc.reward(s, mean, std, eps=e, want_d=True)
    torch.cuda.synchronize()
    d_t, kl_t = _torch_ref(kind, p, s, mean, std, e)
    # against the torch restatement: every sample
    assert_close(fw["logit"].cpu().numpy(), d_t.cpu().numpy(), "logit vs torch float64")
    assert_close(fw["reward"].cpu().numpy(), _reward(d_t.cpu().numpy()), "reward vs torch float64")
    assert torch.equal(r, fw["reward"]) and torch.equal(d, fw["logit"]), "om_disc_reward and om_disc_forward differ"
    if kind == "vail":
        assert_close(fw["kl"].cpu().numpy(), kl_t.cpu().numpy(), "kl vs torch float64")
    # against the float64 oracle: every sample, or a sample of them for large n
    rng = np.random.default_rng(n)
    idx = np.arange(n) if n <= 4096 else np.concatenate([np.arange(256), rng.choice(n, 2048, replace=False), np.arange(n - 256, n)])
    sx = s.cpu().numpy().T[idx].astype(np.float64)
    m64, s64 = mean.cpu().numpy().astype(np.float64), std.cpu().numpy().astype(np.float64)
    p64 = {k: v.astype(np.float64) for k, v in p.items()}
    if kind == "vail":
        ex = eps.cpu().numpy().T[idx].astype(np.float64) if e is not None else np.zeros((len(idx), 128))
        d64, mu, lv = L.vail_forward(p64, sx, ex, m64, s64)
        assert_close(fw["kl"].cpu().numpy()[idx], L.vdb_kl(mu, lv), "kl vs float64 oracle")
    else:
        d64 = L.gail_forward(p64, sx, m64, s64)
    assert_close(d.cpu().numpy()[idx], d64, "logit vs float64 oracle")
    assert_close(r.cpu().numpy()[idx], _reward(d64), "reward vs float64 oracle")
    assert np.isfinite(r.cpu().numpy()).all()


@pytest.mark.parametrize("n_in", WIDTHS)
@pytest.mark.parametrize("n", [1, 127, 129, 65536, 160001])
@pytest.mark.parametrize("kind", ["vail", "vail_no_eps", "gail"])
def test_discriminator_widths_vs_oracle_and_torch(kind, n, n_in):
    """Ragged tiles, one tile per CTA and several; VAIL with and without eps; logit, reward and KL."""
    _check_forward(kind.split("_")[0], n_in, n, with_eps=kind == "vail", seed=n + n_in)


@pytest.mark.parametrize("kind", ["vail", "gail"])
def test_discriminator_width_48_one_million_samples(kind):
    _check_forward(kind, 48, 1 << 20, with_eps=True, seed=48)


@pytest.mark.parametrize("n_in", WIDTHS)
@pytest.mark.parametrize("kind", ["vail", "gail"])
def test_no_read_beyond_the_inputs(kind, n_in):
    """s is a row slice of a larger buffer whose rows beyond n_in and whose padding columns (ld > n) are NaN, and so is
    the standardiser snapshot beyond n_in: the outputs are finite and equal to those of the unpadded call."""
    import torch
    from olympics_mujoco_b200 import _lib
    from olympics_mujoco_b200 import kernels as Kn
    lib = _lib.load()
    n, ld = 1000, 1037
    disc = Kn.Discriminator(kind, _params(kind, n_in, seed=3))
    s, mean, std, eps = _inputs(n_in, n, seed=5)
    e = eps if kind == "vail" else None
    r_ref, d_ref = disc.reward(s, mean, std, eps=e, want_d=True)
    nan = float("nan")
    big = torch.full((n_in + 40, ld), nan, device="cuda")
    big[:n_in, :n] = s
    mean_p, std_p = torch.full((n_in + 40,), nan, device="cuda"), torch.full((n_in + 40,), nan, device="cuda")
    mean_p[:n_in], std_p[:n_in] = mean, std
    eps_p = None
    if e is not None:
        eps_p = torch.full((128, ld), nan, device="cuda")
        eps_p[:, :n] = e
    r, d = torch.full((ld,), nan, device="cuda"), torch.full((ld,), nan, device="cuda")
    P = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(lib.om_disc_reward(disc.handle, P(big[:n_in]), P(mean_p), P(std_p), P(eps_p), n, ld, P(r), P(d), st))
    torch.cuda.synchronize()
    assert bool(torch.isfinite(r[:n]).all()) and bool(torch.isfinite(d[:n]).all())
    assert torch.equal(r[:n], r_ref) and torch.equal(d[:n], d_ref)
    assert bool(torch.isnan(r[n:]).all()) and bool(torch.isnan(d[n:]).all()), "wrote into the padding columns"


def test_refusals(disc_knob):
    """n_in outside 1..64 is refused at create time; a kernel variant forced through a knob takes 32 inputs only and
    refuses another width without launching."""
    import torch
    from olympics_mujoco_b200 import kernels as Kn
    from olympics_mujoco_b200._lib import OmError
    for kind in ("vail", "gail"):
        for n_in in (0, 65):
            p = _params(kind, max(n_in, 1))
            p["w1"] = np.zeros((p["w1"].shape[0], n_in), np.float32)
            with pytest.raises(OmError, match="n_in"):
                Kn.Discriminator(kind, p)
    s, mean, std, eps = _inputs(48, 300, seed=1)
    vail, gail = Kn.Discriminator("vail", _params("vail", 48)), Kn.Discriminator("gail", _params("gail", 48))
    want_v = vail.forward(s, mean, std, eps=eps)["logit"].clone()
    for knob, value in (("disc_vail2", 0), ("disc_vail2", 1), ("disc_vail2", 3), ("disc_vail2", 5), ("disc_vail2", 6),
                        ("disc_vail2", 7)):
        disc_knob(knob, value)
        with pytest.raises(OmError, match="32 inputs only"):
            vail.reward(s, mean, std, eps=eps)
        disc_knob(knob, -1)
    disc_knob("disc_pg2", 0)
    with pytest.raises(OmError, match="32 inputs only"):
        gail.reward(s, mean, std)
    disc_knob("disc_pg2", -1)
    # forcing the default kernels is not a refusal
    disc_knob("disc_vail2", 4)
    assert torch.equal(vail.forward(s, mean, std, eps=eps)["logit"], want_v)
    disc_knob("disc_pg2", 1)
    gail.reward(s, mean, std)
    torch.cuda.synchronize()


VARIANTS = dict(default=(dict(), 32), carry=(dict(hold_weight=True, weight_mass=1.0), 32),
                noback=(dict(disable_back_joint=True), 30), arms=(dict(disable_arms=False), 48),
                arms_noback=(dict(disable_arms=False, disable_back_joint=True), 46))


def _variant_env(name, n_envs):
    import olympics_mujoco_b200 as om
    from olympics_mujoco_b200 import mjcf, synthetic
    from oracle import h1 as OH
    kw, _ = VARIANTS[name]
    model = mjcf.unitree_h1_variant(**kw) if kw else mjcf.load_builtin("unitree_h1")
    keys = OH.keys(model)
    d = synthetic.h1_walk_dataset(n_traj=3, t_raw=80, seed=4, model=model)
    tab = np.stack([np.asarray(d[k]).reshape(3, 80) for k in keys])
    tab[2:] = tab[2:].astype(np.float32).astype(np.float64)
    return om.LocoEnvBase.make("UnitreeH1.walk.real", n_envs=n_envs, traj_params=dict(table=tab), seed=9, **kw)


@pytest.mark.parametrize("name", list(VARIANTS))
def test_learner_hooks_on_played_variant_observations(name):
    """Each variant plays a short episode; its kinematic observations go through make_discrim_reward (VAIL and GAIL) and
    one VAIL fit_batch against an ExpertDataset masked the same way, restated step by step with the oracle."""
    import torch
    from olympics_mujoco_b200.learners import DiscriminatorReward, ExpertDataset, VDBLoss
    from oracle import learner as L
    _, width = VARIANTS[name]
    env = _variant_env(name, n_envs=4)
    mask = np.asarray(env.get_kinematic_obs_mask())
    assert len(mask) == width
    obs = env.play_trajectory_from_velocity(1, 30, render=False, want=("obs",))["obs"]       # [T, C, n]
    states = obs[:, torch.as_tensor(mask, device="cuda"), :].permute(1, 0, 2).reshape(width, -1).contiguous()
    n = states.shape[1]
    s_np = states.cpu().numpy().T.astype(np.float64)
    rng = np.random.default_rng(width)
    eps = rng.normal(0, 1, (2 * n, 128)).astype(np.float32)
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32), device="cuda")
    for kind in ("vail", "gail"):
        p = _params(kind, width, seed=11)
        p64 = {k: v.astype(np.float64) for k, v in p.items()}
        dr = DiscriminatorReward(kind, p, seed=0)
        ref_std = L.Standardizer()
        for half in (s_np[: n // 2], s_np[n // 2:]):
            e = eps[: len(half)]
            r = dr.make_discrim_reward(t(half.T), eps=t(e.T) if kind == "vail" else None)
            ref_std.update_mean_std(half)
            torch.cuda.synchronize()
            assert_close(dr.standardizer.mean.cpu().numpy(), ref_std.mean, "standardiser mean", rtol=1e-9, atol=1e-12)
            assert_close(dr.standardizer.std.cpu().numpy(), ref_std.std, "standardiser std", rtol=1e-9, atol=1e-12)
            m32 = ref_std.mean.astype(np.float32).astype(np.float64)
            s32 = ref_std.std.astype(np.float32).astype(np.float64)
            if kind == "vail":
                d64, _, _ = L.vail_forward(p64, half, e, m32, s32)
            else:
                d64 = L.gail_forward(p64, half, m32, s32)
            assert_close(r.cpu().numpy(), _reward(d64), f"{kind} reward")
    # one discriminator-fit epoch on the played batch
    ds = env.create_dataset()
    ex = ExpertDataset(ds, state_mask=mask, seed=4)
    full = np.concatenate([np.asarray(ds["states"]), np.asarray(ds["next_states"])[-1:]])[:, mask].astype(np.float32)
    p = _params("vail", width, seed=12)
    dr = DiscriminatorReward("vail", p, seed=0)
    vl = VDBLoss(0.5, 1e-5)
    value, st, batch = dr.fit_batch(states, ex, vl, eps=t(eps.T))
    torch.cuda.synchronize()
    idx = L.expert_indices(4, 0, n, ex.n)
    inputs = np.concatenate([s_np.astype(np.float32), full[idx]])
    assert np.array_equal(batch["inputs"].cpu().numpy().T, inputs)
    sd = L.Standardizer()
    sd.update_mean_std(inputs)
    sd.forward(inputs)
    mean32, std32 = sd.mean.astype(np.float32).astype(np.float64), sd.std.astype(np.float32).astype(np.float64)
    d64, mu, lv = L.vail_forward({k: v.astype(np.float64) for k, v in p.items()}, inputs, eps, mean32, std32)
    assert_close(batch["logit"].cpu().numpy(), d64, "fit logit")
    assert_close(batch["kl"].cpu().numpy(), L.vdb_kl(mu, lv), "fit kl")
    tgt = np.concatenate([np.zeros(n), np.ones(n)])
    want, beta = L.vdb_loss(d64, L.vdb_kl(mu, lv), tgt, 0.1, 0.5, 1e-5)
    assert abs(value - want) < 1e-5 * abs(want) and abs(vl.beta - beta) < 1e-9
    sig = 1 / (1 + np.exp(-d64))
    assert abs(st["d_out_gen"] - sig[:n].mean()) < 1e-5 and abs(st["d_out_exp"] - sig[n:].mean()) < 1e-5
    assert_close(batch["dlogit"].cpu().numpy(), (sig - tgt) / (2 * n), "bce gradient", rtol=1e-4, atol=1e-8)
    run = dr.standardizer.running.cpu().numpy()
    assert_close(run[:width], sd._sum, "running sum", rtol=1e-12, atol=1e-9)
    assert_close(run[width:2 * width], sd._sumsq, "running sum of squares", rtol=1e-12, atol=1e-9)
