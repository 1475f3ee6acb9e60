"""CPU: the per-env carried weight of UnitreeH1 -- the generated FK with the weight's mass as a runtime argument (compiled
as plain C++) against the float64 oracle, the host side of the per-env draw contract, and the constructor checks."""
import ctypes
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest

from conftest import ROOT, assert_close


def _carry(weight):
    from olympics_mujoco_b200 import mjcf
    return mjcf.unitree_h1_variant(hold_weight=True, weight_mass=weight)


def test_runtime_mass_fk_matches_oracle_on_host():
    """One generated function serves every weight: at body masses 0.2, 2, 10, 20 (the valid weights) and an unlisted 7.3
    it agrees with the oracle run on the model that has that mass; the emitted code folds no weight mass."""
    from olympics_mujoco_b200 import codegen, mjcf, synthetic
    from oracle import h1 as OH
    from oracle import kinematics as K
    base = _carry(mjcf.H1_VALID_WEIGHTS[0])
    body = base.body_id("weight")
    src = codegen.generate_fk(base, "om_fk_h1_carry_env", env_mass_body=body)
    body_of = lambda s: s.split("\n", 1)[1]               # past the header line (it names the tables' fingerprint)
    assert "env_mass" in src
    assert body_of(src) == body_of(codegen.generate_fk(_carry(5.0), "om_fk_h1_carry_env", env_mass_body=body))
    assert codegen.generate_fk(base, "f") == codegen.generate_fk(base, "f", env_mass_body=None)
    d = Path(tempfile.mkdtemp())
    (d / "fk_h1_carry_env.cuh").write_text(src)
    subprocess.check_call(["g++", "-O1", "-shared", "-fPIC", "-I", str(d), "-I", str(ROOT / "olympics_mujoco_b200/csrc"),
                           str(ROOT / "tests/host/fk_env_mass_harness.cpp"), "-o", str(d / "h.so")])
    lib = ctypes.CDLL(str(d / "h.so"))
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    data = synthetic.h1_walk_dataset(n_traj=2, t_raw=300, seed=5, model=base)
    sample = np.stack([data[k] for k in OH.keys(base)], axis=1)[::3]
    qpos, qvel = OH.set_sim_state(base, sample)
    q32, v32 = np.ascontiguousarray(qpos, np.float32), np.ascontiguousarray(qvel, np.float32)
    n, nb = q32.shape[0], base.nbody
    for mass in (0.2, 2.0, 10.0, 20.0, 7.3):
        model = _carry(mass / 2)
        m32 = np.full(n, mass, np.float32)
        xp = np.zeros((n, nb, 3), np.float32); xq = np.zeros((n, nb, 4), np.float32)
        sp = np.zeros((n, model.nsite, 3), np.float32); cv = np.zeros((n, nb, 6), np.float32)
        cm = np.zeros((n, 3), np.float32)
        lib.host_fk_h1_carry_env(P(q32), P(v32), P(m32), n, P(xp), P(xq), P(sp), P(cv), P(cm))
        ref = K.forward(model, q32.astype(np.float64), v32.astype(np.float64))
        assert_close(xp, ref["xpos"], f"xpos {mass}"); assert_close(xq, ref["xquat"], f"xquat {mass}")
        assert_close(sp, ref["site_xpos"], f"site_xpos {mass}"); assert_close(cv, ref["cvel"], f"cvel {mass}")
        assert_close(cm, ref["subtree_com"][:, 1], f"com {mass}")
    # the mass moves the COM: a different mass is not within tolerance of the oracle
    other = K.forward(_carry(10.0), q32.astype(np.float64), v32.astype(np.float64))
    assert np.abs(other["subtree_com"][:, 1] - cm).max() > 1e-3


def _shared_sequence(seed, env_id0, resets, n_models, random):
    """What LocoEnvBase._next_model picks for a shared env object (_current_model_idx after each reset)."""
    from olympics_mujoco_b200.utils.philox import STREAM_MODEL_RESET, philox_randint
    idx, out = 0, []
    for k in range(resets):
        idx = philox_randint(seed, env_id0, k, STREAM_MODEL_RESET, n_models) if random else (idx + 1) % n_models
        out.append(idx)
    return out


@pytest.mark.parametrize("random", [True, False])
def test_per_env_draw_contract_on_host(random):
    """env_model_draw: the documented formula; env 0 of the first shard == the shared object's picks; a single env (the
    reference's n_envs=None shape) == shared mode; the draw depends on the global env id only (sharding-independent);
    a batch holds every weight."""
    from olympics_mujoco_b200.utils.philox import STREAM_MODEL_RESET, env_model_draw, philox_randint
    seed, n, resets = 11, 64, 9
    table = np.array([[env_model_draw(seed, e, k, 4, random) for e in range(n)] for k in range(resets)])
    for k in range(resets):
        for e in (0, 5, 63):
            want = philox_randint(seed, e, k, STREAM_MODEL_RESET, 4) if random else (e + k + 1) % 4
            assert table[k, e] == want
    assert table[:, 0].tolist() == _shared_sequence(seed, 0, resets, 4, random)
    # a one-env object (n_envs=None) behaves like the shared object: at env_id0 0, and in random mode at any global id
    # (round robin starts every env at its own offset: (env_id0 + k + 1) mod 4)
    for env_id0 in ((0, 3, 40) if random else (0,)):
        assert [env_model_draw(seed, env_id0, k, 4, random) for k in range(resets)] == \
            _shared_sequence(seed, env_id0, resets, 4, random)
    # two shards [0, 24) and [24, 64): local env e of shard s is global env env_id0 + e
    shards = np.concatenate([[[env_model_draw(seed, env_id0 + e, k, 4, random) for e in range(size)]
                              for k in range(resets)] for env_id0, size in ((0, 24), (24, 40))], axis=1)
    assert np.array_equal(shards, table)
    assert all(set(row) == {0, 1, 2, 3} for row in table)
    if random:
        assert len({tuple(table[:, e]) for e in range(n)}) > n // 2


def test_per_env_weight_constructor_checks():
    """per_env_weight needs the carry task's list of weights: without hold_weight, or with a fixed weight, it is rejected
    before any device work."""
    import olympics_mujoco_b200 as om
    from olympics_mujoco_b200.environments.unitree_h1 import UnitreeH1
    with pytest.raises(ValueError):
        UnitreeH1(per_env_weight=True, n_envs=4)
    with pytest.raises(ValueError):
        UnitreeH1(hold_weight=True, weight_mass=5.0, per_env_weight=True, n_envs=4)
    with pytest.raises(ValueError):
        om.LocoEnvBase.make("UnitreeH1.walk.real", n_envs=4, per_env_weight=True)
