"""CPU: host-side logic -- MJCF compiler, code generator, Trajectory load path, C-ABI surface."""
import ctypes
import re
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, a3_random_states, assert_close


def test_library_exports_every_declared_symbol():
    """The shared library loads and exports every function include/om_b200.h declares (no compute calls)."""
    from olympics_mujoco_b200 import _lib
    from olympics_mujoco_b200 import build
    build.build(verbose=False)
    header = (ROOT / "include" / "om_b200.h").read_text()
    declared = set(re.findall(r"\b(om_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 20
    lib = ctypes.CDLL(str(_lib.LIB_PATH))
    missing = [s for s in sorted(declared) if not hasattr(lib, s)]
    assert not missing, f"declared but not exported: {missing}"
    assert declared == set(_lib.PROTOTYPES), "ctypes prototypes out of sync with the header"
    assert _lib.load().om_abi_version() == 2


def test_compute_entry_points_fail_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from olympics_mujoco_b200 import _lib, mjcf
    from olympics_mujoco_b200 import kernels as Kn
    with pytest.raises(_lib.OmError, match="no CUDA device"):
        Kn.DeviceModel(mjcf.load_builtin("unitree_h1"))
    with pytest.raises(_lib.OmError):
        Kn.DeviceTrajectory(np.zeros((34, 1, 5)), 4)
    with pytest.raises(_lib.OmError, match="CUDA tensor"):
        Kn.h1_has_fallen(torch.zeros((4, 3)))


def test_generated_fk_matches_oracle_on_host(h1_model, a3_model, h1_states):
    """The code generator's output, compiled as plain C++ (fp32), agrees with the float64 oracle: checks the
    generator in a container without a GPU.  The harness is test-only; the product has no CPU path."""
    from olympics_mujoco_b200 import codegen
    from oracle import kinematics as K
    d = Path(tempfile.mkdtemp())
    (d / "fk_unitree_h1.cuh").write_text(codegen.generate_fk(h1_model, "om_fk_unitree_h1"))
    (d / "fk_stick_figure_a3.cuh").write_text(codegen.generate_fk(a3_model, "om_fk_stick_figure_a3"))
    (d / "fk_pos_stick_figure_a3.cuh").write_text(codegen.generate_fk_pos(a3_model, "om_fk_pos_stick_figure_a3"))
    parts = codegen.split_parts(h1_model, 3)
    assert sorted(b for p in parts for b in p) == list(range(h1_model.nbody))      # a partition of the bodies
    (d / "fk_unitree_h1_parts.cuh").write_text("".join(
        codegen.generate_fk(h1_model, f"om_fk_unitree_h1_part{k}", part=p) for k, p in enumerate(parts)))
    parts_a3 = codegen.split_parts(a3_model, 3)
    assert sorted(b for p in parts_a3 for b in p) == list(range(a3_model.nbody))
    (d / "fk_stick_figure_a3_parts.cuh").write_text("".join(
        codegen.generate_fk(a3_model, f"om_fk_stick_figure_a3_part{k}", part=p) for k, p in enumerate(parts_a3)))
    subprocess.check_call(["g++", "-O1", "-shared", "-fPIC", "-I", str(d), "-I", str(ROOT / "olympics_mujoco_b200/csrc"),
                           str(ROOT / "tests/host/fk_host_harness.cpp"),
                           "-o", str(d / "h.so")])
    lib = ctypes.CDLL(str(d / "h.so"))
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    for model, fn, (q, v) in ((h1_model, "host_fk_h1", h1_states), (h1_model, "host_fk_h1_parts", h1_states),
                              (a3_model, "host_fk_a3", a3_random_states(a3_model, 128, seed=8)),
                              (a3_model, "host_fk_a3_parts", a3_random_states(a3_model, 128, seed=10))):
        n = q.shape[0]
        q32, v32 = np.ascontiguousarray(q, np.float32), np.ascontiguousarray(v, np.float32)
        xp = np.zeros((n, model.nbody, 3), np.float32); xq = np.zeros((n, model.nbody, 4), np.float32)
        sp = np.zeros((n, model.nsite, 3), np.float32); sm = np.zeros((n, model.nsite, 3, 3), np.float32)
        cv = np.zeros((n, model.nbody, 6), np.float32); cm = np.zeros((n, 3), np.float32)
        getattr(lib, fn)(P(q32), P(v32), n, P(xp), P(xq), P(sp), P(sm), P(cv), P(cm))
        ref = K.forward(model, q32.astype(np.float64), v32.astype(np.float64))
        assert_close(xp, ref["xpos"], "xpos"); assert_close(xq, ref["xquat"], "xquat")
        assert_close(sp, ref["site_xpos"], "site_xpos"); assert_close(sm, ref["site_xmat"], "site_xmat")
        assert_close(cv, ref["cvel"], "cvel"); assert_close(cm, ref["subtree_com"][:, 1], "com")
    # matrix-chain variant used by the A3 task kernels: positions vs the oracle, point velocities vs the quaternion chain
    q, v = a3_random_states(a3_model, 256, seed=9)
    n = q.shape[0]
    q32, v32 = np.ascontiguousarray(q, np.float32), np.ascontiguousarray(v, np.float32)
    xp = np.zeros((n, 17, 3), np.float32); xq = np.zeros((n, 17, 4), np.float32); sp = np.zeros((n, 2, 3), np.float32)
    vp = np.zeros((n, 17, 6), np.float32); vq = np.zeros((n, 17, 6), np.float32)
    lib.host_fk_a3_pos(P(q32), P(v32), n, P(xp), P(xq), P(sp), P(vp), P(vq))
    ref = K.forward(a3_model, q32.astype(np.float64), v32.astype(np.float64))
    assert_close(xp[:, 1:], ref["xpos"][:, 1:], "xpos (matrix chain)"); assert_close(sp, ref["site_xpos"], "site_xpos (matrix chain)")
    assert_close(xq[:, 1], ref["xquat"][:, 1], "root xquat (matrix chain)")
    assert np.abs(vq[:, 1:]).max() > 1.0
    assert_close(vp[:, 1:], vq[:, 1:], "vel_p (matrix chain vs quaternion chain)", rtol=1e-5, atol=2e-5)


def test_mjcf_compiler_on_a_small_model(tmp_path):
    from olympics_mujoco_b200 import mjcf
    xml = """<mujoco model="toy"><compiler angle="radian" autolimits="true"/>
      <default><default class="c"><joint damping="1"/><geom type="capsule" density="500"/></default></default>
      <worldbody><body name="a" pos="0 0 1" childclass="c"><freejoint name="root"/>
        <geom type="sphere" size="0.1"/>
        <body name="b" pos="0.2 0 0" quat="2 0 0 0"><joint name="j1" axis="0 2 0" range="-1 1" pos="0 0 0.05"/>
          <geom fromto="0 0 0 0 0 -0.4" size="0.05"/><site name="tip" pos="0 0 -0.4"/>
          <body name="c" pos="0 0 -0.4"><joint name="j2" type="slide" axis="1 0 0"/><inertial pos="0 0 0.1" mass="2"/></body>
        </body></body></worldbody>
      <actuator><motor name="m1" joint="j1" gear="3"/></actuator></mujoco>"""
    p = tmp_path / "toy.xml"
    p.write_text(xml)
    m = mjcf.compile_mjcf(p)
    assert (m.nbody, m.njnt, m.nq, m.nv, m.nsite, m.nu) == (4, 3, 9, 8, 1, 1)
    assert list(m.jnt_type) == [mjcf.JNT_FREE, mjcf.JNT_HINGE, mjcf.JNT_SLIDE]
    assert_close(m.body_quat[2], [1, 0, 0, 0], "quat normalised", rtol=0, atol=1e-15)
    assert_close(m.jnt_axis[1], [0, 1, 0], "axis normalised", rtol=0, atol=1e-15)
    assert bool(m.jnt_limited[1]) and not bool(m.jnt_limited[2])
    r, h = 0.05, 0.2
    assert_close(m.body_mass[2], 500 * (np.pi * r * r * 2 * h + 4 / 3 * np.pi * r ** 3), "capsule mass", rtol=1e-12, atol=0)
    assert_close(m.body_ipos[2], [0, 0, -0.2], "capsule com", rtol=0, atol=1e-15)
    assert_close(m.body_mass[1], 500 * 4 / 3 * np.pi * 1e-3, "sphere mass (class density)", rtol=1e-12, atol=0)
    assert_close(m.qpos0, [0, 0, 1, 1, 0, 0, 0, 0, 0], "qpos0", rtol=0, atol=0)
    rt = mjcf.KinematicModel.from_dict(m.to_dict())
    assert rt.body_names == m.body_names and np.array_equal(rt.jnt_range, m.jnt_range)
    with pytest.raises(ValueError):
        mjcf.compile_mjcf(p, remove_joints=["nope"])


def test_trajectory_load_path_matches_reference_class():
    """Range clipping, splitting and cubic re-sampling reproduce the reference's Trajectory bit for bit."""
    from olympics_mujoco_b200 import mjcf
    from olympics_mujoco_b200.utils.trajectory import Trajectory, resample_table
    z = np.load(GOLDEN / "trajectory_ref.npz")
    data = {k[3:]: z[k] for k in z.files if k.startswith("in_")}
    model = mjcf.load_builtin("unitree_h1")
    assert np.array_equal(resample_table(data, model), z["table"])
    keys = [k for k in data if k != "split_points"]
    tr = Trajectory(keys=keys, low=z["low"][2:], high=z["high"][2:], joint_pos_idx=np.arange(17), traj_files=dict(data),
                    traj_dt=1 / 500, control_dt=1 / 100, clip_trajectory_to_joint_ranges=True, warn=False)
    assert tr.trajectory_length == 50 and tr.number_of_trajectories == 3
    assert np.array_equal(tr.split_points, z["split_points"])
    ds = tr.create_dataset(ignore_keys=["q_pelvis_tx", "q_pelvis_tz"])
    for k in ("states", "next_states", "absorbing", "last"):
        assert np.array_equal(ds[k], z["ds_" + k])
    # ragged input is rejected exactly like the reference (trajectory.py:207-224)
    bad = dict(data)
    bad["split_points"] = np.array([0, 100, 750])
    with pytest.raises(AssertionError, match="equal length"):
        Trajectory(keys=keys, low=z["low"][2:], high=z["high"][2:], joint_pos_idx=np.arange(17), traj_files=bad, warn=False)
    with pytest.raises(AssertionError):
        Trajectory(keys=keys, low=None, high=None, joint_pos_idx=np.arange(17))


def test_env_name_grammar_and_registry():
    import olympics_mujoco_b200 as om
    assert "UnitreeH1" in om.LocoEnvBase.list_registered_loco_mujoco()
    names = om.LocoEnvBase.get_all_task_names()
    assert "UnitreeH1.walk.real" in names and "UnitreeH1.carry.perfect" not in names
    with pytest.raises(ValueError, match="does not exit"):
        om.LocoEnvBase.make("UnitreeH1.fly.real")
    with pytest.raises(ValueError, match="does not exit"):
        om.LocoEnvBase.make("UnitreeH1.walk.imaginary")
    with pytest.raises(KeyError):
        om.LocoEnvBase.make("Nope.walk")


def test_synthetic_dataset_is_non_terminal(h1_model):
    from olympics_mujoco_b200 import synthetic
    from oracle import h1 as OH
    d = synthetic.h1_walk_dataset(n_traj=2, t_raw=500, seed=11, model=h1_model)
    keys = OH.keys(h1_model)
    assert [k for k in d if k != "split_points"] == keys
    obs = np.stack([d[k] for k in keys], axis=1)[:, 2:]
    assert not OH.has_fallen(obs).any()
    for i, j in enumerate(OH.spec_joints(h1_model)):
        jid = h1_model.jnt_names.index(j)
        if h1_model.jnt_limited[jid]:
            lo, hi = h1_model.jnt_range[jid]
            assert d["q_" + j].min() >= lo and d["q_" + j].max() <= hi


def test_a3_task_device_functions_on_host(a3_model):
    """The A3 step-tail device functions (csrc/om_a3_task.cuh, fp32), compiled as plain C++, against the fixture
    produced by the reference's own WalkingTask: integer state and done flags bit-exact, observations and
    reward terms within 1e-5.  Checks the kernel arithmetic in a container without a GPU (test-only harness)."""
    import a3_common as A
    from olympics_mujoco_b200 import build
    from oracle import a3 as OA
    build.generate()
    d = Path(tempfile.mkdtemp())
    csrc = ROOT / "olympics_mujoco_b200" / "csrc"
    subprocess.check_call(["g++", "-O1", "-shared", "-fPIC", "-I", str(csrc), str(ROOT / "tests/host/a3_host_harness.cpp"),
                           "-o", str(d / "a3.so")])
    lib = ctypes.CDLL(str(d / "a3.so"))
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    gold = A.golden()
    lut = np.ascontiguousarray(A.lut6())
    consts = (P(lut), OA.PERIOD, OA.DELAY_FRAMES, ctypes.c_double(0.2), ctypes.c_double(0.80), ctypes.c_double(0.01),
              ctypes.c_float(a3_model.total_mass * 9.8 * 0.5))
    n_env, T = gold["step_done"].shape
    it = float(gold["iteration_count"])
    h = float(np.clip((it - 3000) / 8000, 0, 1) * 0.1)
    init = OA.init_qpos().astype(np.float32)
    for e in range(n_env):
        q, v = np.zeros(25, np.float32), np.zeros(24, np.float32)
        ints, seq, obs0 = np.zeros(7, np.int32), np.zeros(80, np.float32), np.zeros(41, np.float32)
        lib.host_a3_reset(*consts, P(init), ctypes.c_ulonglong(int(gold["seed"])), e, 0, ctypes.c_float(h), P(q), P(v),
                          P(ints), P(seq), P(obs0))
        assert list(ints) == list(gold["reset_ints"][e])
        assert_close(q, gold["reset_qpos"][e], "reset qpos"); assert_close(v, gold["reset_qvel"][e], "reset qvel")
        assert_close(seq.reshape(20, 4), gold["reset_sequence"][e], "sequence")
        ref_obs0, ref_obs, ref_total = A.oracle_obs(a3_model, gold, e, upto=T if e < 2 else 40)
        assert_close(obs0, ref_obs0, "reset obs")
        # step replay from the REFERENCE's reset state (so that the two checks are independent)
        ints = gold["reset_ints"][e].astype(np.int32)
        seq = np.ascontiguousarray(gold["reset_sequence"][e].reshape(-1), np.float32)
        qpos, qvel = np.ascontiguousarray(gold["step_qpos"][e]), np.ascontiguousarray(gold["step_qvel"][e])
        con = np.ascontiguousarray(A.contact4(gold["step_contact"][e]))
        obs, terms = np.zeros((T, 41), np.float32), np.zeros((T, 6), np.float32)
        reward, done = np.zeros(T, np.float32), np.zeros(T, np.uint8)
        # per-step state trace: run the harness one step at a time
        trace = []
        for t in range(T):
            lib.host_a3_rollout(*consts, P(qpos[t]), P(qvel[t]), P(con[t]), 1, P(ints), P(seq), P(obs[t]), P(terms[t]),
                                P(reward[t:t + 1]), P(done[t:t + 1]))
            trace.append(ints.copy())
        np.testing.assert_array_equal(np.array(trace), gold["step_ints"][e])
        np.testing.assert_array_equal(done.astype(bool), gold["step_done"][e])
        assert_close(terms, gold["step_terms"][e], "terms")
        assert_close(reward, gold["step_terms"][e].sum(axis=1), "reward")
        assert_close(obs[:, 33:], gold["step_goal"][e], "goal steps")
        assert_close(obs[:len(ref_obs)], ref_obs, "obs")
        # the multi-step entry (T steps in one call) gives the same answer as T single steps
        ints2 = gold["reset_ints"][e].astype(np.int32)
        obs2, terms2 = np.zeros_like(obs), np.zeros_like(terms)
        reward2, done2 = np.zeros_like(reward), np.zeros_like(done)
        lib.host_a3_rollout(*consts, P(qpos), P(qvel), P(con), T, P(ints2), P(seq), P(obs2), P(terms2), P(reward2), P(done2))
        assert np.array_equal(obs2, obs) and np.array_equal(done2, done) and np.array_equal(ints2, trace[-1])
        # the time-parallel split (what a3_feat_kernel + a3_seq_kernel compute) agrees with the fused path
        ints3 = gold["reset_ints"][e].astype(np.int32)
        obs3, terms3 = np.zeros_like(obs), np.zeros_like(terms)
        reward3, done3 = np.zeros_like(reward), np.zeros_like(done)
        lib.host_a3_rollout_split(*consts, P(qpos), P(qvel), P(con), T, P(ints3), P(seq), P(obs3), P(terms3), P(reward3), P(done3))
        assert np.array_equal(ints3, trace[-1]) and np.array_equal(done3, done)
        assert_close(obs3, obs, "split obs", rtol=1e-6, atol=1e-6); assert_close(terms3, terms, "split terms", rtol=1e-6, atol=1e-6)
        assert_close(reward3, reward, "split reward", rtol=1e-6, atol=1e-6)
    # candidate-bit state machine under stress: short delays and a radius that makes "near" frequent or permanent, so the
    # target advances every few steps, the candidate chain clamps at the last target and calls split into sub-calls
    e = 0
    qpos, qvel = np.ascontiguousarray(gold["step_qpos"][e]), np.ascontiguousarray(gold["step_qvel"][e])
    con = np.ascontiguousarray(A.contact4(gold["step_contact"][e]))
    seq = np.ascontiguousarray(gold["reset_sequence"][e].reshape(-1), np.float32)
    advanced = 0
    for delay, radius in ((0, 5.0), (1, 5.0), (2, 0.9), (5, 0.6), (30, 5.0), (7, 0.35)):
        c2 = (P(lut), OA.PERIOD, delay, ctypes.c_double(radius), ctypes.c_double(0.80), ctypes.c_double(0.01),
              ctypes.c_float(a3_model.total_mass * 9.8 * 0.5))
        for start in (gold["reset_ints"][e].astype(np.int32), np.array([3, 4, 5, 1, 1, 20, 1], np.int32),
                      np.array([7, 2, 3, max(delay - 1, 0), 1, 20, 1], np.int32), np.array([7, 18, 19, delay + 3, 1, 20, 1], np.int32)):
            ia, ib = start.copy(), start.copy()
            oa, ta = np.zeros((T, 41), np.float32), np.zeros((T, 6), np.float32)
            ra, da = np.zeros(T, np.float32), np.zeros(T, np.uint8)
            ob, tb, rb, db = np.zeros_like(oa), np.zeros_like(ta), np.zeros_like(ra), np.zeros_like(da)
            lib.host_a3_rollout(*c2, P(qpos), P(qvel), P(con), T, P(ia), P(seq), P(oa), P(ta), P(ra), P(da))
            lib.host_a3_rollout_split(*c2, P(qpos), P(qvel), P(con), T, P(ib), P(seq), P(ob), P(tb), P(rb), P(db))
            assert np.array_equal(ia, ib), (delay, radius, ia, ib)
            assert np.array_equal(da, db)
            assert_close(ob, oa, "stress obs", rtol=1e-6, atol=1e-6); assert_close(rb, ra, "stress reward", rtol=1e-6, atol=1e-6)
            advanced += int(ia[1] != start[1])
    assert advanced >= 10
    # bounded-range sin / cos / tan (om_math.cuh) against float64 libm: joint-angle range, many periods, the libm fallback
    rng = np.random.default_rng(21)
    xs = np.concatenate([rng.uniform(-3.2, 3.2, 200000), rng.uniform(-1000, 1000, 100000), rng.uniform(-1e5, 1e5, 50000),
                         [0.0, -0.0, 1e6, -3e7, np.pi / 2, -np.pi]]).astype(np.float32)
    sn, cs, tn = (np.zeros(xs.size, np.float32) for _ in range(3))
    lib.host_trig(P(xs), xs.size, P(sn), P(cs), P(tn))
    x64 = xs.astype(np.float64)
    assert np.abs(sn - np.sin(x64)).max() < 1.5e-7 and np.abs(cs - np.cos(x64)).max() < 1.5e-7
    small = (np.abs(x64) <= 0.7854) & (np.abs(x64) > 1e-30)
    assert np.abs(tn[small] / np.tan(x64[small]) - 1.0).max() < 3e-7
    small = np.abs(x64) <= 0.7854
    assert_close(tn[~small], np.tan(x64[~small]), "tan fallback", rtol=2e-6, atol=1e-6)
    ya = np.concatenate([rng.normal(0, 1, 300000), [0.0, -0.0, 0.0, 1.0, -1.0, 1e-20, 3.0, -0.0]]).astype(np.float32)
    xa = np.concatenate([rng.normal(0, 1, 300000), [1.0, -1.0, 0.0, 0.0, 0.0, 1e-25, -1e-20, -2.0]]).astype(np.float32)
    ra = np.zeros(ya.size, np.float32)
    lib.host_atan2(P(ya), P(xa), ya.size, P(ra))
    assert np.abs(ra - np.arctan2(ya.astype(np.float64), xa.astype(np.float64))).max() < 4e-7        # 1.3 ulp at pi
    # closed-form root roll / pitch quaternion against the literal quat2euler -> euler2quat path and the float64 oracle:
    # random orientations of any scale and sign, yaw near +-pi, pitch up to 80 degrees
    from oracle import tf3 as T3
    rng = np.random.default_rng(12)
    m = 4000
    roll, pitch, yaw = rng.uniform(-3.1, 3.1, m), rng.uniform(-1.4, 1.4, m), rng.uniform(-np.pi, np.pi, m)
    yaw[:50] = np.pi - 1e-4 * rng.random(50); yaw[50:100] = -np.pi + 1e-4 * rng.random(50)
    quat = np.array([T3.euler2quat(r, p_, y) for r, p_, y in zip(roll, pitch, yaw)])
    quat *= (rng.uniform(0.5, 2.0, m) * rng.choice([-1.0, 1.0], m))[:, None]           # unnormalised, either sign
    q32 = np.ascontiguousarray(quat, np.float32)
    closed, literal = np.zeros((m, 4), np.float32), np.zeros((m, 4), np.float32)
    lib.host_a3_root_orient(P(q32), m, P(closed), P(literal))
    want = np.array([T3.euler2quat(*T3.quat2euler(qq)[:2], 0.0) for qq in q32.astype(np.float64)])
    assert_close(literal, want, "literal path vs oracle", rtol=0, atol=2e-6)
    assert_close(closed, want, "closed form vs oracle", rtol=0, atol=2e-6)
    # candidate pruning: bits of targets that cannot be reached yet are never consulted, for any bit pattern
    rng = np.random.default_rng(5)
    for trial in range(4000):
        delay = int(rng.choice([0, 1, 2, 3, 7, 30]))
        dm = max(delay, 1)
        T_ = int(rng.integers(1, 7 * dm + 1))
        ncand = min(8, 1 + -(-T_ // dm))
        frames0 = int(rng.integers(0, delay + 4))
        p_one = rng.choice([0.2, 0.6, 0.95, 1.0])
        bits = np.packbits((rng.random((T_, 8)) < p_one), axis=1, bitorder="little").ravel().astype(np.uint8)
        bad = lib.host_a3_walk_pruning_check(delay, frames0, int(rng.integers(0, 2)), ncand, T_, P(np.ascontiguousarray(bits)))
        assert bad == -1, (delay, frames0, ncand, T_, bad)


def test_perfect_dataset_conversion_matches_reference_restatement():
    """N4: LocoEnvBase.load_dataset_and_get_traj_files (vectorised) against the loop-for-loop restatement of
    loco_env_base.py:970-1044 (oracle/trajectory.py), with and without velocity integration, and the round trip
    create_dataset -> converter -> Trajectory.  Host logic only (no GPU)."""
    from types import SimpleNamespace
    from olympics_mujoco_b200.environments.loco_env_base import LocoEnvBase
    from oracle import h1 as OH
    from oracle import trajectory as OT
    from olympics_mujoco_b200 import mjcf
    model = mjcf.load_builtin("unitree_h1")
    keys = OH.keys(model)
    rng = np.random.default_rng(4)
    N = 257
    states = rng.normal(0, 1, (N, 32))
    last = np.zeros(N)
    last[[40, 41, 120, 256]] = 1                                   # adjacent episode ends, and the final sample
    fake = SimpleNamespace(obs_helper=SimpleNamespace(observation_spec=[(k, k[2:] if k.startswith("q_") else k[3:], None) for k in keys]),
                           _dataset=None)
    for freq in (None, 100.0):
        got = LocoEnvBase.load_dataset_and_get_traj_files(fake, dict(states=states, last=last), freq=freq)
        ref = OT.load_dataset_and_get_traj_files(states, last, keys, freq=freq)
        assert list(got.keys()) == list(ref.keys())
        for k in ref:
            np.testing.assert_allclose(got[k], ref[k], rtol=0, atol=1e-12, err_msg=k)
    assert list(got["split_points"]) == [0, 41, 42, 121, 257]
    assert got["q_pelvis_tx"][41] == 0.0 and got["q_pelvis_tx"][42] == 0.0 and got["q_pelvis_tx"][121] == 0.0


def test_a3_threshold_decisions_are_float64_exact_on_host(a3_model):
    """A10 target_reached / A12 done: the fp32 device functions decide near their thresholds through a float64 forward
    pass of the same inputs (om_a3_task.cuh: a3_done_height, a3_near_exact).  On adversarial inputs whose margin is a few
    fp32 ulps (1e-8 m; the fp32 chain's own error is 1e-6 m) every flag equals the float64 oracle's -- no excusals."""
    import a3_common as A
    from olympics_mujoco_b200 import build
    from oracle import a3 as OA
    from oracle import kinematics as K
    build.generate()
    d = Path(tempfile.mkdtemp())
    csrc = ROOT / "olympics_mujoco_b200" / "csrc"
    subprocess.check_call(["g++", "-O1", "-shared", "-fPIC", "-I", str(csrc), str(ROOT / "tests/host/a3_host_harness.cpp"),
                           "-o", str(d / "a3.so")])
    lib = ctypes.CDLL(str(d / "a3.so"))
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    cases = A.threshold_cases(a3_model, n=200, seed=3)
    q = np.ascontiguousarray(cases["qpos"])
    n = len(q)
    assert cases["planted"].mean() > 0.95 and np.median(cases["margin"]) < 1e-6
    assert 0.1 < cases["want_done"].mean() < 0.9 and 0.1 < cases["want_reached"].mean() < 0.9
    # the float64 twin of the position FK against the oracle
    ls, rs = np.zeros((n, 3)), np.zeros((n, 3))
    lib.host_a3_sites_f64(P(q), n, P(ls), P(rs))
    fk = K.forward(a3_model, q.astype(np.float64), np.zeros((n, 24)))
    assert_close(ls, fk["site_xpos"][:, a3_model.site_id("lf_force")], "float64 left site", rtol=1e-13, atol=1e-13)
    assert_close(rs, fk["site_xpos"][:, a3_model.site_id("rf_force")], "float64 right site", rtol=1e-13, atol=1e-13)
    lut = np.ascontiguousarray(A.lut6())
    consts = (P(lut), OA.PERIOD, OA.DELAY_FRAMES, ctypes.c_double(0.2), ctypes.c_double(0.80), ctypes.c_double(0.01),
              ctypes.c_float(a3_model.total_mass * 9.8 * 0.5))
    v, con = np.zeros(24, np.float32), np.array([100.0, 100.0, 0.0, 1.0], np.float32)
    for fn in (lib.host_a3_rollout, lib.host_a3_rollout_split):
        got_done, got_reached = np.zeros(n, bool), np.zeros(n, bool)
        for i in range(n):
            ints, seq = cases["ints"][i].copy(), np.ascontiguousarray(cases["seq"][i])
            obs, terms = np.zeros(41, np.float32), np.zeros(6, np.float32)
            rew, dn = np.zeros(1, np.float32), np.zeros(1, np.uint8)
            fn(*consts, P(q[i]), P(v), P(con), 1, P(ints), P(seq), P(obs), P(terms), P(rew), P(dn))
            got_done[i], got_reached[i] = bool(dn[0]), bool(ints[6])
        assert np.array_equal(got_done, cases["want_done"]), np.flatnonzero(got_done != cases["want_done"])
        assert np.array_equal(got_reached, cases["want_reached"]), np.flatnonzero(got_reached != cases["want_reached"])


def _mjcf_of(m):
    """An MJCF document that compiles to the model ``m``: its bodies with explicit inertials, joints with axis, anchor,
    range, limited flag and reference position, sites, and one motor per actuator (slide / hinge joints only)."""
    import xml.etree.ElementTree as ET
    from olympics_mujoco_b200 import mjcf
    f = lambda v: " ".join(repr(float(x)) for x in np.atleast_1d(v))
    types = {v: k for k, v in mjcf._JNT_NAMES.items()}
    root = ET.Element("mujoco", model=m.name)
    ET.SubElement(root, "compiler", angle="radian")
    ET.SubElement(root, "option", timestep=repr(m.timestep))
    elems = {0: ET.SubElement(root, "worldbody")}
    for b in range(m.nbody):                             # body ids are MuJoCo's depth-first order: parents come first
        if b > 0:
            e = elems[b] = ET.SubElement(elems[int(m.body_parentid[b])], "body", name=m.body_names[b],
                                         pos=f(m.body_pos[b]), quat=f(m.body_quat[b]))
            ET.SubElement(e, "inertial", pos=f(m.body_ipos[b]), mass=f(m.body_mass[b]))
        for j in np.flatnonzero(m.jnt_bodyid == b):
            assert int(m.jnt_type[j]) in (mjcf.JNT_SLIDE, mjcf.JNT_HINGE)
            ET.SubElement(elems[b], "joint", name=m.jnt_names[j], type=types[int(m.jnt_type[j])], axis=f(m.jnt_axis[j]),
                          pos=f(m.jnt_pos[j]), range=f(m.jnt_range[j]), limited=str(bool(m.jnt_limited[j])).lower(),
                          ref=f(m.qpos0[m.jnt_qposadr[j]]))
        for s in np.flatnonzero(m.site_bodyid == b):
            ET.SubElement(elems[b], "site", name=m.site_names[s], pos=f(m.site_pos[s]), quat=f(m.site_quat[s]))
    act = ET.SubElement(root, "actuator")
    for a in range(m.nu):
        ET.SubElement(act, "motor", name=m.actuator_names[a], joint=m.actuator_joint[a], gear=f(m.actuator_gear[a]),
                      ctrlrange=f(m.actuator_ctrlrange[a]), ctrllimited=str(bool(m.actuator_ctrllimited[a])).lower())
    return ET.tostring(root, encoding="unicode")


def _assert_same_model(m, ref, what):
    from olympics_mujoco_b200 import mjcf
    for k in mjcf.KinematicModel._ARRAYS:
        assert np.array_equal(np.asarray(getattr(m, k)), np.asarray(getattr(ref, k))), (what, k)
    for k in ("jnt_names", "actuator_names", "actuator_joint", "body_names", "site_names", "nq", "nv"):
        assert getattr(m, k) == getattr(ref, k), (what, k)


def test_unitree_h1_variants_from_shipped_tables(tmp_path):
    """UnitreeH1.py:38-111: every constructor variant (arms, back joint, carried weight) is derived from the shipped tables
    by table-level edits; each equals a compile of the MJCF with the constructor's edits, and its kinematics equal the
    INDEPENDENT checker's fixture.  The shipped tables are the compiles of the reference's h1.xml (tools/gen_models.py):
    unitree_h1_arms.json unedited, unitree_h1.json with the arms removed and re-oriented.  The MJCF compiled here is
    written back out of unitree_h1_arms.json; it is first shown to compile to exactly that table and, with the arm edits,
    to exactly unitree_h1.json."""
    from olympics_mujoco_b200 import mjcf
    from oracle import kinematics as K
    g = np.load(ROOT / "tests" / "golden" / "fk_independent_ref.npz")
    full, default = mjcf.load_builtin("unitree_h1_arms"), mjcf.load_builtin("unitree_h1")
    xml = tmp_path / "h1.xml"
    xml.write_text(_mjcf_of(full))
    _assert_same_model(mjcf.compile_unitree_h1(xml, disable_arms=False), full, "MJCF written out of unitree_h1_arms.json")
    _assert_same_model(mjcf.compile_unitree_h1(xml), default, "arm edits in the MJCF vs the reference's compile")
    _assert_same_model(mjcf.unitree_h1_variant(base=full), default, "arm edits on the tables vs the reference's compile")
    for kw in (dict(), dict(disable_back_joint=True), dict(disable_arms=False), dict(disable_arms=False, disable_back_joint=True),
               dict(hold_weight=True, weight_mass=5.0)):
        _assert_same_model(mjcf.unitree_h1_variant(**kw), mjcf.compile_unitree_h1(xml, **kw), kw)
    for name, m in (("h1_noback", mjcf.unitree_h1_variant(disable_back_joint=True)),
                    ("h1_carry", mjcf.unitree_h1_variant(hold_weight=True, weight_mass=5.0))):
        out = K.forward(m, g[name + "_qpos"], g[name + "_qvel"])
        assert list(g[name + "_body_names"][1:]) == list(m.body_names[1:])
        assert_close(m.body_mass, g[name + "_body_mass"], "masses", rtol=1e-12, atol=1e-12)
        for k in ("xpos", "site_xpos", "subtree_com"):
            assert_close(out[k], g[f"{name}_{k}"], f"{name} {k}", rtol=1e-12, atol=1e-12)
        assert_close(out["cvel"], g[name + "_cvel"], f"{name} cvel", rtol=1e-8, atol=5e-9)
    carry = mjcf.unitree_h1_variant(hold_weight=True, weight_mass=1.0)
    assert carry.body_names[-1] == "weight" and carry.body_mass[-1] == 2.0 and carry.nq == 17
    # arms are NOT re-oriented when a weight is held (UnitreeH1.py:84-85)
    assert_close(carry.body_quat[carry.body_id("left_shoulder_pitch_link")],
                 mjcf.load_builtin("unitree_h1_arms").body_quat[carry.body_id("left_shoulder_pitch_link")], "arm quat", 0, 0)
    with pytest.raises(AssertionError, match="disable the arms"):
        mjcf.unitree_h1_variant(disable_arms=False, hold_weight=True, weight_mass=1.0)


def test_host_philox_matches_the_contract():
    from olympics_mujoco_b200.utils import philox as HP
    from oracle import philox as OP
    for seed, env, cnt, stream in ((0, 0, 0, 0), (1234, 77, 3, 32), (2 ** 40 + 5, 4095, 9, 16)):
        want = [int(x) for x in OP.draw(seed, np.uint32(env), np.uint32(cnt), stream)]
        assert list(HP.philox4x32_10((env, cnt, stream, 0), (seed & 0xFFFFFFFF, seed >> 32))) == want
        assert HP.philox_randint(seed, env, cnt, stream, 4) == int(OP.to_int(np.uint32(want[0]), 4))


def test_bench_helpers_without_a_gpu():
    """bench.py's clock sampler degrades to "no samples" when neither NVML nor nvidia-smi answers (this container), and
    compact() keeps the few numbers of a side measurement, including how its device time was taken."""
    import time
    import bench
    s = bench.ClockSampler(0)
    s.start()
    time.sleep(0.25)
    c = s.stop()
    assert set(c) == {"sm_mhz", "sm_max_mhz", "reasons", "samples"} and c["reasons"] == [] or c["samples"] > 0
    d = bench.compact({"value": 2.0, "ms_per_step": 0.1234567, "timing": "CUDA-graph replay of the same launches",
                       "roofline": {"frac": 0.70123, "bound": "hbm", "peak": 6454.6}, "noise": [1, 2, 3]})
    assert d == {"value": 2.0, "ms_per_step": 0.12346, "timing": "graph", "frac": 0.7012, "bound": "hbm", "peak": 6454.6}
    assert bench.compact([{"value": 1.0, "timing": "eager launches"}]) == [{"value": 1.0, "timing": "eager"}]
    assert bench.compact({"error": "x"}) == {"error": "x"}


def test_bench_dump_outputs_writes_a_fixed_sample_within_64_mb(tmp_path):
    """bench.py --dump-outputs: every returned buffer restricted to the same seeded envs and steps, float32 kept, integer
    and flag buffers as float64, the moment sums whole; the written files stay below 64 MB at the bench's buffer shapes
    for any horizon (envs are sampled first, steps too once one env's horizon alone is over the budget)."""
    import torch
    import bench
    from olympics_mujoco_b200 import mjcf
    m = mjcf.load_builtin("unitree_h1")
    widths = dict(xpos=m.nbody * 3, xquat=m.nbody * 4, site_xpos=m.nsite * 3, cvel=m.nbody * 6, obs=32)   # make_rollout_buffers

    def buffers(T, n, seed):
        g = torch.Generator().manual_seed(seed)
        big = lambda *s: torch.randn((1,) + s[1:], generator=g).expand(*s)        # full bench shapes, one step of memory
        out = {k: big(T, c, n) for k, c in widths.items()}
        out.update(reward=big(T, n), fallen=torch.randint(0, 2, (1, n), dtype=torch.uint8, generator=g).expand(T, n),
                   traj_no_t=torch.randint(0, 4, (1, n), dtype=torch.int32, generator=g).expand(T, n),
                   step_no_t=torch.arange(T, dtype=torch.int32)[:, None].expand(T, n))
        return out, big(T, n), big(T, n), torch.randn(68, dtype=torch.float64, generator=g)

    for T, n, budget in ((500, 4096, bench.DUMP_BYTES), (1000, 4096, bench.DUMP_BYTES), (200, 50, 100_000)):
        out, vt, adv, mom = buffers(T, n, T)
        for d in ("a", "b"):
            bench.write_dump(tmp_path / f"{T}{d}", bench.dump_sample(out, vt, adv, mom, budget=budget))
        files = sorted((tmp_path / f"{T}a").glob("*.npy"))
        assert sum(p.stat().st_size for p in files) <= budget + 256 * len(files) < 64e6
        got = {p.stem: np.load(p) for p in files}
        assert set(got) == {*out, "v_target", "adv", "adv_moments", "obs_moments", "env_index", "step_index"}
        envs, steps = got["env_index"].astype(np.int64), got["step_index"].astype(np.int64)
        assert len(set(envs)) == len(envs) and envs.max() < n and len(set(steps)) == len(steps) and steps.max() < T
        assert (len(steps) == T) == (budget > 10 ** 6), "steps are sampled only when one env's horizon is over the budget"
        for k, v in (*out.items(), ("v_target", vt), ("adv", adv)):
            assert got[k].dtype == (np.float32 if v.dtype == torch.float32 else np.float64), k
            assert np.array_equal(got[k], v.numpy()[steps][..., envs]), k
        assert np.array_equal(got["adv_moments"], mom[:3].numpy()) and np.array_equal(got["obs_moments"], mom[3:].numpy())
        for p in files:
            assert p.read_bytes() == (tmp_path / f"{T}b" / p.name).read_bytes(), p.name
