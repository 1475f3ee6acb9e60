"""CPU: the kinematics oracle (oracle/kinematics.py, a restatement of MuJoCo's recursions) against an INDEPENDENT second
checker (tools/fk_independent.py: its own MJCF reader, 4x4 homogeneous transforms, velocities by numerical differentiation
of q(t) = q (+) t qdot, then transported to subtree_com[root]) -- fixture tests/golden/fk_independent_ref.npz -- plus the
analytic known answers SURVEY.md 8(c) lists.  MuJoCo itself (mujoco==2.3.6) cannot be installed here; two restatements
that share no helper and derive velocities by different means are what pins A1 / A2 in its place."""
import importlib.util
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, assert_close
from oracle import kinematics as K

VARIANTS = {"h1": "unitree_h1", "h1_arms": "unitree_h1_arms", "a3": "stick_figure_a3"}


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLDEN / "fk_independent_ref.npz")


def _model(name):
    from olympics_mujoco_b200 import mjcf
    return mjcf.load_builtin(VARIANTS[name])


def _same_rotation(q_oracle, q_ref):
    s = np.sign(np.sum(q_oracle * q_ref, axis=-1, keepdims=True))     # q and -q are the same rotation
    return q_ref * np.where(s == 0, 1.0, s)


@pytest.mark.parametrize("name", list(VARIANTS))
def test_oracle_matches_independent_checker(gold, name):
    m = _model(name)
    q, v = gold[name + "_qpos"], gold[name + "_qvel"]
    assert list(gold[name + "_body_names"][1:]) == list(m.body_names[1:])
    assert_close(m.body_mass, gold[name + "_body_mass"], "body masses (A3: derived from the geoms)", rtol=1e-12, atol=1e-12)
    out = K.forward(m, q, v)
    for k in ("xpos", "xipos", "site_xpos", "subtree_com"):
        assert_close(out[k], gold[f"{name}_{k}"], k, rtol=1e-12, atol=1e-12)
    assert_close(out["xmat"], gold[name + "_xmat"], "xmat", rtol=1e-12, atol=1e-12)
    assert_close(out["site_xmat"], gold[name + "_site_xmat"], "site_xmat", rtol=1e-12, atol=1e-12)
    assert_close(out["xquat"], _same_rotation(out["xquat"], gold[name + "_xquat"]), "xquat", rtol=1e-12, atol=1e-12)
    # numerical differentiation (h = 1e-6, float64): 1e-9 of agreement on velocities of a few m/s
    assert_close(out["cvel"], gold[name + "_cvel"], "cvel = [omega; v at subtree_com[root]]", rtol=1e-8, atol=5e-9)


def test_object_velocity_matches_numerical_origin_velocity(gold):
    """A2: mj_objectVelocity(mjOBJ_XBODY, flg_local=0) of the two feet, reordered [lin, ang]
    (mujoco_robot_interface.py:299-327), against the numerically differentiated velocity of the body-frame origin."""
    m = _model("a3")
    out = K.forward(m, gold["a3_qpos"], gold["a3_qvel"])
    for col, body in enumerate(("left_foot", "right_foot")):
        res = K.mj_objectVelocity_xbody(m, out["xpos"], out["subtree_com"], out["cvel"], m.body_id(body))   # [ang, lin]
        assert_close(np.concatenate([res[:, 3:], res[:, :3]], axis=1), gold["a3_foot_objvel"][:, col], body, rtol=1e-8, atol=5e-9)


def test_analytic_known_answers_h1(gold):
    """SURVEY 8(c): at the zero pose xpos is the sum of the body offsets down the chain."""
    m = _model("h1")
    assert not gold["h1_qpos"][0].any()
    for src in (gold["h1_xpos"][0], K.forward(m, gold["h1_qpos"][:1], gold["h1_qvel"][:1])["xpos"][0]):
        assert_close(src[m.body_id("left_ankle_link")], [0.039468, 0.0875 + 0.11536, 1.045 - 0.1742 - 0.4 - 0.4],
                     "left_ankle_link at the zero pose", rtol=1e-12, atol=1e-12)
        assert_close(src[m.body_id("right_ankle_link")], [0.039468, -0.0875 - 0.11536, 1.045 - 0.1742 - 0.4 - 0.4],
                     "right_ankle_link at the zero pose", rtol=1e-12, atol=1e-12)
    assert abs(gold["h1_body_mass"].sum() - 51.437) < 1e-9 and abs(gold["a3_body_mass"].sum() - 40.8214) < 1e-4


@pytest.mark.parametrize("side,sign", [("right", -1.0), ("left", 1.0)])
def test_analytic_known_answers_a3_off_centre_joints(side, sign):
    """a3.xml:67,71,72 (right) and :86,90,91 (left): the knee hinges about a point 0.02 above the shin origin, the ankle
    joints about points 0.04 and 0.08 above the foot origin.  A single-joint rotation by theta turns the child body about
    the ANCHOR (body origin + pos), which stays where it was: closed-form positions."""
    m = _model("a3")
    zero = m.qpos0.copy()[None]
    base = K.forward(m, zero, np.zeros((1, m.nv)))
    shin, foot = m.body_id(f"{side}_shin"), m.body_id(f"{side}_foot")
    hip_y = 1.5 - 0.26 - 0.165 - 0.1                                  # torso z + lower_waist + pelvis + thigh offsets
    assert_close(base["xpos"][0, shin], [-0.01, sign * 0.1, hip_y - 0.4], "shin origin at the zero pose", rtol=1e-12, atol=1e-12)
    assert_close(base["xpos"][0, foot], [-0.01, sign * 0.1, hip_y - 0.8], "foot origin at the zero pose", rtol=1e-12, atol=1e-12)
    th = 0.7

    def posed(joint):
        q = zero.copy()
        q[0, m.jnt_qposadr[m.joint_id(joint)]] = th
        return K.forward(m, q, np.zeros((1, m.nv)))["xpos"][0]

    c, s = np.cos(th), np.sin(th)
    # knee: axis y through (0, 0, 0.02) of the shin frame; a point at offset d from the anchor moves to Ry(th) d
    p = posed(f"{side}_knee")
    anchor = base["xpos"][0, shin] + [0, 0, 0.02]
    for body, d in ((shin, np.array([0, 0, -0.02])), (foot, np.array([0, 0, -0.42]))):
        assert_close(p[body], anchor + [c * d[0] + s * d[2], d[1], -s * d[0] + c * d[2]], f"knee rotation, body {body}", rtol=1e-12, atol=1e-12)
    # ankle_x: axis x through (0, 0, 0.04) of the foot frame: Rx(th) d = (dx, c dy - s dz, s dy + c dz)
    p = posed(f"{side}_ankle_x")
    d = np.array([0, 0, -0.04])
    assert_close(p[foot], base["xpos"][0, foot] + [0, 0, 0.04] + [d[0], c * d[1] - s * d[2], s * d[1] + c * d[2]], "ankle_x", rtol=1e-12, atol=1e-12)
    assert_close(p[shin], base["xpos"][0, shin], "ankle_x leaves the shin alone", rtol=0, atol=1e-15)
    # ankle_y: axis y through (0, 0, 0.08)
    p = posed(f"{side}_ankle_y")
    d = np.array([0, 0, -0.08])
    assert_close(p[foot], base["xpos"][0, foot] + [0, 0, 0.08] + [c * d[0] + s * d[2], d[1], -s * d[0] + c * d[2]], "ankle_y", rtol=1e-12, atol=1e-12)
    # the force site rides on the foot: (0.03, 0, -0.03) in the foot frame
    site = m.site_id("rf_force" if side == "right" else "lf_force")
    assert_close(base["site_xpos"][0, site], base["xpos"][0, foot] + [0.03, 0, -0.03], "force site", rtol=1e-12, atol=1e-12)


def test_independent_checker_shares_no_code_with_the_oracle():
    """The checker that wrote the fixture (tools/fk_independent.py) imports nothing from the oracle or the package."""
    spec = importlib.util.spec_from_file_location("fk_independent", ROOT / "tools" / "fk_independent.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    assert "oracle" not in mod.__dict__ and not any(k.startswith("oracle") for k in vars(mod))     # shares nothing
    src = (ROOT / "tools" / "fk_independent.py").read_text()
    assert "import oracle" not in src and "from oracle" not in src and "olympics_mujoco_b200" not in src.split('"""', 2)[2]
