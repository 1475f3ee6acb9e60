"""Model compiler back end: KinematicModel -> topology-specialised CUDA device function.

The B200 design point (DESIGN.md, "K1"): one THREAD per environment, structure-of-arrays HBM layout, and
the whole body tree unrolled into straight-line fp32 code with every model constant folded in -- zero
terms vanish, axis-aligned joints become 8-FMA quaternion products, fixed bodies inherit their parent's
spatial velocity for free.  This module emits that code from the same tables the oracle and the
table-driven kernel use; ``build.py`` runs it for the two in-scope robots before nvcc.

The emitted function restates MuJoCo's ``mj_kinematics`` + ``mj_comPos`` + ``mj_comVel``
(mujoco==2.3.6 ``engine_core_smooth.c``; reference call sites ``loco_env_base.py:410,525,1160``) with one
algebraic re-association: body spatial velocities are accumulated about the root body's origin P and
shifted to the subtree centre of mass at the end (``v_com = v_P + w x (com - P)``), so that kinematics
and velocities run in a single pass.
"""
from __future__ import annotations

import hashlib

import numpy as np

from .mjcf import JNT_BALL, JNT_FREE, JNT_HINGE, JNT_SLIDE


# Scalar type of the code being emitted: "float" (the kernels' arithmetic) or "double" (the exact slow path of the A3
# threshold decisions, generate_fk_pos(..., scalar="double")).  Constants are rounded to fp32 only in float mode.
_SCALAR = "float"


def _f(x):
    """Shortest literal that round-trips in the scalar type being emitted."""
    if _SCALAR == "double":
        return repr(float(x)) if float(x) != int(float(x)) or abs(float(x)) > 1e15 else f"{float(x):.1f}"
    v = np.float32(x)
    if v == 0:
        return "0.0f"
    return np.format_float_scientific(v, unique=True, trim="0") + "f"


def _num(c):
    return float(c) if _SCALAR == "double" else np.float32(c)


class E:
    """A scalar that is either a compile-time constant or a named C variable."""
    __slots__ = ("c", "n")

    def __init__(self, c=None, n=None):
        self.c = None if c is None else (float(c) if _SCALAR == "double" else float(np.float32(c)))
        self.n = n

    @property
    def is_const(self):
        return self.n is None

    def __str__(self):
        return _f(self.c) if self.is_const else self.n


ZERO, ONE = E(0.0), E(1.0)


class Gen:
    def __init__(self):
        self.lines = []
        self.k = 0

    def emit(self, s):
        self.lines.append("  " + s)

    def tmp(self, expr):
        self.k += 1
        name = f"t{self.k}"
        self.emit(f"{_SCALAR} {name} = {expr};")
        return E(n=name)

    # ---- scalar algebra with folding
    def neg(self, a):
        if a.is_const:
            return E(-a.c)
        return self.tmp(f"-{a}")

    def mul(self, a, b):
        if a.is_const and b.is_const:
            return E(_num(a.c) * _num(b.c))
        if a.is_const:
            a, b = b, a
        if b.is_const:
            if b.c == 0.0:
                return ZERO
            if b.c == 1.0:
                return a
            if b.c == -1.0:
                return self.neg(a)
        return self.tmp(f"{a} * {b}")

    def add(self, a, b):
        if a.is_const and b.is_const:
            return E(_num(a.c) + _num(b.c))
        if a.is_const and a.c == 0.0:
            return b
        if b.is_const and b.c == 0.0:
            return a
        return self.tmp(f"{a} + {b}")

    def sub(self, a, b):
        if a.is_const and b.is_const:
            return E(_num(a.c) - _num(b.c))
        if b.is_const and b.c == 0.0:
            return a
        if a.is_const and a.c == 0.0:
            return self.neg(b)
        if not a.is_const and not b.is_const and a.n == b.n:
            return ZERO
        return self.tmp(f"{a} - {b}")

    def fma(self, a, b, c):
        """a*b + c with folding; emitted as fmaf so the contraction does not depend on nvcc flags."""
        if (a.is_const and a.c == 0.0) or (b.is_const and b.c == 0.0):
            return c
        if a.is_const and b.is_const:
            return self.add(E(_num(a.c) * _num(b.c)), c)
        if c.is_const and c.c == 0.0:
            return self.mul(a, b)
        if a.is_const and a.c == 1.0:
            return self.add(b, c)
        if b.is_const and b.c == 1.0:
            return self.add(a, c)
        if a.is_const and a.c == -1.0:
            return self.sub(c, b)
        if b.is_const and b.c == -1.0:
            return self.sub(c, a)
        return self.tmp(f"{'fma' if _SCALAR == 'double' else 'fmaf'}({a}, {b}, {c})")

    def dot(self, a, b):
        acc = ZERO
        for x, y in zip(a, b):
            acc = self.fma(x, y, acc)
        return acc

    # ---- vectors / quaternions
    def vadd(self, a, b):
        return [self.add(x, y) for x, y in zip(a, b)]

    def vsub(self, a, b):
        return [self.sub(x, y) for x, y in zip(a, b)]

    def vscale(self, a, s):
        return [self.mul(x, s) for x in a]

    def vfma(self, a, s, c):
        return [self.fma(x, s, y) for x, y in zip(a, c)]

    def cross(self, a, b):
        return [self.sub(self.mul(a[1], b[2]), self.mul(a[2], b[1])),
                self.sub(self.mul(a[2], b[0]), self.mul(a[0], b[2])),
                self.sub(self.mul(a[0], b[1]), self.mul(a[1], b[0]))]

    def qmul(self, a, b):
        """mju_mulQuat."""
        w = self.sub(self.sub(self.sub(self.mul(a[0], b[0]), self.mul(a[1], b[1])), self.mul(a[2], b[2])),
                     self.mul(a[3], b[3]))
        x = self.sub(self.add(self.add(self.mul(a[0], b[1]), self.mul(a[1], b[0])), self.mul(a[2], b[3])),
                     self.mul(a[3], b[2]))
        y = self.add(self.add(self.sub(self.mul(a[0], b[2]), self.mul(a[1], b[3])), self.mul(a[2], b[0])),
                     self.mul(a[3], b[1]))
        z = self.add(self.sub(self.add(self.mul(a[0], b[3]), self.mul(a[1], b[2])), self.mul(a[2], b[1])),
                     self.mul(a[3], b[0]))
        return [w, x, y, z]

    def qrot(self, q, v):
        """mju_rotVecQuat: v + 2 u x (u x v + w v)."""
        if all(x.is_const and x.c == 0.0 for x in v):
            return [ZERO, ZERO, ZERO]
        if q[0].is_const and q[0].c == 1.0 and all(x.is_const and x.c == 0.0 for x in q[1:]):
            return list(v)
        u = q[1:]
        t = self.vadd(self.vscale(v, q[0]), self.cross(u, v))
        c = self.cross(u, t)
        return [self.fma(E(2.0), c[i], v[i]) for i in range(3)]

    def qnormalize(self, q):
        if all(x.is_const for x in q):
            a = np.array([x.c for x in q], dtype=np.float64)
            a = a / np.linalg.norm(a)
            return [E(x) for x in a]
        n2 = self.dot(q, q)
        inv = self.tmp(f"1.0 / sqrt({n2})" if _SCALAR == "double" else f"rsqrtf({n2})")
        return [self.mul(x, inv) for x in q]

    def quat2mat(self, q):
        """mju_quat2Mat, row-major 9."""
        w, x, y, z = q
        ww, xx, yy, zz = self.mul(w, w), self.mul(x, x), self.mul(y, y), self.mul(z, z)
        xy, xz, yz = self.mul(x, y), self.mul(x, z), self.mul(y, z)
        wx, wy, wz = self.mul(w, x), self.mul(w, y), self.mul(w, z)
        two = E(2.0)
        return [self.sub(self.sub(self.add(ww, xx), yy), zz), self.mul(two, self.sub(xy, wz)), self.mul(two, self.add(xz, wy)),
                self.mul(two, self.add(xy, wz)), self.sub(self.add(self.sub(ww, xx), yy), zz), self.mul(two, self.sub(yz, wx)),
                self.mul(two, self.sub(xz, wy)), self.mul(two, self.add(yz, wx)), self.add(self.sub(self.sub(ww, xx), yy), zz)]


def model_fingerprint(model):
    """Hash of the float32 tables the generated code bakes in (checked again by om_model_create)."""
    h = hashlib.sha256()
    for a in (model.body_parentid, model.body_jntadr, model.body_jntnum, model.jnt_type, model.jnt_qposadr,
              model.jnt_dofadr, model.site_bodyid):
        h.update(np.asarray(a, np.int32).tobytes())
    for a in (model.body_pos, model.body_quat, model.body_ipos, model.body_mass, model.jnt_axis, model.jnt_pos,
              model.qpos0, model.site_pos, model.site_quat):
        h.update(np.asarray(a, np.float32).tobytes())
    return h.hexdigest()[:16]


def split_parts(model, nparts):
    """Partition the bodies of a single-tree model into ``nparts`` groups of whole subtrees hanging off the tree root
    (UnitreeH1: right leg / left leg / torso with the arms), balanced by a rough cost (hinges weigh 3, fixed bodies
    1); the root body and the world go to the lightest group.  -> list of body-id sets."""
    nb = model.nbody
    root = 1
    kids = [i for i in range(2, nb) if int(model.body_parentid[i]) == root]
    sub = {k: [k] for k in kids}
    for i in range(2, nb):
        j = i
        while int(model.body_parentid[j]) != root:
            j = int(model.body_parentid[j])
            if j == 0:
                raise ValueError("split_parts needs a single tree hanging off body 1")
        if j != i:
            sub[j].append(i)
    cost = {k: sum(1 + 3 * int(model.body_jntnum[b]) for b in v) for k, v in sub.items()}
    parts = [set() for _ in range(nparts)]
    load = [0] * nparts
    for k in sorted(kids, key=lambda k: -cost[k]):
        p = load.index(min(load))
        parts[p].update(sub[k])
        load[p] += cost[k]
    parts[load.index(min(load))].update({0, root})
    return parts


def generate_fk(model, fn_name, part=None, env_mass_body=None):
    """Return CUDA source text of ``template<class Sink> __device__ void <fn_name>(q, qd, S)``.

    With ``part=(own_bodies, Exchange)`` the function evaluates only the bodies in ``own_bodies`` and their ancestors,
    emits sink calls for ``own_bodies`` alone, and obtains the tree's centre of mass from a second template argument:
    ``X.com_exchange(sx, sy, sz, 1/M, cx, cy, cz)`` receives this part's sum of m * xipos and returns the normalised total
    (the caller combines the parts -- through shared memory in h1_step_split_kernel).

    With ``env_mass_body=b`` the mass of body ``b`` is a runtime argument, ``<fn_name>(q, qd, S, env_mass)``: its
    m * xipos term and ``1 / (M0 + env_mass)`` of its tree are emitted instead of folded (M0 = the tree's other bodies).
    The carried weight of UnitreeH1 is such a body: one function serves every mass.

    Sink interface (all indices are literals so unused outputs are dead-code eliminated):
      S.xpos(b,x,y,z)  S.xquat(b,w,x,y,z)  S.site_xpos(s,x,y,z)  S.site_xmat(s,m0..m8)
      S.cvel(b,wx,wy,wz,vx,vy,vz)  S.com(x,y,z)
      S.vel_p(b,wx,wy,wz,vx,vy,vz)   [w; v of the body-fixed point at xpos[rootid]]
    """
    if env_mass_body is not None and (part is not None or not 0 < env_mass_body < model.nbody):
        raise ValueError("env_mass_body names one body of a whole-model FK")
    g = Gen()
    nb = model.nbody
    own = set(range(nb)) if part is None else set(part)
    needed = set(own)
    for b in list(own):
        while b != 0:
            b = int(model.body_parentid[b])
            needed.add(b)
    c3 = lambda v: [E(x) for x in v]
    pos = {0: [ZERO, ZERO, ZERO]}
    quat = {0: [ONE, ZERO, ZERO, ZERO]}
    wvel = {0: [ZERO, ZERO, ZERO]}         # angular velocity of body
    lvel = {0: [ZERO, ZERO, ZERO]}         # linear velocity of the body-fixed point at P (tree root origin)
    P = {}                                 # root body id -> reference point
    com_acc = {}                           # root body id -> sum m*xipos
    com_mass = {}

    def q_in(k):
        return E(n=f"q[{k}]")

    def qd_in(k):
        return E(n=f"qd[{k}]")

    if 0 in own:
        g.emit("S.xpos(0, 0.0f, 0.0f, 0.0f);")
        g.emit("S.xquat(0, 1.0f, 0.0f, 0.0f, 0.0f);")
        g.emit("S.cvel(0, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f);")
    for i in range(1, nb):
        if i not in needed:
            continue
        g.emit(f"// ---- body {i}: {model.body_names[i]}")
        pid = int(model.body_parentid[i])
        rid = int(model.body_rootid[i])
        jadr, jnum = int(model.body_jntadr[i]), int(model.body_jntnum[i])
        w_i, v_i = list(wvel[pid]), list(lvel[pid])
        if jnum == 1 and model.jnt_type[jadr] == JNT_FREE:
            qa, da = int(model.jnt_qposadr[jadr]), int(model.jnt_dofadr[jadr])
            p = [q_in(qa + k) for k in range(3)]
            qt = g.qnormalize([q_in(qa + 3 + k) for k in range(4)])
            if rid == i:
                P[rid] = p
            # dofs 0-2: world-axis translation; dofs 3-5: rotation about the body axes through xpos
            v_i = [g.add(v_i[k], qd_in(da + k)) for k in range(3)]
            arm = g.vsub(P[rid], p)                       # (P - anchor), zero when this body is the root
            for k in range(3):
                ek = [ONE if m == k else ZERO for m in range(3)]
                axis = g.qrot(qt, ek)                     # column k of xmat
                w_i = g.vfma(axis, qd_in(da + 3 + k), w_i)
                v_i = g.vfma(g.cross(axis, arm), qd_in(da + 3 + k), v_i)
        else:
            p = g.vadd(pos[pid], g.qrot(quat[pid], c3(model.body_pos[i])))
            bq = model.body_quat[i]
            qt = quat[pid] if (abs(bq[0] - 1.0) < 1e-15 and np.all(np.abs(bq[1:]) < 1e-15)) else g.qmul(quat[pid], c3(bq))
            joints = []
            for j in range(jadr, jadr + jnum):
                jt = int(model.jnt_type[j])
                qa, da = int(model.jnt_qposadr[j]), int(model.jnt_dofadr[j])
                axis_w = g.qrot(qt, c3(model.jnt_axis[j]))
                anchor = g.vadd(g.qrot(qt, c3(model.jnt_pos[j])), p)
                joints.append((jt, da, axis_w, anchor))
                dq = g.sub(q_in(qa), E(model.qpos0[qa]))
                if jt == JNT_SLIDE:
                    p = g.vfma(axis_w, dq, p)
                elif jt == JNT_HINGE:
                    g.emit(f"float s{j}, c{j}; om::om_sincos(0.5f * ({dq}), &s{j}, &c{j});")
                    sj, cj = E(n=f"s{j}"), E(n=f"c{j}")
                    qloc = [cj] + [g.mul(E(a), sj) for a in model.jnt_axis[j]]
                    qt = g.qmul(qt, qloc)
                    jp = c3(model.jnt_pos[j])
                    if any(x.c != 0.0 for x in jp):
                        p = g.vsub(anchor, g.qrot(qt, jp))
                else:
                    raise NotImplementedError("ball joints are served by the table-driven kernel only")
            if rid == i:
                P[rid] = p
            for jt, da, axis_w, anchor in joints:
                if jt == JNT_SLIDE:
                    v_i = g.vfma(axis_w, qd_in(da), v_i)
                else:
                    w_i = g.vfma(axis_w, qd_in(da), w_i)
                    v_i = g.vfma(g.cross(axis_w, g.vsub(P[rid], anchor)), qd_in(da), v_i)
            qt = g.qnormalize(qt)
        pos[i], quat[i], wvel[i], lvel[i] = p, qt, w_i, v_i
        if i not in own:
            continue
        g.emit(f"S.xpos({i}, {p[0]}, {p[1]}, {p[2]});")
        g.emit(f"S.xquat({i}, {qt[0]}, {qt[1]}, {qt[2]}, {qt[3]});")
        # spatial velocity about the tree root's origin P (before the shift to the subtree COM): lets a
        # consumer that only needs point velocities (mj_objectVelocity) skip the COM pass entirely
        g.emit(f"S.vel_p({i}, {w_i[0]}, {w_i[1]}, {w_i[2]}, {v_i[0]}, {v_i[1]}, {v_i[2]});")
        m = float(model.body_mass[i])
        if i == env_mass_body:
            xi = g.vadd(p, g.qrot(qt, c3(model.body_ipos[i])))
            acc = com_acc.get(rid, [ZERO, ZERO, ZERO])
            com_acc[rid] = g.vfma(xi, E(n="env_mass"), acc)
            com_mass.setdefault(rid, 0.0)
        elif m > 0:
            xi = g.vadd(p, g.qrot(qt, c3(model.body_ipos[i])))
            acc = com_acc.get(rid, [ZERO, ZERO, ZERO])
            com_acc[rid] = g.vfma(xi, E(m), acc)
            com_mass[rid] = com_mass.get(rid, 0.0) + m
        for s in range(model.nsite):
            if int(model.site_bodyid[s]) != i:
                continue
            sp = g.vadd(p, g.qrot(qt, c3(model.site_pos[s])))
            g.emit(f"S.site_xpos({s}, {sp[0]}, {sp[1]}, {sp[2]});")
            sq = model.site_quat[s]
            sqt = qt if (abs(sq[0] - 1.0) < 1e-15 and np.all(np.abs(sq[1:]) < 1e-15)) else g.qmul(qt, c3(sq))
            g.emit(f"if (S.want_site_xmat) {{")
            mat = g.quat2mat(sqt)
            g.emit(f"S.site_xmat({s}, " + ", ".join(str(x) for x in mat) + "); }")

    g.emit("// ---- subtree centre of mass of each kinematic tree, then shift velocities to it")
    dvec = {}
    if part is not None:
        if set(P) != {1}:
            raise ValueError("a split FK needs a single kinematic tree rooted at body 1")
        com_total_mass = float(sum(float(model.body_mass[b]) for b in range(1, nb) if int(model.body_rootid[b]) == 1))
        acc = com_acc.get(1, [ZERO, ZERO, ZERO])
        g.emit("float com_x, com_y, com_z;")
        g.emit(f"X.com_exchange({acc[0]}, {acc[1]}, {acc[2]}, {_f(1.0 / com_total_mass)}, com_x, com_y, com_z);")
        com = [E(n="com_x"), E(n="com_y"), E(n="com_z")]
        if 1 in own:
            g.emit("S.com(com_x, com_y, com_z);")
        dvec[1] = g.vsub(com, P[1])
    else:
        env_root = None if env_mass_body is None else int(model.body_rootid[env_mass_body])
        for rid, acc in com_acc.items():
            if rid == env_root:
                inv = g.tmp(f"1.0f / ({_f(com_mass[rid])} + env_mass)")
                com = g.vscale(acc, inv)
            else:
                com = g.vscale(acc, E(1.0 / com_mass[rid]))
            if rid == 1:
                g.emit(f"S.com({com[0]}, {com[1]}, {com[2]});")
            dvec[rid] = g.vsub(com, P[rid])
    # bodies without joints share their parent's cvel: emit each distinct value once
    for i in range(1, nb):
        if i not in own:
            continue
        rid = int(model.body_rootid[i])
        lin = g.vadd(lvel[i], g.cross(wvel[i], dvec[rid])) if rid in dvec else lvel[i]
        w = wvel[i]
        g.emit(f"S.cvel({i}, {w[0]}, {w[1]}, {w[2]}, {lin[0]}, {lin[1]}, {lin[2]});")

    # the site_xmat block opened a scope in which temporaries were declared const; those are only used inside
    body = "\n".join(g.lines)
    head = (f"// GENERATED by olympics_mujoco_b200/codegen.py from model '{model.name}' "
            f"(fingerprint {model_fingerprint(model)}) -- do not edit.\n"
            f"// nbody={model.nbody} njnt={model.njnt} nq={model.nq} nv={model.nv} nsite={model.nsite}\n"
            + (f"// part: bodies {sorted(own)}\n" if part is not None else "") +
            (f"// runtime mass: body {env_mass_body} ({model.body_names[env_mass_body]})\n"
             if env_mass_body is not None else "") +
            (f"template <class Sink, class Exchange>\n" if part is not None else f"template <class Sink>\n") +
            f"OM_HD void {fn_name}(const float (&q)[{model.nq}], const float (&qd)[{model.nv}], Sink& S"
            + (", Exchange& X" if part is not None else "") + (", float env_mass" if env_mass_body is not None else "")
            + ") {\n")
    return head + body + "\n}\n"


def generate_fk_pos(model, fn_name, scalar="float"):
    global _SCALAR, ZERO, ONE
    prev = _SCALAR
    _SCALAR = scalar
    try:
        return _generate_fk_pos(model, fn_name)
    finally:
        _SCALAR = prev


def _generate_fk_pos(model, fn_name):
    """Position/velocity-only variant for consumers that never read body orientations (the A3 walking task reads
    xpos / site_xpos / point velocities and the root quaternion, which is qpos itself): the chain is carried as
    ROTATION MATRICES, so an axis-aligned hinge costs 12 multiply-adds (two columns rotate) instead of a quaternion
    product, a renormalisation and three quaternion-vector rotations, and a world joint axis is a column of the
    parent's matrix.  Same quantities as ``generate_fk`` to fp32 round-off (checked against the float64 oracle by
    tests/test_host.py).  Sink calls: S.xpos, S.site_xpos, S.vel_p for every body; S.xquat for free-joint bodies only.
    """
    g = Gen()
    nb = model.nbody
    c3 = lambda v: [E(x) for x in v]
    I3 = [ONE, ZERO, ZERO, ZERO, ONE, ZERO, ZERO, ZERO, ONE]
    pos = {0: [ZERO, ZERO, ZERO]}
    rot = {0: list(I3)}
    wvel = {0: [ZERO, ZERO, ZERO]}
    lvel = {0: [ZERO, ZERO, ZERO]}
    P = {}

    def mv(R, v):
        return [g.dot(R[3 * r:3 * r + 3], v) for r in range(3)]

    def mm(A, B):
        return [g.dot(A[3 * r:3 * r + 3], [B[c], B[3 + c], B[6 + c]]) for r in range(3) for c in range(3)]

    def const_mat(q):
        w, x, y, z = [float(v) for v in np.asarray(q, np.float64) / np.linalg.norm(q)]
        return [E(v) for v in (1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y),
                               2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x),
                               2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y))]

    def is_identity_quat(q):
        return abs(q[0] - 1.0) < 1e-15 and np.all(np.abs(q[1:]) < 1e-15)

    q_in = lambda k: E(n=f"q[{k}]")
    qd_in = lambda k: E(n=f"qd[{k}]")
    g.emit(f"S.xpos(0, {_f(0.0)}, {_f(0.0)}, {_f(0.0)});")
    for i in range(1, nb):
        g.emit(f"// ---- body {i}: {model.body_names[i]}")
        pid = int(model.body_parentid[i])
        rid = int(model.body_rootid[i])
        jadr, jnum = int(model.body_jntadr[i]), int(model.body_jntnum[i])
        w_i, v_i = list(wvel[pid]), list(lvel[pid])
        if jnum == 1 and model.jnt_type[jadr] == JNT_FREE:
            qa, da = int(model.jnt_qposadr[jadr]), int(model.jnt_dofadr[jadr])
            p = [q_in(qa + k) for k in range(3)]
            qt = g.qnormalize([q_in(qa + 3 + k) for k in range(4)])
            g.emit(f"S.xquat({i}, {qt[0]}, {qt[1]}, {qt[2]}, {qt[3]});")
            w, x, y, z = qt
            two = E(2.0)
            xx, yy, zz = g.mul(x, x), g.mul(y, y), g.mul(z, z)
            xy, xz, yz, wx, wy, wz = g.mul(x, y), g.mul(x, z), g.mul(y, z), g.mul(w, x), g.mul(w, y), g.mul(w, z)
            one_m2 = lambda a, b: g.fma(E(-2.0), g.add(a, b), ONE)
            R = [one_m2(yy, zz), g.mul(two, g.sub(xy, wz)), g.mul(two, g.add(xz, wy)),
                 g.mul(two, g.add(xy, wz)), one_m2(xx, zz), g.mul(two, g.sub(yz, wx)),
                 g.mul(two, g.sub(xz, wy)), g.mul(two, g.add(yz, wx)), one_m2(xx, yy)]
            if rid == i:
                P[rid] = p
            v_i = [g.add(v_i[k], qd_in(da + k)) for k in range(3)]
            arm = g.vsub(P[rid], p)
            for k in range(3):
                axis = [R[k], R[3 + k], R[6 + k]]
                w_i = g.vfma(axis, qd_in(da + 3 + k), w_i)
                v_i = g.vfma(g.cross(axis, arm), qd_in(da + 3 + k), v_i)
        else:
            p = g.vadd(pos[pid], mv(rot[pid], c3(model.body_pos[i])))
            bq = model.body_quat[i]
            R = rot[pid] if is_identity_quat(bq) else mm(rot[pid], const_mat(bq))
            joints = []
            for j in range(jadr, jadr + jnum):
                jt = int(model.jnt_type[j])
                qa, da = int(model.jnt_qposadr[j]), int(model.jnt_dofadr[j])
                ax = np.asarray(model.jnt_axis[j], np.float64)
                axis_w = mv(R, c3(ax))
                anchor = g.vadd(mv(R, c3(model.jnt_pos[j])), p)
                joints.append((jt, da, axis_w, anchor))
                dq = g.sub(q_in(qa), E(model.qpos0[qa]))
                if jt == JNT_SLIDE:
                    p = g.vfma(axis_w, dq, p)
                elif jt == JNT_HINGE:
                    if _SCALAR == "double":
                        g.emit(f"double s{j}, c{j}; sincos({dq}, &s{j}, &c{j});")
                    else:
                        g.emit(f"float s{j}, c{j}; om::om_sincos_hinge({dq}, &s{j}, &c{j});")
                    sj, cj = E(n=f"s{j}"), E(n=f"c{j}")
                    # Rodrigues: c I + (1 - c) a a^T + s [a]x, constants folded (axis-aligned: four live entries)
                    omc = None
                    K = [[0.0, -ax[2], ax[1]], [ax[2], 0.0, -ax[0]], [-ax[1], ax[0], 0.0]]
                    rodr = []
                    for r in range(3):
                        for c in range(3):
                            aa = float(_num(ax[r] * ax[c]))
                            if abs(aa - (1.0 if r == c else 0.0)) < 1e-7 and abs(K[r][c]) < 1e-7 and r == c:
                                rodr.append(ONE)               # diagonal entry on the axis itself
                                continue
                            e = g.mul(E(1.0 if r == c else 0.0), cj)
                            if abs(aa) > 1e-7 and not (r == c and abs(aa - 1.0) < 1e-7):
                                if omc is None:
                                    omc = g.sub(ONE, cj)
                                e = g.fma(E(aa), omc, e)
                            e = g.fma(E(K[r][c]), sj, e)
                            rodr.append(e)
                    R = mm(R, rodr)
                    jp = c3(model.jnt_pos[j])
                    if any(x.c != 0.0 for x in jp):
                        p = g.vsub(anchor, mv(R, jp))
                else:
                    raise NotImplementedError("ball joints are served by the table-driven kernel only")
            if rid == i:
                P[rid] = p
            for jt, da, axis_w, anchor in joints:
                if jt == JNT_SLIDE:
                    v_i = g.vfma(axis_w, qd_in(da), v_i)
                else:
                    w_i = g.vfma(axis_w, qd_in(da), w_i)
                    v_i = g.vfma(g.cross(axis_w, g.vsub(P[rid], anchor)), qd_in(da), v_i)
        pos[i], rot[i], wvel[i], lvel[i] = p, R, w_i, v_i
        g.emit(f"S.xpos({i}, {p[0]}, {p[1]}, {p[2]});")
        g.emit(f"S.vel_p({i}, {w_i[0]}, {w_i[1]}, {w_i[2]}, {v_i[0]}, {v_i[1]}, {v_i[2]});")
        for s in range(model.nsite):
            if int(model.site_bodyid[s]) != i:
                continue
            sp = g.vadd(p, mv(R, c3(model.site_pos[s])))
            g.emit(f"S.site_xpos({s}, {sp[0]}, {sp[1]}, {sp[2]});")
    body = "\n".join(g.lines)
    head = (f"// GENERATED by olympics_mujoco_b200/codegen.py (generate_fk_pos) from model '{model.name}' "
            f"(fingerprint {model_fingerprint(model)}) -- do not edit.\n"
            f"template <class Sink>\nOM_HD void {fn_name}(const {_SCALAR} (&q)[{model.nq}], "
            f"const {_SCALAR} (&qd)[{model.nv}], Sink& S) {{\n")
    return head + body + "\n}\n"


def generate_tables(model, prefix):
    """Host-side constant tables used by om_model_create to verify that a model handed over the C ABI is
    the one the specialised kernel was generated from."""
    def arr(name, a, ctype, fmt):
        a = np.asarray(a).reshape(-1)
        vals = ", ".join(fmt(x) for x in a) if a.size else "0"
        return f"static const {ctype} {prefix}_{name}[] = {{{vals}}};\n"
    fi = lambda x: str(int(x))
    ff = lambda x: _f(x)
    s = f"// GENERATED tables for '{model.name}'\n"
    s += f"static const int {prefix}_nbody = {model.nbody}, {prefix}_njnt = {model.njnt}, {prefix}_nsite = {model.nsite}, " \
         f"{prefix}_nq = {model.nq}, {prefix}_nv = {model.nv};\n"
    s += arr("body_parentid", model.body_parentid, "int", fi)
    s += arr("body_jntadr", model.body_jntadr, "int", fi)
    s += arr("body_jntnum", model.body_jntnum, "int", fi)
    s += arr("jnt_type", model.jnt_type, "int", fi)
    s += arr("jnt_qposadr", model.jnt_qposadr, "int", fi)
    s += arr("site_bodyid", model.site_bodyid, "int", fi)
    s += arr("body_pos", model.body_pos, "float", ff)
    s += arr("body_quat", model.body_quat, "float", ff)
    s += arr("body_ipos", model.body_ipos, "float", ff)
    s += arr("body_mass", model.body_mass, "float", ff)
    s += arr("jnt_axis", model.jnt_axis, "float", ff)
    s += arr("jnt_pos", model.jnt_pos, "float", ff)
    s += arr("qpos0", model.qpos0, "float", ff)
    s += arr("site_pos", model.site_pos, "float", ff)
    s += arr("site_quat", model.site_quat, "float", ff)
    return s
