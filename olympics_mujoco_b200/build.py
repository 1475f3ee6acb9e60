"""Build libom_b200.so in-tree: run the model code generator, then nvcc for sm_100a.

    python -m olympics_mujoco_b200.build [--force]

The shared library lands at ``olympics_mujoco_b200/libom_b200.so`` (git-ignored, travels with gpurun).
nvcc cross-compiles without a GPU, so this also runs in the authoring container.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from pathlib import Path

from . import codegen, mjcf

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
GEN = CSRC / "gen"
H1V = GEN / "h1v"
LIB = PKG / "libom_b200.so"
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC",
         "--expt-relaxed-constexpr", "-Xptxas", "-v"]

H1_SPEC_JOINTS = ["pelvis_tx", "pelvis_tz", "pelvis_ty", "pelvis_tilt", "pelvis_list", "pelvis_rotation", "back_bkz",
                  "hip_flexion_r", "hip_adduction_r", "hip_rotation_r", "knee_angle_r", "ankle_angle_r",
                  "hip_flexion_l", "hip_adduction_l", "hip_rotation_l", "knee_angle_l", "ankle_angle_l"]


def _write_if_changed(path: Path, text: str):
    if path.exists() and path.read_text() == text:
        return False
    path.write_text(text)
    return True


def generate():
    """(Re)generate csrc/gen/* from the shipped model tables."""
    GEN.mkdir(exist_ok=True)
    h1 = mjcf.load_builtin("unitree_h1")
    a3 = mjcf.load_builtin("stick_figure_a3")
    _write_if_changed(GEN / "fk_unitree_h1.cuh", "#pragma once\n" + codegen.generate_fk(h1, "om_fk_unitree_h1"))
    _write_if_changed(GEN / "fk_stick_figure_a3.cuh", "#pragma once\n" + codegen.generate_fk(a3, "om_fk_stick_figure_a3"))
    _write_if_changed(GEN / "fk_pos_stick_figure_a3.cuh",
                      "#pragma once\n" + codegen.generate_fk_pos(a3, "om_fk_pos_stick_figure_a3"))
    # float64 twin of the position FK: the exact slow path of the A3 threshold decisions (done, target_reached)
    _write_if_changed(GEN / "fk_pos_f64_stick_figure_a3.cuh",
                      "#pragma once\n" + codegen.generate_fk_pos(a3, "om_fk_pos_f64_stick_figure_a3", scalar="double"))
    parts = codegen.split_parts(h1, 3)
    _write_if_changed(GEN / "fk_unitree_h1_parts.cuh", "#pragma once\n" + "".join(
        codegen.generate_fk(h1, f"om_fk_unitree_h1_part{k}", part=p) for k, p in enumerate(parts)))
    _write_if_changed(GEN / "tables_unitree_h1.h", "#pragma once\n" + codegen.generate_tables(h1, "om_tab_h1"))
    _write_if_changed(GEN / "tables_stick_figure_a3.h", "#pragma once\n" + codegen.generate_tables(a3, "om_tab_a3"))
    perm = [int(h1.jnt_qposadr[h1.jnt_names.index(j)]) for j in H1_SPEC_JOINTS]
    txt = ("#pragma once\n// GENERATED: qpos/qvel address of UnitreeH1 observation-spec entry k "
           "(UnitreeH1.py:303-355 minus the arm joints)\n"
           f"__device__ constexpr int OM_H1_PERM[17] = {{{', '.join(map(str, perm))}}};\n"
           f"static const int OM_H1_PERM_HOST[17] = {{{', '.join(map(str, perm))}}};\n")
    _write_if_changed(GEN / "h1_perm.h", txt)
    ids = dict(ROOT=a3.body_id("torso"), HEAD=a3.body_id("head"), LFOOT=a3.body_id("left_foot"),
               RFOOT=a3.body_id("right_foot"), LSITE=a3.site_id("lf_force"), RSITE=a3.site_id("rf_force"))
    txt = ("#pragma once\n// GENERATED: body / site ids the WalkingTask reads (StickFigureA3.py:95-103, "
           "walking_task.py:254-263) and the model's total mass (mj_getTotalmass)\n" +
           "".join(f"constexpr int OM_A3_{k} = {v};\n" for k, v in ids.items()) +
           f"constexpr float OM_A3_TOTAL_MASS = {codegen._f(a3.total_mass)};\n")
    _write_if_changed(GEN / "a3_ids.h", txt)
    _generate_h1_variants()


# The UnitreeH1 constructor variants with fused playback / live-step kernels: (name, unitree_h1_variant kwargs).  Id 1 is the
# default model (arms disabled, back joint kept); the ids below follow it.  A carried weight changes the FK (the COM and
# cvel see its mass), so each valid weight is a model of its own, recognised by exact table match like the others.
H1_VARIANTS = [("noback", dict(disable_back_joint=True)),
               ("arms", dict(disable_arms=False)),
               ("arms_noback", dict(disable_arms=False, disable_back_joint=True))] + \
              [(f"carry_{str(w).rstrip('0').rstrip('.').replace('.', 'p')}", dict(hold_weight=True, weight_mass=w))
               for w in mjcf.H1_VALID_WEIGHTS]
# One more kernel set for the carry models: the mass of the jointless "weight" body is read per env at run time
# (om_model_bind_env_body_mass), so a batch can hold every valid weight at once.  It is not a model of its own: a bound
# carry model launches it instead of its own variant's kernels.
H1_CARRY_ENV = "carry_env"


def _h1_descriptor(m, name, vid, env_mass_body=None):
    """FK + observation permutation + kernel descriptor of one variant (gen/h1v/<name>.cuh)."""
    from .synthetic import H1_SPEC_JOINTS as ALL_SPEC_JOINTS
    js = [j for j in ALL_SPEC_JOINTS if j in m.jnt_names]
    perm = [int(m.jnt_qposadr[m.jnt_names.index(j)]) for j in js]
    assert len(perm) == m.nq == m.nv, name
    up, p = name.upper(), ", ".join(map(str, perm))
    env = env_mass_body is not None
    return ("#pragma once\n" + codegen.generate_fk(m, f"om_fk_h1v_{name}", env_mass_body=env_mass_body) +
            f"// GENERATED: qpos/qvel address of observation-spec entry k\n"
            f"__device__ constexpr int OM_H1V_{up}_PERM[{m.nq}] = {{{p}}};\n"
            f"static const int OM_H1V_{up}_PERM_HOST[{m.nq}] = {{{p}}};\n"
            f"struct H1V_{name} {{\n"
            f"  static constexpr int ID = {vid}, NQ = {m.nq}, NBODY = {m.nbody}, NSITE = {m.nsite};\n"
            f"  static constexpr bool ENV_MASS = {'true' if env else 'false'};   // fk takes the env's body mass\n"
            f"  static OM_HD int perm(int k) {{ return OM_H1V_{up}_PERM[k]; }}\n"
            f"  static const int* perm_host() {{ return OM_H1V_{up}_PERM_HOST; }}\n"
            f"  template <class Sink>\n" +
            (f"  static OM_HD void fk(const float (&q)[NQ], const float (&qd)[NQ], Sink& S, float m) "
             f"{{ om_fk_h1v_{name}(q, qd, S, m); }}\n" if env else
             f"  static OM_HD void fk(const float (&q)[NQ], const float (&qd)[NQ], Sink& S) {{ om_fk_h1v_{name}(q, qd, S); }}\n") +
            f"}};\n")


def _generate_h1_variants():
    """Per variant, into gen/h1v/ (build products, not kept in git): FK + observation permutation + kernel descriptor
    (<name>.cuh) and the model tables it is recognised by (tables_<name>.h); list.h lists (id, name) for the model and
    trajectory code, tables.h includes every table.  om_traj.cu is compiled once per variant against its descriptor.
    carry_env.cuh: the carry model with the weight's mass as a runtime argument (no tables: no model is recognised as it)."""
    H1V.mkdir(exist_ok=True)
    listing, tables, carry_ids = [], [], []
    for vid, (name, kw) in enumerate(H1_VARIANTS, start=2):
        m = mjcf.unitree_h1_variant(**kw)
        _write_if_changed(H1V / f"{name}.cuh", _h1_descriptor(m, name, vid))
        _write_if_changed(H1V / f"tables_{name}.h", "#pragma once\n" + codegen.generate_tables(m, f"om_tab_h1v_{name}"))
        listing.append(f"X({vid}, {name})")
        tables.append(f'#include "tables_{name}.h"\n')
        if kw.get("hold_weight"):
            carry_ids.append(vid)
    carry = mjcf.unitree_h1_variant(hold_weight=True, weight_mass=mjcf.H1_VALID_WEIGHTS[0])
    body = carry.body_id("weight")
    _write_if_changed(H1V / f"{H1_CARRY_ENV}.cuh", _h1_descriptor(carry, H1_CARRY_ENV, 0, env_mass_body=body))
    _write_if_changed(H1V / "list.h",
                      "#pragma once\n// GENERATED: (variant id, name) of every UnitreeH1 variant with its own kernels\n"
                      "#define OM_H1_VARIANTS(X) " + " ".join(listing) + "\n"
                      "// the carry variants, whose weight body may take a per-env mass (kernels h1k_carry_env)\n"
                      "#define OM_H1_IS_CARRY(id) (" + " || ".join(f"(id) == {v}" for v in carry_ids) + ")\n"
                      f"#define OM_H1_CARRY_WEIGHT_BODY {body}\n")
    _write_if_changed(H1V / "tables.h", "#pragma once\n" + "".join(tables))


def compile_units():
    """(source, extra nvcc flags, object name): every .cu once, and om_traj.cu once more per UnitreeH1 variant (and for
    the per-env carry kernels)."""
    units = [(src, [], src.stem) for src in sources()]
    units += [(CSRC / "om_traj.cu", [f"-DOM_H1_VARIANT={name}", f'-DOM_H1_VARIANT_HEADER="gen/h1v/{name}.cuh"'],
               f"om_traj_h1v_{name}") for name in [n for n, _ in H1_VARIANTS] + [H1_CARRY_ENV]]
    return units


def sources():
    return sorted(CSRC.glob("*.cu"))


def _digest():
    h = hashlib.sha256()
    for p in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + list(GEN.glob("*.*")) + list(H1V.glob("*")) +
                    [PKG.parent / "include" / "om_b200.h", Path(__file__)]):
        h.update(p.name.encode())
        h.update(p.read_bytes())
    return h.hexdigest()


def build(force=False, verbose=True):
    generate()
    stamp = PKG / ".libom_b200.stamp"
    dig = _digest()
    if not force and LIB.exists() and stamp.exists() and stamp.read_text() == dig:
        return LIB
    objs = []
    objdir = PKG / "build"
    objdir.mkdir(exist_ok=True)
    procs = []
    for src, extra, stem in compile_units():
        obj = objdir / (stem + ".o")
        cmd = [NVCC, *ARCH, *FLAGS, *extra, "-I", str(PKG.parent / "include"), "-c", str(src), "-o", str(obj)]
        procs.append((stem, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = []
    failed = False
    for stem, p in procs:
        out, _ = p.communicate()
        log.append(f"==== {stem}\n{out}")
        if p.returncode != 0:
            failed = True
    (objdir / "ptxas.log").write_text("\n".join(log))
    if failed:
        sys.stderr.write("\n".join(log))
        raise RuntimeError("nvcc failed (see output above)")
    cmd = [NVCC, *ARCH, "-shared", "-o", str(LIB), *map(str, objs), "-lcudart"]
    subprocess.check_call(cmd)
    stamp.write_text(dig)
    if verbose:
        print(f"built {LIB} ({LIB.stat().st_size / 1e6:.1f} MB)")
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv)
