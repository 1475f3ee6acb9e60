// K1, table-driven flavour: mj_kinematics + mj_comPos + mj_comVel for ANY model that fits ModelTab.
// One thread per environment, the model tables ("topology") staged in shared memory once per CTA,
// structure-of-arrays HBM I/O (every load/store of a warp is one 128-byte line).  Per-thread body state
// lives in local memory (L1-resident); the generated kernels in gen/fk_*.cuh are the register-only,
// constant-folded version of exactly this loop for the two in-scope robots.
#pragma once
#include "om_common.cuh"

namespace om {

struct FkOut {
  float* xpos; float* xquat; float* site_xpos; float* site_xmat; float* cvel; float* com;
};

// ENV_MASS: body em.body's mass is em.mass[env] (om_model_bind_env_body_mass), its tree's inverse mass 1 / (em.m0 + mass)
struct FkEnvMass {
  const float* mass;
  int body;
  float m0;
};

template <bool ENV_MASS>
__global__ void __launch_bounds__(128) fk_generic_kernel(const ModelTab* __restrict__ gtab,
                                                         const float* __restrict__ qpos,
                                                         const float* __restrict__ qvel, int n, int ld, FkOut o,
                                                         FkEnvMass em) {
  __shared__ ModelTab tab;
  {
    const int* src = reinterpret_cast<const int*>(gtab);
    int* dst = reinterpret_cast<int*>(&tab);
    for (int i = threadIdx.x; i < (int)(sizeof(ModelTab) / 4); i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n) return;
  const int nb = tab.nbody;
  const float env_m = ENV_MASS ? em.mass[env] : 0.f;

  float px[MAXB], py[MAXB], pz[MAXB];
  float qw[MAXB], qx[MAXB], qy[MAXB], qz[MAXB];
  float wx[MAXB], wy[MAXB], wz[MAXB], vx[MAXB], vy[MAXB], vz[MAXB];
  float cax[MAXB], cay[MAXB], caz[MAXB];     // per tree root: sum m*xipos, later com - P
  float Px[MAXB], Py[MAXB], Pz[MAXB];        // per tree root: reference point (root body origin)
  px[0] = py[0] = pz[0] = 0.f; qw[0] = 1.f; qx[0] = qy[0] = qz[0] = 0.f;
  wx[0] = wy[0] = wz[0] = vx[0] = vy[0] = vz[0] = 0.f;
  for (int i = 0; i < nb; ++i) { cax[i] = cay[i] = caz[i] = 0.f; Px[i] = Py[i] = Pz[i] = 0.f; }

  auto Q = [&](int k) { return qpos[(size_t)k * ld + env]; };
  auto QD = [&](int k) { return qvel ? qvel[(size_t)k * ld + env] : 0.f; };

  for (int i = 1; i < nb; ++i) {
    const int pid = tab.body_parent[i], rid = tab.body_root[i];
    const int jadr = tab.body_jntadr[i], jnum = tab.body_jntnum[i];
    V3 p; Q4 qt;
    V3 w{wx[pid], wy[pid], wz[pid]}, v{vx[pid], vy[pid], vz[pid]};
    if (jnum == 1 && tab.jnt_type[jadr] == OM_JNT_FREE) {
      const int qa = tab.jnt_qposadr[jadr], da = tab.jnt_dofadr[jadr];
      p = V3{Q(qa), Q(qa + 1), Q(qa + 2)};
      qt = qnormalize(Q4{Q(qa + 3), Q(qa + 4), Q(qa + 5), Q(qa + 6)});
      if (rid == i) { Px[rid] = p.x; Py[rid] = p.y; Pz[rid] = p.z; }
      v = v + V3{QD(da), QD(da + 1), QD(da + 2)};
      V3 arm = V3{Px[rid], Py[rid], Pz[rid]} - p;
      for (int k = 0; k < 3; ++k) {
        V3 axis = qrot(qt, V3{k == 0 ? 1.f : 0.f, k == 1 ? 1.f : 0.f, k == 2 ? 1.f : 0.f});
        float d = QD(da + 3 + k);
        w = fma3(axis, d, w);
        v = fma3(cross(axis, arm), d, v);
      }
    } else {
      Q4 pq{qw[pid], qx[pid], qy[pid], qz[pid]};
      p = V3{px[pid], py[pid], pz[pid]} + qrot(pq, V3{tab.body_pos[3 * i], tab.body_pos[3 * i + 1], tab.body_pos[3 * i + 2]});
      qt = qmul(pq, Q4{tab.body_quat[4 * i], tab.body_quat[4 * i + 1], tab.body_quat[4 * i + 2], tab.body_quat[4 * i + 3]});
      V3 jaxis[8], janchor[8];
      for (int jj = 0; jj < jnum; ++jj) {
        const int j = jadr + jj, jt = tab.jnt_type[j], qa = tab.jnt_qposadr[j];
        V3 ax{tab.jnt_axis[3 * j], tab.jnt_axis[3 * j + 1], tab.jnt_axis[3 * j + 2]};
        V3 jp{tab.jnt_pos[3 * j], tab.jnt_pos[3 * j + 1], tab.jnt_pos[3 * j + 2]};
        jaxis[jj] = qrot(qt, ax);
        janchor[jj] = qrot(qt, jp) + p;
        if (jt == OM_JNT_SLIDE) {
          p = fma3(jaxis[jj], Q(qa) - tab.qpos0[qa], p);
        } else if (jt == OM_JNT_HINGE) {
          float s, c;
          om_sincos(0.5f * (Q(qa) - tab.qpos0[qa]), &s, &c);
          qt = qmul(qt, Q4{c, ax.x * s, ax.y * s, ax.z * s});
          p = janchor[jj] - qrot(qt, jp);
        } else if (jt == OM_JNT_BALL) {
          qt = qmul(qt, qnormalize(Q4{Q(qa), Q(qa + 1), Q(qa + 2), Q(qa + 3)}));
          p = janchor[jj] - qrot(qt, jp);
        }
      }
      if (rid == i) { Px[rid] = p.x; Py[rid] = p.y; Pz[rid] = p.z; }
      const V3 P{Px[rid], Py[rid], Pz[rid]};
      for (int jj = 0; jj < jnum; ++jj) {
        const int j = jadr + jj, jt = tab.jnt_type[j], da = tab.jnt_dofadr[j];
        if (jt == OM_JNT_SLIDE) {
          v = fma3(jaxis[jj], QD(da), v);
        } else if (jt == OM_JNT_HINGE) {
          float d = QD(da);
          w = fma3(jaxis[jj], d, w);
          v = fma3(cross(jaxis[jj], P - janchor[jj]), d, v);
        } else if (jt == OM_JNT_BALL) {
          // rotation about the body axes (columns of the FINAL xmat, mj_comPos) through the anchor
          Q4 qf = qnormalize(qt);
          for (int k = 0; k < 3; ++k) {
            V3 axis = qrot(qf, V3{k == 0 ? 1.f : 0.f, k == 1 ? 1.f : 0.f, k == 2 ? 1.f : 0.f});
            float d = QD(da + k);
            w = fma3(axis, d, w);
            v = fma3(cross(axis, P - janchor[jj]), d, v);
          }
        }
      }
      qt = qnormalize(qt);
    }
    px[i] = p.x; py[i] = p.y; pz[i] = p.z;
    qw[i] = qt.w; qx[i] = qt.x; qy[i] = qt.y; qz[i] = qt.z;
    wx[i] = w.x; wy[i] = w.y; wz[i] = w.z; vx[i] = v.x; vy[i] = v.y; vz[i] = v.z;
    const float m = (ENV_MASS && i == em.body) ? env_m : tab.body_mass[i];
    V3 xi = p + qrot(qt, V3{tab.body_ipos[3 * i], tab.body_ipos[3 * i + 1], tab.body_ipos[3 * i + 2]});
    cax[rid] = fmaf(xi.x, m, cax[rid]); cay[rid] = fmaf(xi.y, m, cay[rid]); caz[rid] = fmaf(xi.z, m, caz[rid]);
  }

  // outputs
  if (o.xpos)
    for (int i = 0; i < nb; ++i) {
      o.xpos[(size_t)(3 * i) * ld + env] = px[i];
      o.xpos[(size_t)(3 * i + 1) * ld + env] = py[i];
      o.xpos[(size_t)(3 * i + 2) * ld + env] = pz[i];
    }
  if (o.xquat)
    for (int i = 0; i < nb; ++i) {
      o.xquat[(size_t)(4 * i) * ld + env] = qw[i];
      o.xquat[(size_t)(4 * i + 1) * ld + env] = qx[i];
      o.xquat[(size_t)(4 * i + 2) * ld + env] = qy[i];
      o.xquat[(size_t)(4 * i + 3) * ld + env] = qz[i];
    }
  for (int s = 0; s < tab.nsite; ++s) {
    const int b = tab.site_body[s];
    Q4 bq{qw[b], qx[b], qy[b], qz[b]};
    if (o.site_xpos) {
      V3 sp = V3{px[b], py[b], pz[b]} + qrot(bq, V3{tab.site_pos[3 * s], tab.site_pos[3 * s + 1], tab.site_pos[3 * s + 2]});
      o.site_xpos[(size_t)(3 * s) * ld + env] = sp.x;
      o.site_xpos[(size_t)(3 * s + 1) * ld + env] = sp.y;
      o.site_xpos[(size_t)(3 * s + 2) * ld + env] = sp.z;
    }
    if (o.site_xmat) {
      float mm[9];
      quat2mat(qmul(bq, Q4{tab.site_quat[4 * s], tab.site_quat[4 * s + 1], tab.site_quat[4 * s + 2], tab.site_quat[4 * s + 3]}), mm);
      for (int k = 0; k < 9; ++k) o.site_xmat[(size_t)(9 * s + k) * ld + env] = mm[k];
    }
  }
  // com - P per tree; a massless tree falls back to its root's position (mj_comPos: xipos)
  for (int i = 1; i < nb; ++i)
    if (tab.body_root[i] == i) {
      const float im = (ENV_MASS && i == tab.body_root[em.body]) ? 1.f / (em.m0 + env_m) : tab.tree_inv_mass[i];
      if (im > 0.f) { cax[i] = cax[i] * im; cay[i] = cay[i] * im; caz[i] = caz[i] * im; }
      else { cax[i] = px[i]; cay[i] = py[i]; caz[i] = pz[i]; }
      if (i == 1 && o.com) {
        o.com[env] = cax[i]; o.com[(size_t)ld + env] = cay[i]; o.com[(size_t)2 * ld + env] = caz[i];
      }
      cax[i] -= Px[i]; cay[i] -= Py[i]; caz[i] -= Pz[i];
    }
  if (o.cvel)
    for (int i = 0; i < nb; ++i) {
      const int rid = tab.body_root[i];
      V3 w{wx[i], wy[i], wz[i]};
      V3 lin = V3{vx[i], vy[i], vz[i]} + cross(w, V3{cax[rid], cay[rid], caz[rid]});
      if (i == 0) lin = V3{0.f, 0.f, 0.f};
      o.cvel[(size_t)(6 * i) * ld + env] = w.x;
      o.cvel[(size_t)(6 * i + 1) * ld + env] = w.y;
      o.cvel[(size_t)(6 * i + 2) * ld + env] = w.z;
      o.cvel[(size_t)(6 * i + 3) * ld + env] = lin.x;
      o.cvel[(size_t)(6 * i + 4) * ld + env] = lin.y;
      o.cvel[(size_t)(6 * i + 5) * ld + env] = lin.z;
    }
}

}  // namespace om
