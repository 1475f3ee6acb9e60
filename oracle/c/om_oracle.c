/*
 * om_oracle.c -- CPU oracle in plain C, float64 (TEST INFRASTRUCTURE, NOT PRODUCT).
 *
 * A second, independently written restatement of the reference's hot path, used (a) to cross-check the
 * NumPy oracle (tests/test_oracle_c.py) and (b) as the CPU baseline timed beside the GPU numbers
 * (bench.py cpu_baseline / --impl reference): one env at a time in the reference's control flow,
 * OpenMP across envs the way the reference runs one env per Ray worker (rl/algos/ppo.py:200-230).
 *
 * Follows MuJoCo 2.3.6 engine_core_smooth.c (mj_kinematics, mj_comPos, mj_comVel) in the engine's own
 * formulation (xmat-based rotations, explicit cdof), which is NOT in /root/reference: parity unpinned by the
 * reference, see oracle/__init__.py.  H1 step logic follows loco_env_base.py:444-560, UnitreeH1.py:162-203,
 * utils/reward.py:66-74; trajectory logic utils/trajectory.py:289-323,389-401; GAE restates
 * mushroom_rl.utils.value_functions.compute_gae (call site gail_TRPO.py:126); returns rl/algos/ppo.py:68-84.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define JNT_FREE 0
#define JNT_BALL 1
#define JNT_SLIDE 2
#define JNT_HINGE 3
#define MINVAL 1e-15
#define MAXB 64
#define MAXJ 64
#define MAXV 64

typedef struct {
  int nbody, njnt, nsite, nq, nv;
  const int *body_parentid, *body_rootid, *body_jntadr, *body_jntnum;
  const int *jnt_type, *jnt_qposadr, *jnt_dofadr, *jnt_bodyid, *site_bodyid;
  const double *body_pos, *body_quat, *body_ipos, *body_mass;
  const double *jnt_axis, *jnt_pos, *qpos0, *site_pos, *site_quat;
} OrModel;

/* ---------------------------------------------------------------- mju_* helpers */
static void mul_quat(double* r, const double* a, const double* b) {
  double t[4] = {a[0] * b[0] - a[1] * b[1] - a[2] * b[2] - a[3] * b[3], a[0] * b[1] + a[1] * b[0] + a[2] * b[3] - a[3] * b[2],
                 a[0] * b[2] - a[1] * b[3] + a[2] * b[0] + a[3] * b[1], a[0] * b[3] + a[1] * b[2] - a[2] * b[1] + a[3] * b[0]};
  memcpy(r, t, sizeof t);
}
static void normalize4(double* q) {
  double n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  if (n < MINVAL) { q[0] = 1; q[1] = q[2] = q[3] = 0; return; }
  for (int i = 0; i < 4; ++i) q[i] /= n;
}
static void quat2mat(double* m, const double* q) {
  double q00 = q[0] * q[0], q01 = q[0] * q[1], q02 = q[0] * q[2], q03 = q[0] * q[3];
  double q11 = q[1] * q[1], q12 = q[1] * q[2], q13 = q[1] * q[3], q22 = q[2] * q[2], q23 = q[2] * q[3], q33 = q[3] * q[3];
  m[0] = q00 + q11 - q22 - q33; m[4] = q00 - q11 + q22 - q33; m[8] = q00 - q11 - q22 + q33;
  m[1] = 2 * (q12 - q03); m[2] = 2 * (q13 + q02); m[3] = 2 * (q12 + q03);
  m[5] = 2 * (q23 - q01); m[6] = 2 * (q13 - q02); m[7] = 2 * (q23 + q01);
}
static void rot_vec_mat(double* r, const double* v, const double* m) {
  double t[3] = {m[0] * v[0] + m[1] * v[1] + m[2] * v[2], m[3] * v[0] + m[4] * v[1] + m[5] * v[2], m[6] * v[0] + m[7] * v[1] + m[8] * v[2]};
  memcpy(r, t, sizeof t);
}
static void rot_vec_quat(double* r, const double* v, const double* q) {
  double m[9];
  quat2mat(m, q);                      /* the engine's older formulation: through the rotation matrix */
  rot_vec_mat(r, v, m);
}
static void cross3(double* r, const double* a, const double* b) {
  double t[3] = {a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]};
  memcpy(r, t, sizeof t);
}

/* ---------------------------------------------------------------- mj_kinematics + mj_comPos + mj_comVel, one env */
void or_forward(const OrModel* m, const double* qpos, const double* qvel, double* xpos, double* xquat, double* site_xpos,
                double* site_xmat, double* cvel, double* subtree_com) {
  double xmat[MAXB * 9], xipos[MAXB * 3], xanchor[MAXJ * 3], xaxis[MAXJ * 3], cdof[MAXV * 6], stm[MAXB], sub[MAXB * 3];
  const int nb = m->nbody;
  memset(xpos, 0, 3 * sizeof(double));
  xquat[0] = 1; xquat[1] = xquat[2] = xquat[3] = 0;
  memset(xmat, 0, 9 * sizeof(double)); xmat[0] = xmat[4] = xmat[8] = 1;
  memset(xipos, 0, 3 * sizeof(double));
  for (int i = 1; i < nb; ++i) {
    double pos[3], quat[4], vec[3];
    const int jadr = m->body_jntadr[i], jnum = m->body_jntnum[i];
    if (jnum == 1 && m->jnt_type[jadr] == JNT_FREE) {
      const int qa = m->jnt_qposadr[jadr];
      memcpy(pos, qpos + qa, 3 * sizeof(double));
      memcpy(quat, qpos + qa + 3, 4 * sizeof(double));
      normalize4(quat);
      memcpy(xanchor + 3 * jadr, pos, 3 * sizeof(double));
      memcpy(xaxis + 3 * jadr, m->jnt_axis + 3 * jadr, 3 * sizeof(double));
    } else {
      const int pid = m->body_parentid[i];
      rot_vec_mat(vec, m->body_pos + 3 * i, xmat + 9 * pid);
      for (int k = 0; k < 3; ++k) pos[k] = xpos[3 * pid + k] + vec[k];
      mul_quat(quat, xquat + 4 * pid, m->body_quat + 4 * i);
      for (int j = jadr; j < jadr + jnum; ++j) {
        const int qa = m->jnt_qposadr[j], jt = m->jnt_type[j];
        rot_vec_quat(xaxis + 3 * j, m->jnt_axis + 3 * j, quat);
        rot_vec_quat(xanchor + 3 * j, m->jnt_pos + 3 * j, quat);
        for (int k = 0; k < 3; ++k) xanchor[3 * j + k] += pos[k];
        if (jt == JNT_SLIDE) {
          for (int k = 0; k < 3; ++k) pos[k] += xaxis[3 * j + k] * (qpos[qa] - m->qpos0[qa]);
        } else {
          double qloc[4];
          if (jt == JNT_BALL) { memcpy(qloc, qpos + qa, 4 * sizeof(double)); normalize4(qloc); }
          else {
            const double a = qpos[qa] - m->qpos0[qa], s = sin(a * 0.5);
            qloc[0] = cos(a * 0.5);
            for (int k = 0; k < 3; ++k) qloc[1 + k] = m->jnt_axis[3 * j + k] * s;
          }
          mul_quat(quat, quat, qloc);
          rot_vec_quat(vec, m->jnt_pos + 3 * j, quat);
          for (int k = 0; k < 3; ++k) pos[k] = xanchor[3 * j + k] - vec[k];
        }
      }
    }
    normalize4(quat);
    memcpy(xquat + 4 * i, quat, sizeof quat);
    memcpy(xpos + 3 * i, pos, sizeof pos);
    quat2mat(xmat + 9 * i, quat);
  }
  for (int i = 1; i < nb; ++i) {
    double v[3];
    rot_vec_mat(v, m->body_ipos + 3 * i, xmat + 9 * i);
    for (int k = 0; k < 3; ++k) xipos[3 * i + k] = xpos[3 * i + k] + v[k];
  }
  for (int s = 0; s < m->nsite; ++s) {
    const int b = m->site_bodyid[s];
    double v[3], q[4];
    rot_vec_mat(v, m->site_pos + 3 * s, xmat + 9 * b);
    if (site_xpos) for (int k = 0; k < 3; ++k) site_xpos[3 * s + k] = xpos[3 * b + k] + v[k];
    if (site_xmat) { mul_quat(q, xquat + 4 * b, m->site_quat + 4 * s); quat2mat(site_xmat + 9 * s, q); }
  }
  /* mj_comPos */
  for (int i = 0; i < nb; ++i) stm[i] = m->body_mass[i];
  for (int i = nb - 1; i > 0; --i) stm[m->body_parentid[i]] += stm[i];
  memset(sub, 0, sizeof(double) * 3 * nb);
  for (int i = nb - 1; i >= 0; --i) {
    for (int k = 0; k < 3; ++k) sub[3 * i + k] += xipos[3 * i + k] * m->body_mass[i];
    if (i) for (int k = 0; k < 3; ++k) sub[3 * m->body_parentid[i] + k] += sub[3 * i + k];
    if (stm[i] < MINVAL) memcpy(sub + 3 * i, xipos + 3 * i, 3 * sizeof(double));
    else for (int k = 0; k < 3; ++k) sub[3 * i + k] *= 1.0 / (stm[i] > MINVAL ? stm[i] : MINVAL);
  }
  if (subtree_com) memcpy(subtree_com, sub, sizeof(double) * 3 * nb);
  memset(cdof, 0, sizeof(double) * 6 * m->nv);
  for (int j = 0; j < m->njnt; ++j) {
    int da = 6 * m->jnt_dofadr[j];
    const int bi = m->jnt_bodyid[j];
    double off[3], axis[3];
    for (int k = 0; k < 3; ++k) off[k] = sub[3 * m->body_rootid[bi] + k] - xanchor[3 * j + k];
    switch (m->jnt_type[j]) {
      case JNT_FREE:
        for (int i = 0; i < 3; ++i) cdof[da + 3 + 7 * i] = 1;
        da += 18;
        /* fall through */
      case JNT_BALL:
        for (int i = 0; i < 3; ++i) {
          axis[0] = xmat[9 * bi + i]; axis[1] = xmat[9 * bi + i + 3]; axis[2] = xmat[9 * bi + i + 6];
          memcpy(cdof + da + 6 * i, axis, sizeof axis);
          cross3(cdof + da + 6 * i + 3, axis, off);
        }
        break;
      case JNT_SLIDE:
        memcpy(cdof + da + 3, xaxis + 3 * j, 3 * sizeof(double));
        break;
      case JNT_HINGE:
        memcpy(cdof + da, xaxis + 3 * j, 3 * sizeof(double));
        cross3(cdof + da + 3, xaxis + 3 * j, off);
        break;
    }
  }
  /* mj_comVel */
  if (cvel) {
    memset(cvel, 0, 6 * sizeof(double));
    for (int i = 1; i < nb; ++i) {
      double v[6];
      memcpy(v, cvel + 6 * m->body_parentid[i], sizeof v);
      for (int j = m->body_jntadr[i]; j < m->body_jntadr[i] + m->body_jntnum[i]; ++j) {
        const int da = m->jnt_dofadr[j];
        const int nd = m->jnt_type[j] == JNT_FREE ? 6 : (m->jnt_type[j] == JNT_BALL ? 3 : 1);
        for (int d = da; d < da + nd; ++d)
          for (int k = 0; k < 6; ++k) v[k] += cdof[6 * d + k] * qvel[d];
      }
      memcpy(cvel + 6 * i, v, sizeof v);
    }
  }
}

void or_forward_batch(const OrModel* m, const double* qpos, const double* qvel, int n, double* xpos, double* xquat,
                      double* site_xpos, double* site_xmat, double* cvel, double* subtree_com) {
#pragma omp parallel for schedule(static)
  for (int e = 0; e < n; ++e)
    or_forward(m, qpos + (size_t)e * m->nq, qvel + (size_t)e * m->nv, xpos + (size_t)e * m->nbody * 3,
               xquat + (size_t)e * m->nbody * 4, site_xpos ? site_xpos + (size_t)e * m->nsite * 3 : 0,
               site_xmat ? site_xmat + (size_t)e * m->nsite * 9 : 0, cvel + (size_t)e * m->nbody * 6,
               subtree_com ? subtree_com + (size_t)e * m->nbody * 3 : 0);
}

/* ---------------------------------------------------------------- Philox contract (oracle/philox.py) */
static void philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out) {
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
static void traj_draw(uint64_t seed, uint32_t env, uint32_t count, int n_traj, int T, int* traj_no, int* step_no) {
  uint32_t w[4];
  philox(env, count, 0, 0, (uint32_t)seed, (uint32_t)(seed >> 32), w);
  *traj_no = (int)(((uint64_t)w[0] * (uint64_t)n_traj) >> 32);
  *step_no = (int)(((uint64_t)w[1] * (uint64_t)T) >> 32);
}

/* ---------------------------------------------------------------- H1 step pieces */
static int h1_has_fallen(const double* obs) {
  const double PI = 3.141592653589793;
  return (obs[0] < -0.3) || (obs[0] > 0.1) || (obs[1] < (-PI / 4.5)) || (obs[1] > (PI / 12)) ||
         (obs[2] < -PI / 12) || (obs[2] > PI / 8) || (obs[3] < (-PI / 8)) || (obs[3] > (PI / 8));
}

/* What one env carries from one playback call to the next (the device's OmPlayState), env-major: traj_no, step_no,
 * reset_count [n_env]; xy_off [n_env][2]; curr_qpos [n_env][K/2]; pending [n_env][K], the loop's `sample` variable
 * (x, y re-centred), which stays the stale one across the end-of-episode reset; prev_x_vel [n_env], dq_pelvis_tx of
 * the previous observation. */
typedef struct {
  int32_t *traj_no, *step_no;
  uint32_t* reset_count;
  double *xy_off, *curr_qpos, *pending, *prev_x_vel;
} OrPlayState;

/* play_trajectory_from_velocity for the envs env_id0 .. env_id0 + n_env - 1: n_episodes episodes of n_steps
 * (loco_env_base.py:444-560), each ending with reset() (:555-557).  start_reset: the call begins with reset()
 * (:481-508); 0 carries the state of the previous call on (the device's continue_episode).  `ps` is read at the start
 * and written at the end; NULL = a fresh env (reset_count 0, start_reset required) whose final state is dropped.
 * table [K][n_traj][T] float64.  Outputs (any may be NULL) are env-major [n_env][n_episodes * n_steps][...];
 * `checksum` [n_env] always receives a sum over everything computed, so that a timing run without outputs cannot be
 * optimised away. */
void or_h1_play_chain(const OrModel* m, const int* perm, const double* table, int K, int n_traj, int T, uint64_t seed,
                      uint32_t env_id0, int n_env, int n_episodes, int n_steps, int start_reset, double dt, double target,
                      const OrPlayState* ps, double* xpos, double* xquat, double* site_xpos, double* cvel, double* obs,
                      double* reward, uint8_t* fallen, int32_t* traj_no_t, int32_t* step_no_t, double* checksum) {
  const int nj = K / 2, nb = m->nbody;
  const size_t n_slots = (size_t)n_episodes * n_steps;
#pragma omp parallel for schedule(static)
  for (int e = 0; e < n_env; ++e) {
    double sample[64], curr[32], qpos[MAXV], qvel[MAXV], bx[MAXB * 3], bq[MAXB * 4], bs[24], bc[MAXB * 6], ob[64];
    int tr = 0, st = 0;
    uint32_t rc = ps ? ps->reset_count[e] : 0;
    double ox = 0.0, oy = 0.0, acc = 0.0, prev_xv = 0.0;
#define TAB(k, tr_, s_) table[((size_t)(k) * n_traj + (tr_)) * T + (s_)]
#define LOAD_SAMPLE()                                                          \
  do {                                                                         \
    for (int k = 0; k < K; ++k) sample[k] = TAB(k, tr, st);                    \
    sample[0] -= ox; sample[1] -= oy;                                          \
  } while (0)
    if (start_reset || !ps) {
      traj_draw(seed, env_id0 + e, rc++, n_traj, T, &tr, &st);                  /* :481 reset() */
      ox = TAB(0, tr, st); oy = TAB(1, tr, st);
      LOAD_SAMPLE();                                                            /* :483 */
      prev_xv = sample[nj];                                                     /* obs[15] of reset() */
      for (int k = 0; k < nj; ++k) curr[k] = sample[k];                         /* :508 */
    } else {
      tr = ps->traj_no[e]; st = ps->step_no[e];
      ox = ps->xy_off[2 * e]; oy = ps->xy_off[2 * e + 1];
      memcpy(sample, ps->pending + (size_t)e * K, sizeof(double) * K);
      memcpy(curr, ps->curr_qpos + (size_t)e * nj, sizeof(double) * nj);
      prev_xv = ps->prev_x_vel[e];
    }
    for (int ep = 0; ep < n_episodes; ++ep) {
      for (int s = 0; s < n_steps; ++s) {
        for (int k = 0; k < nj; ++k) {                                          /* :515-521 */
          const double qs = curr[k] + dt * sample[nj + k];
          qpos[perm[k]] = qs; qvel[perm[k]] = sample[nj + k];
          curr[k] = qs;                                                         /* :529 */
        }
        or_forward(m, qpos, qvel, bx, bq, bs, 0, bc, 0);                        /* :525 mj_forward subset */
        const size_t slot = (size_t)e * n_slots + (size_t)ep * n_steps + s;
        if (xpos) memcpy(xpos + slot * nb * 3, bx, sizeof(double) * nb * 3);
        if (xquat) memcpy(xquat + slot * nb * 4, bq, sizeof(double) * nb * 4);
        if (site_xpos) memcpy(site_xpos + slot * m->nsite * 3, bs, sizeof(double) * m->nsite * 3);
        if (cvel) memcpy(cvel + slot * nb * 6, bc, sizeof(double) * nb * 6);
        acc += bx[3 * (nb - 1)] + bq[4 * (nb - 1)] + bc[6 * (nb - 1) + 3];
        ++st;                                                                   /* :532 */
        if (st == T) {                                                          /* :534-537 */
          traj_draw(seed, env_id0 + e, rc++, n_traj, T, &tr, &st);
          ox = TAB(0, tr, st); oy = TAB(1, tr, st);
          LOAD_SAMPLE();
          for (int k = 0; k < nj; ++k) curr[k] = sample[k];
        } else {
          LOAD_SAMPLE();
        }
        for (int k = 0; k < K - 2; ++k) ob[k] = sample[k + 2];                  /* :539 */
        const int f = h1_has_fallen(ob);                                        /* :541 */
        const double r = exp(-(prev_xv - target) * (prev_xv - target));         /* reward.py:72-74 on the previous obs */
        prev_xv = ob[nj - 2];
        if (obs) memcpy(obs + slot * (K - 2), ob, sizeof(double) * (K - 2));
        if (reward) reward[slot] = r;
        if (fallen) fallen[slot] = (uint8_t)f;
        if (traj_no_t) traj_no_t[slot] = tr;
        if (step_no_t) step_no_t[slot] = st;
        acc += r + f + ob[0];
      }
      traj_draw(seed, env_id0 + e, rc++, n_traj, T, &tr, &st);                  /* :555 reset(); `sample` stays stale */
      ox = TAB(0, tr, st); oy = TAB(1, tr, st);
      curr[0] = 0.0; curr[1] = 0.0;                                             /* :557, x and y re-centred: exactly 0 */
      for (int k = 2; k < nj; ++k) curr[k] = TAB(k, tr, st);
      prev_xv = TAB(nj, tr, st);
    }
    checksum[e] = acc;
    if (ps) {
      ps->traj_no[e] = tr; ps->step_no[e] = st; ps->reset_count[e] = rc;
      ps->xy_off[2 * e] = ox; ps->xy_off[2 * e + 1] = oy;
      memcpy(ps->pending + (size_t)e * K, sample, sizeof(double) * K);
      memcpy(ps->curr_qpos + (size_t)e * nj, curr, sizeof(double) * nj);
      ps->prev_x_vel[e] = prev_xv;
    }
#undef TAB
#undef LOAD_SAMPLE
  }
}

/* One episode of n_steps from a fresh reset for each env (outputs [n_env][n_steps][...]): the CPU baseline's call. */
void or_h1_play(const OrModel* m, const int* perm, const double* table, int K, int n_traj, int T, uint64_t seed,
                uint32_t env_id0, int n_env, int n_steps, double dt, double target, double* xpos, double* xquat,
                double* site_xpos, double* cvel, double* obs, double* reward, uint8_t* fallen, int32_t* traj_no_t,
                int32_t* step_no_t, double* checksum) {
  or_h1_play_chain(m, perm, table, K, n_traj, T, seed, env_id0, n_env, 1, n_steps, 1, dt, target, 0, xpos, xquat,
                   site_xpos, cvel, obs, reward, fallen, traj_no_t, step_no_t, checksum);
}

/* ---------------------------------------------------------------- compute_gae per env over [n_env][T] (env-major) */
void or_gae(const double* r, const double* v, const double* v_next, const uint8_t* absorbing, const uint8_t* last,
            double gamma, double lam, int n_env, int T, double* adv, double* v_target) {
#pragma omp parallel for schedule(static)
  for (int e = 0; e < n_env; ++e) {
    const size_t o = (size_t)e * T;
    for (int k = T - 1; k >= 0; --k) {
      if ((last && last[o + k]) || k == T - 1) {
        adv[o + k] = r[o + k] - v[o + k];
        if (!(absorbing && absorbing[o + k])) adv[o + k] += gamma * v_next[o + k];
      } else {
        adv[o + k] = r[o + k] + gamma * v_next[o + k] - v[o + k] + gamma * lam * adv[o + k + 1];
      }
    }
    for (int k = 0; k < T; ++k) v_target[o + k] = adv[o + k] + v[o + k];
  }
}

/* PPOBuffer.finish_path for n_env single paths of length T (rl/algos/ppo.py:68-84) */
void or_ppo_returns(const double* r, const double* last_val, double gamma, int n_env, int T, double* ret) {
#pragma omp parallel for schedule(static)
  for (int e = 0; e < n_env; ++e) {
    double R = last_val[e];
    for (int k = T - 1; k >= 0; --k) { R = gamma * R + r[(size_t)e * T + k]; ret[(size_t)e * T + k] = R; }
  }
}

int or_num_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

/* torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU baseline is supposed to use the host cores */
void or_set_num_threads(int n) {
#ifdef _OPENMP
  if (n > 0) omp_set_num_threads(n);
#else
  (void)n;
#endif
}
