// K1 entry point (om_fk) and K2/H1 (om_h1_step, om_h1_has_fallen).
#include <cstdlib>

#include "om_common.cuh"
#include "om_fk_generic.cuh"
#include "om_sinks.cuh"
#include "gen/fk_unitree_h1.cuh"
#include "gen/h1_perm.h"
#include "gen/fk_unitree_h1_parts.cuh"
#include "gen/fk_stick_figure_a3.cuh"

namespace om {

// ---------------------------------------------------------------- specialised FK kernels
template <int MODEL> struct FkSpec;
template <> struct FkSpec<SPEC_H1> {
  static constexpr int NQ = 17, NV = 17;
  template <class S> static OM_HD void run(const float (&q)[17], const float (&qd)[17], S& s) { om_fk_unitree_h1(q, qd, s); }
};
template <> struct FkSpec<SPEC_A3> {
  static constexpr int NQ = 25, NV = 24;
  template <class S> static OM_HD void run(const float (&q)[25], const float (&qd)[24], S& s) { om_fk_stick_figure_a3(q, qd, s); }
};

template <int MODEL, int BLOCK>
__global__ void __launch_bounds__(BLOCK) fk_spec_kernel(const float* __restrict__ qpos, const float* __restrict__ qvel,
                                                        int n, int ld, FkOut o) {
  using M = FkSpec<MODEL>;
  const int env = blockIdx.x * BLOCK + threadIdx.x;
  if (env >= n) return;
  float q[M::NQ], qd[M::NV];
#pragma unroll
  for (int k = 0; k < M::NQ; ++k) q[k] = qpos[(size_t)k * ld + env];
#pragma unroll
  for (int k = 0; k < M::NV; ++k) qd[k] = qvel ? qvel[(size_t)k * ld + env] : 0.f;
  SoaSink<true> S{o.xpos, o.xquat, o.site_xpos, o.site_xmat, o.cvel, o.com, (size_t)ld, (size_t)env};
  M::run(q, qd, S);
}

// ---------------------------------------------------------------- H1 observation / reward / absorbing
// has_fallen thresholds are float64 in the reference (UnitreeH1.py:176-179); comparing the fp32 value in
// double keeps the flag bit-exact with the float64 oracle on fp32-representable inputs.
OM_HD bool h1_has_fallen(float y, float tilt, float lst, float rot) {
  const double PI = 3.141592653589793;
  const double dy = y, dt = tilt, dl = lst, dr = rot;
  const bool cy = (dy < -0.3) || (dy > 0.1);
  const bool ct = (dt < (-PI / 4.5)) || (dt > (PI / 12));
  const bool cl = (dl < -PI / 12) || (dl > PI / 8);
  const bool cr = (dr < (-PI / 8)) || (dr > (PI / 8));
  return cy || ct || cl || cr;
}

struct H1SpecDev {
  int n_obs_q, x_vel_idx, use_absorbing;
  float target;
  int perm[32];
};

// obs / reward / absorbing from qpos/qvel (SoA pass; one thread per env, every access coalesced)
__device__ __forceinline__ void h1_obs_reward(const H1SpecDev& sp, const float* __restrict__ qpos,
                                              const float* __restrict__ qvel, const float* __restrict__ prev_x_vel,
                                              int ld, int env, float* __restrict__ obs, float* __restrict__ reward,
                                              uint8_t* __restrict__ absorbing) {
  const int nq = sp.n_obs_q;
  float head[4] = {0.f, 0.f, 0.f, 0.f};
  // fixed trip count + predicate: the (up to 64) loads issue back to back instead of one round trip per iteration
  float qv[32], dv[32];
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    if (k < nq) {
      qv[k] = qpos[(size_t)sp.perm[k] * ld + env];
      dv[k] = qvel[(size_t)sp.perm[k] * ld + env];
    }
  }
#pragma unroll
  for (int k = 2; k < 32; ++k) {
    if (k < nq) {
      if (k < 6) head[k - 2] = qv[k];
      if (obs) obs[(size_t)(k - 2) * ld + env] = qv[k];
    }
  }
  if (obs) {
#pragma unroll
    for (int k = 0; k < 32; ++k)
      if (k < nq) obs[(size_t)(nq - 2 + k) * ld + env] = dv[k];
  }
  if (absorbing) absorbing[env] = (sp.use_absorbing && h1_has_fallen(head[0], head[1], head[2], head[3])) ? 1 : 0;
  if (reward) {
    const float d = prev_x_vel[env] - sp.target;
    reward[env] = expf(-(d * d));
  }
}

// STATIC_PERM: the observation spec is UnitreeH1's own (checked on the host against the generated table), so the
// observation rows are a compile-time permutation of the 34 values the FK loads anyway -- no second, indirectly indexed
// pass over qpos / qvel (whose runtime-length loop issued its 34 loads one round trip at a time: two thirds of a thread's
// life at 1M envs).
// STREAM: the FK outputs leave through streaming stores.  Measured on CUDA-graph replays of consecutive steps: 131 072 envs
// 32.8 -> 29.4 us (0.85 -> 0.95 of HBM), 1 048 576 envs 0.249 -> 0.253 ms -- chosen by the batch size on the host.
constexpr int H1_STREAM_MAX_ENVS = 524288;
template <int BLOCK, bool WRITE_FK, bool STATIC_PERM, bool STREAM>
__global__ void __launch_bounds__(BLOCK) h1_step_kernel(H1SpecDev sp, const float* __restrict__ qpos,
                                                        const float* __restrict__ qvel,
                                                        const float* __restrict__ prev_x_vel, int n, int ld, FkOut o,
                                                        float* __restrict__ obs, float* __restrict__ reward,
                                                        uint8_t* __restrict__ absorbing) {
  const int env = blockIdx.x * BLOCK + threadIdx.x;
  if (env >= n) return;
  if (!STATIC_PERM) h1_obs_reward(sp, qpos, qvel, prev_x_vel, ld, env, obs, reward, absorbing);
  if (WRITE_FK || STATIC_PERM) {
    float q[17], qd[17];
#pragma unroll
    for (int k = 0; k < 17; ++k) q[k] = qpos[(size_t)k * ld + env];
#pragma unroll
    for (int k = 0; k < 17; ++k) qd[k] = qvel[(size_t)k * ld + env];
    if (STATIC_PERM) {
      if (obs) {
#pragma unroll
        for (int k = 2; k < 17; ++k) obs[(size_t)(k - 2) * ld + env] = q[OM_H1_PERM[k]];
#pragma unroll
        for (int k = 0; k < 17; ++k) obs[(size_t)(15 + k) * ld + env] = qd[OM_H1_PERM[k]];
      }
      if (absorbing)
        absorbing[env] = (sp.use_absorbing && h1_has_fallen(q[OM_H1_PERM[2]], q[OM_H1_PERM[3]], q[OM_H1_PERM[4]], q[OM_H1_PERM[5]])) ? 1 : 0;
      if (reward) {
        const float d = prev_x_vel[env] - sp.target;
        reward[env] = expf(-(d * d));
      }
    }
    if (WRITE_FK) {
      SoaSink<false, STREAM> S{o.xpos, o.xquat, o.site_xpos, nullptr, o.cvel, o.com, (size_t)ld, (size_t)env};
      om_fk_unitree_h1(q, qd, S);
    }
  }
}

// ---------------------------------------------------------------- H1 step, three threads per env
// For SMALL batches (a few thousand envs cannot fill 148 SMs with one thread each) the H1 tree splits at the pelvis into three subtrees of similar cost -- left leg, right
// leg, torso with the (jointless) arms -- so a CTA of three warps takes 32 envs: warp w evaluates subtree w (and the
// six pelvis joints above it, redundantly) with the generated part functions; lanes stay on the env axis, every warp
// runs one code path.  The only exchange is the tree's centre of mass (3 floats per part and env through shared memory,
// one barrier), needed to shift the body velocities to cvel.
struct PredSoaSink {
  static constexpr bool want_site_xmat = false;
  SoaSink<false> s;
  bool live;
  OM_HD void xpos(int b, float x, float y, float z) const { if (live) s.xpos(b, x, y, z); }
  OM_HD void xquat(int b, float w, float x, float y, float z) const { if (live) s.xquat(b, w, x, y, z); }
  OM_HD void site_xpos(int i, float x, float y, float z) const { if (live) s.site_xpos(i, x, y, z); }
  OM_HD void site_xmat(int, float, float, float, float, float, float, float, float, float) const {}
  OM_HD void cvel(int b, float wx, float wy, float wz, float vx, float vy, float vz) const { if (live) s.cvel(b, wx, wy, wz, vx, vy, vz); }
  OM_HD void com(float x, float y, float z) const { if (live) s.com(x, y, z); }
  OM_HD void vel_p(int, float, float, float, float, float, float) const {}
};
struct SmemComExchange {
  float (*part_sum)[3][32];          // [part][xyz][lane]
  int part, lane;
  __device__ __forceinline__ void com_exchange(float sx, float sy, float sz, float inv_mass, float& cx, float& cy, float& cz) const {
    part_sum[part][0][lane] = sx; part_sum[part][1][lane] = sy; part_sum[part][2][lane] = sz;
    __syncthreads();
    // same summation order in every part: the three warps see bit-identical centres of mass
    cx = ((part_sum[0][0][lane] + part_sum[1][0][lane]) + part_sum[2][0][lane]) * inv_mass;
    cy = ((part_sum[0][1][lane] + part_sum[1][1][lane]) + part_sum[2][1][lane]) * inv_mass;
    cz = ((part_sum[0][2][lane] + part_sum[1][2][lane]) + part_sum[2][2][lane]) * inv_mass;
  }
};

template <bool STATIC_PERM>
__global__ void __launch_bounds__(96) h1_step_split_kernel(H1SpecDev sp, const float* __restrict__ qpos,
                                                           const float* __restrict__ qvel,
                                                           const float* __restrict__ prev_x_vel, int n, int ld, FkOut o,
                                                           float* __restrict__ obs, float* __restrict__ reward,
                                                           uint8_t* __restrict__ absorbing) {
  __shared__ float part_sum[3][3][32];
  const int lane = threadIdx.x, part = threadIdx.y;
  const int env = blockIdx.x * 32 + lane;
  const bool live = env < n;
  const int e = live ? env : n - 1;                  // dead lanes compute on the last env, store nothing
  float q[17], qd[17];
#pragma unroll
  for (int k = 0; k < 17; ++k) q[k] = qpos[(size_t)k * ld + e];       // each part keeps the loads it uses
#pragma unroll
  for (int k = 0; k < 17; ++k) qd[k] = qvel[(size_t)k * ld + e];
  // observation rows (a permuted copy of qpos / qvel), reward and flag: split over the three warps
  if (live) {
    if (STATIC_PERM) {                               // UnitreeH1's own spec: rows straight out of the registers
      if (obs) {
#pragma unroll
        for (int k = 2; k < 17; ++k)
          if ((k - 2) % 3 == part) obs[(size_t)(k - 2) * ld + env] = q[OM_H1_PERM[k]];
#pragma unroll
        for (int k = 0; k < 17; ++k)
          if (k % 3 == part) obs[(size_t)(15 + k) * ld + env] = qd[OM_H1_PERM[k]];
      }
      if (part == 0 && absorbing)
        absorbing[env] = (sp.use_absorbing && h1_has_fallen(q[OM_H1_PERM[2]], q[OM_H1_PERM[3]], q[OM_H1_PERM[4]], q[OM_H1_PERM[5]])) ? 1 : 0;
    } else {
      const int nq = sp.n_obs_q;
      for (int k = 2 + part; k < nq; k += 3) {
        if (obs) obs[(size_t)(k - 2) * ld + env] = qpos[(size_t)sp.perm[k] * ld + env];
      }
      for (int k = part; k < nq; k += 3) {
        if (obs) obs[(size_t)(nq - 2 + k) * ld + env] = qvel[(size_t)sp.perm[k] * ld + env];
      }
      if (part == 0 && absorbing) {
        const float y = qpos[(size_t)sp.perm[2] * ld + env], ti = qpos[(size_t)sp.perm[3] * ld + env];
        const float li = qpos[(size_t)sp.perm[4] * ld + env], ro = qpos[(size_t)sp.perm[5] * ld + env];
        absorbing[env] = (sp.use_absorbing && h1_has_fallen(y, ti, li, ro)) ? 1 : 0;
      }
    }
    if (part == 1 && reward) {
      const float d = prev_x_vel[env] - sp.target;
      reward[env] = expf(-(d * d));
    }
  }
  PredSoaSink S{{o.xpos, o.xquat, o.site_xpos, nullptr, o.cvel, o.com, (size_t)ld, (size_t)e}, live};
  SmemComExchange X{part_sum, part, lane};
  if (part == 0) om_fk_unitree_h1_part0(q, qd, S, X);
  else if (part == 1) om_fk_unitree_h1_part1(q, qd, S, X);
  else om_fk_unitree_h1_part2(q, qd, S, X);
}

__global__ void __launch_bounds__(128) h1_obs_kernel(H1SpecDev sp, const float* __restrict__ qpos,
                                                     const float* __restrict__ qvel, const float* __restrict__ prev_x_vel,
                                                     int n, int ld, float* __restrict__ obs, float* __restrict__ reward,
                                                     uint8_t* __restrict__ absorbing) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n) return;
  h1_obs_reward(sp, qpos, qvel, prev_x_vel, ld, env, obs, reward, absorbing);
}

__global__ void __launch_bounds__(256) h1_fallen_kernel(const float* __restrict__ obs, int n, int ld,
                                                        uint8_t* __restrict__ fallen) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n) return;
  fallen[env] = h1_has_fallen(obs[env], obs[(size_t)ld + env], obs[(size_t)2 * ld + env], obs[(size_t)3 * ld + env]) ? 1 : 0;
}

// set_sim_state (loco_env_base.py:659-684): sample rows in observation-spec order -> qpos / qvel rows in MJCF order
__global__ void __launch_bounds__(256) set_sim_state_kernel(H1SpecDev sp, const float* __restrict__ sample, int n, int ld,
                                                            float* __restrict__ qpos, float* __restrict__ qvel) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n) return;
  const int nq = sp.n_obs_q;
  for (int k = 0; k < nq; ++k) {
    qpos[(size_t)sp.perm[k] * ld + env] = sample[(size_t)k * ld + env];
    qvel[(size_t)sp.perm[k] * ld + env] = sample[(size_t)(nq + k) * ld + env];
  }
}

int make_spec(const OmH1Spec* spec, const OmModel* m, H1SpecDev* out) {
  OM_REQUIRE(spec->n_obs_q >= 6 && spec->n_obs_q <= 32, "OmH1Spec.n_obs_q %d outside [6,32]", spec->n_obs_q);
  OM_REQUIRE(spec->n_obs_q <= m->host.nq && spec->n_obs_q <= m->host.nv, "OmH1Spec.n_obs_q exceeds nq/nv");
  out->n_obs_q = spec->n_obs_q;
  out->x_vel_idx = spec->x_vel_idx;
  out->use_absorbing = spec->use_absorbing_states;
  out->target = spec->target_velocity;
  for (int k = 0; k < 32; ++k) {
    out->perm[k] = k < spec->n_obs_q ? spec->obs_perm[k] : 0;
    OM_REQUIRE(out->perm[k] >= 0 && out->perm[k] < m->host.nq, "OmH1Spec.obs_perm[%d] out of range", k);
  }
  return 0;
}

static FkEnvMass env_mass_arg(const OmModel* m) { return FkEnvMass{m->env_mass, m->env_mass_body, m->env_mass_m0}; }

}  // namespace om

using namespace om;

extern "C" int om_fk(const OmModel* m, const float* qpos, const float* qvel, int n, int ld, float* xpos, float* xquat,
                     float* site_xpos, float* site_xmat, float* cvel, float* subtree_com, int force_generic,
                     void* stream) {
  OM_REQUIRE(m, "om_fk: null model");
  OM_REQUIRE(n >= 0 && ld >= n, "om_fk: need 0 <= n <= ld (n=%d ld=%d)", n, ld);
  if (n == 0) return 0;            // empty batch: nothing to enqueue (pointers may be null)
  OM_REQUIRE(qpos, "om_fk: null qpos");
  cudaStream_t st = (cudaStream_t)stream;
  FkOut o{xpos, xquat, site_xpos, site_xmat, cvel, subtree_com};
  constexpr int BLOCK = 128;
  const int grid = ceil_div(n, BLOCK);
  if (!force_generic && m->specialised == SPEC_H1)
    fk_spec_kernel<SPEC_H1, BLOCK><<<grid, BLOCK, 0, st>>>(qpos, qvel, n, ld, o);
  else if (!force_generic && m->specialised == SPEC_A3)
    fk_spec_kernel<SPEC_A3, BLOCK><<<grid, BLOCK, 0, st>>>(qpos, qvel, n, ld, o);
  else if (m->env_mass) {
    OM_REQUIRE(n <= m->env_mass_ld, "om_fk: %d envs, but the bound body mass holds %d", n, m->env_mass_ld);
    fk_generic_kernel<true><<<grid, BLOCK, 0, st>>>(m->dev, qpos, qvel, n, ld, o, env_mass_arg(m));
  } else
    fk_generic_kernel<false><<<grid, BLOCK, 0, st>>>(m->dev, qpos, qvel, n, ld, o, FkEnvMass{});
  OM_LAUNCHED();
  return 0;
}

extern "C" int om_h1_step(const OmModel* m, const OmH1Spec* spec, const float* qpos, const float* qvel,
                          const float* prev_x_vel, int n, int ld, float* xpos, float* xquat, float* site_xpos,
                          float* cvel, float* obs, float* reward, uint8_t* absorbing, void* stream) {
  OM_REQUIRE(m && spec, "om_h1_step: null model or spec");
  OM_REQUIRE(n >= 0 && ld >= n, "om_h1_step: need 0 <= n <= ld (n=%d ld=%d)", n, ld);
  if (n == 0) return 0;
  OM_REQUIRE(qpos && qvel, "om_h1_step: null qpos/qvel");
  OM_REQUIRE(!reward || prev_x_vel, "om_h1_step: reward requested without prev_x_vel");
  H1SpecDev sp;
  if (make_spec(spec, m, &sp)) return 1;
  cudaStream_t st = (cudaStream_t)stream;
  FkOut o{xpos, xquat, site_xpos, nullptr, cvel, nullptr};
  const bool want_fk = xpos || xquat || site_xpos || cvel;
  constexpr int BLOCK = 128;
  const int grid = ceil_div(n, BLOCK);
  if (m->specialised == SPEC_H1) {
    // three threads per env for small batches (measured, CUDA-graph replays, both with the compile-time observation
    // permutation: 16384 envs 7.1 vs 7.3 us, 32768 envs 8.2 vs 9.0 us, 65536 envs 20.8 vs 15.4 us); OM_H1_SPLIT = 0 / 1
    // forces a path (tuning / tests; om_debug_set "h1_split")
    bool own_spec = sp.n_obs_q == 17;                 // UnitreeH1's own observation spec: compile-time permutation
    for (int k = 0; k < 17 && own_spec; ++k) own_spec = sp.perm[k] == OM_H1_PERM_HOST[k];
    bool split3 = want_fk && n <= 32768;
    if (g_knobs.h1_split >= 0) split3 = want_fk && g_knobs.h1_split != 0;
    if (split3 && own_spec) h1_step_split_kernel<true><<<ceil_div(n, 32), dim3(32, 3), 0, st>>>(sp, qpos, qvel, prev_x_vel, n, ld, o, obs, reward, absorbing);
    else if (split3) h1_step_split_kernel<false><<<ceil_div(n, 32), dim3(32, 3), 0, st>>>(sp, qpos, qvel, prev_x_vel, n, ld, o, obs, reward, absorbing);
    else if (want_fk && own_spec && n <= H1_STREAM_MAX_ENVS) h1_step_kernel<BLOCK, true, true, true><<<grid, BLOCK, 0, st>>>(sp, qpos, qvel, prev_x_vel, n, ld, o, obs, reward, absorbing);
    else if (want_fk && own_spec) h1_step_kernel<BLOCK, true, true, false><<<grid, BLOCK, 0, st>>>(sp, qpos, qvel, prev_x_vel, n, ld, o, obs, reward, absorbing);
    else if (want_fk && n <= H1_STREAM_MAX_ENVS) h1_step_kernel<BLOCK, true, false, true><<<grid, BLOCK, 0, st>>>(sp, qpos, qvel, prev_x_vel, n, ld, o, obs, reward, absorbing);
    else if (want_fk) h1_step_kernel<BLOCK, true, false, false><<<grid, BLOCK, 0, st>>>(sp, qpos, qvel, prev_x_vel, n, ld, o, obs, reward, absorbing);
    else if (own_spec) h1_step_kernel<BLOCK, false, true, false><<<grid, BLOCK, 0, st>>>(sp, qpos, qvel, prev_x_vel, n, ld, o, obs, reward, absorbing);
    else h1_step_kernel<BLOCK, false, false, false><<<grid, BLOCK, 0, st>>>(sp, qpos, qvel, prev_x_vel, n, ld, o, obs, reward, absorbing);
    OM_LAUNCHED();
  } else {
    if (want_fk && m->env_mass) {
      OM_REQUIRE(n <= m->env_mass_ld, "om_h1_step: %d envs, but the bound body mass holds %d", n, m->env_mass_ld);
      fk_generic_kernel<true><<<grid, BLOCK, 0, st>>>(m->dev, qpos, qvel, n, ld, o, env_mass_arg(m));
      OM_LAUNCHED();
    } else if (want_fk) {
      fk_generic_kernel<false><<<grid, BLOCK, 0, st>>>(m->dev, qpos, qvel, n, ld, o, FkEnvMass{});
      OM_LAUNCHED();
    }
    h1_obs_kernel<<<grid, BLOCK, 0, st>>>(sp, qpos, qvel, prev_x_vel, n, ld, obs, reward, absorbing);
    OM_LAUNCHED();
  }
  return 0;
}

extern "C" int om_h1_has_fallen(const float* obs, int n, int ld, uint8_t* fallen, void* stream) {
  OM_REQUIRE(n >= 0 && ld >= n, "om_h1_has_fallen: need 0 <= n <= ld");
  if (n == 0) return 0;
  OM_REQUIRE(obs && fallen, "om_h1_has_fallen: null argument");
  h1_fallen_kernel<<<ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(obs, n, ld, fallen);
  OM_LAUNCHED();
  return 0;
}

extern "C" int om_set_sim_state(const OmModel* m, const OmH1Spec* spec, const float* sample, int n, int ld, float* qpos,
                                float* qvel, void* stream) {
  OM_REQUIRE(m && spec, "om_set_sim_state: null model or spec");
  OM_REQUIRE(n >= 0 && ld >= n, "om_set_sim_state: need 0 <= n <= ld");
  if (n == 0) return 0;
  OM_REQUIRE(sample && qpos && qvel, "om_set_sim_state: null argument");
  H1SpecDev sp;
  if (make_spec(spec, m, &sp)) return 1;
  set_sim_state_kernel<<<ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(sp, sample, n, ld, qpos, qvel);
  OM_LAUNCHED();
  return 0;
}
