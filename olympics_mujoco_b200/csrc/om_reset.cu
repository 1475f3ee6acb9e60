// Per-env reset of a UnitreeH1 batch (om_h1_reset_envs): LocoEnvBase.reset for a subset of the envs, and the reset that
// mushroom_rl's Core performs on `last` after every step (auto-reset).  One thread per env, no FK: the reset state is the
// model's qpos0 with the drawn trajectory sample scattered over it, and the observation is that sample's keys 2..K-1.
//
// The kernel is a template over NQ (the observation spec's joints; the trajectory has K = 2 NQ keys) so that every sample
// and observation row is a register; it is instantiated for every NQ an OmH1Spec may hold (6..32), so it serves every model
// om_h1_step accepts -- the default model, its variants, the per-env carry model and models without generated kernels.
#include "om_common.cuh"
#include "om_traj.cuh"

namespace om {

constexpr int RESET_BLOCK = 128;
constexpr int RESET_MAX_MODELS = 16;

struct ResetDev {
  TrajDev t;
  uint64_t seed;
  uint32_t env_id0;
  int n, ld;
  const uint8_t* mask;
  const uint8_t* absorbing;
  int horizon, forced_traj, forced_step, x_vel_idx;
  int32_t* traj_no; int32_t* step_no; uint32_t* reset_count; double* xy_off;
  float* qpos; float* qvel;
  const float* obs_in; float* obs;
  float* prev_x_vel; int32_t* episode_step; uint8_t* last;
  float* grf; int n_grf;
  int32_t* partial_resets; int32_t* model_index; float* mass;
  int n_models, random;
  float masses[RESET_MAX_MODELS];
  int perm[32];                  // qpos / qvel row of observation-spec entry k
  // rows of qpos / qvel that no spec entry covers: qpos0 / 0 after mj_resetData (none for the shipped UnitreeH1 models)
  int n_xq, n_xv;
  uint8_t xq_row[MAXQ], xv_row[MAXQ];
  float xq_val[MAXQ];
};

template <int NQ>
__global__ void __launch_bounds__(RESET_BLOCK) h1_reset_envs_kernel(ResetDev a) {
  constexpr int K = 2 * NQ, KPAD = (K + 3) / 4 * 4, NOBS = K - 2;
  const int env = blockIdx.x * RESET_BLOCK + threadIdx.x;
  if (env >= a.n) return;
  const size_t ld = a.ld, e = env;
  bool go;
  if (a.mask) {
    go = a.mask[e] != 0;
  } else {                                        // Core._step: last = absorbing or episode_steps >= horizon
    const int es = a.episode_step[e] + 1;
    go = a.absorbing[e] != 0 || es >= a.horizon;
    a.last[e] = go ? 1 : 0;
    a.episode_step[e] = go ? 0 : es;
  }
  if (!go) {                                      // the observation of the step stays the env's observation
    if (a.obs && a.obs_in) {
      float v[NOBS];
#pragma unroll
      for (int k = 0; k < NOBS; ++k) v[k] = a.obs_in[k * ld + e];
      // (row x_vel_idx is re-read rather than selected out of v[]: a run-time pick out of a register array would put the
      //  array in local memory)
      const float pxv = a.obs_in[(size_t)a.x_vel_idx * ld + e];
#pragma unroll
      for (int k = 0; k < NOBS; ++k) a.obs[k * ld + e] = v[k];
      for (int c = 0; c < a.n_grf; ++c) a.obs[(NOBS + c) * ld + e] = a.obs_in[(NOBS + c) * ld + e];
      if (!a.mask) a.prev_x_vel[e] = pxv;
    }
    return;
  }
  // ---- the trajectory reset (om_traj_reset's contract) and its sample
  int tr, st;
  const uint32_t rc = a.reset_count[e];
  traj_draw(a.t, a.seed, a.env_id0 + env, rc, tr, st);
  if (a.forced_traj >= 0) tr = min(a.forced_traj, a.t.n_traj - 1);
  if (a.forced_step >= 0) st = min(a.forced_step, a.t.T - 1);
  float samp[KPAD];
  traj_reset_row(a.t, tr, st, samp);
  a.reset_count[e] = rc + 1;
  a.traj_no[e] = tr;
  a.step_no[e] = st;
  a.xy_off[e] = a.t.xy[((size_t)tr * a.t.T + st) * 2];
  a.xy_off[ld + e] = a.t.xy[((size_t)tr * a.t.T + st) * 2 + 1];
  // ---- mj_resetData, then set_sim_state of the sample
  for (int i = 0; i < a.n_xq; ++i) a.qpos[(size_t)a.xq_row[i] * ld + e] = a.xq_val[i];
  for (int i = 0; i < a.n_xv; ++i) a.qvel[(size_t)a.xv_row[i] * ld + e] = 0.f;
#pragma unroll
  for (int k = 0; k < NQ; ++k) {
    a.qpos[(size_t)a.perm[k] * ld + e] = samp[k];
    a.qvel[(size_t)a.perm[k] * ld + e] = samp[NQ + k];
  }
  // ---- observation (_create_observation of _build_obs: keys 2..K-1, then mean_grf / 1000 = 0)
  const float pxv = __ldg(a.t.rows + ((size_t)tr * a.t.T + st) * a.t.kpad + 2 + a.x_vel_idx);   // obs row x_vel_idx
  if (a.obs) {
#pragma unroll
    for (int k = 0; k < NOBS; ++k) a.obs[k * ld + e] = samp[k + 2];
    for (int c = 0; c < a.n_grf; ++c) a.obs[(NOBS + c) * ld + e] = 0.f;
  }
  if (a.grf) {
    for (int c = 0; c < a.n_grf; ++c) a.grf[c * ld + e] = 0.f;
  }
  if (a.prev_x_vel) a.prev_x_vel[e] = pxv;
  if (a.episode_step && a.mask) a.episode_step[e] = 0;
  // ---- the env's own model (per-env carried weight)
  if (a.model_index) {
    const uint32_t j = (uint32_t)a.partial_resets[e];
    const int k = a.random ? to_int(om_draw(a.seed, a.env_id0 + env, j, STREAM_PARTIAL_MODEL_RESET).x, a.n_models)
                           : (a.model_index[e] + 1) % a.n_models;
    a.partial_resets[e] = (int32_t)(j + 1);
    a.model_index[e] = k;
    a.mass[e] = a.masses[k];
  }
}

using ResetKernel = void (*)(ResetDev);
template <int... NQS>
struct ResetTable {
  static ResetKernel get(int nq) {
    ResetKernel k = nullptr;
    ((nq == NQS ? (k = &h1_reset_envs_kernel<NQS>, 0) : 0), ...);
    return k;
  }
};
// every n_obs_q an OmH1Spec may hold
using ResetKernels = ResetTable<6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27, 28, 29,
                                30, 31, 32>;

}  // namespace om

using namespace om;

extern "C" int om_h1_reset_envs(const OmModel* m, const OmH1Spec* spec, const OmTraj* t, uint64_t seed, uint32_t env_id0,
                                const OmH1ResetArgs* args, int n, int ld, void* stream) {
  OM_REQUIRE(m && spec && t && args, "om_h1_reset_envs: null argument");
  OM_REQUIRE(n >= 0 && ld >= n, "om_h1_reset_envs: need 0 <= n <= ld (n=%d ld=%d)", n, ld);
  const int nq = spec->n_obs_q;
  OM_REQUIRE(nq >= 6 && nq <= 32, "om_h1_reset_envs: OmH1Spec.n_obs_q %d outside [6,32]", nq);
  OM_REQUIRE(nq <= m->host.nq && nq <= m->host.nv, "om_h1_reset_envs: OmH1Spec.n_obs_q exceeds nq/nv of the model");
  const TrajDev& td = t->d;
  OM_REQUIRE(td.K == 2 * nq, "om_h1_reset_envs: expects a %d-key trajectory (2 n_obs_q), got %d", 2 * nq, td.K);
  const int nobs = 2 * nq - 2;
  OM_REQUIRE(spec->x_vel_idx >= 0 && spec->x_vel_idx < nobs, "om_h1_reset_envs: x_vel_idx %d outside [0,%d)",
             spec->x_vel_idx, nobs);
  const OmH1ResetArgs& r = *args;
  const int n_grf = r.grf ? r.n_grf : 0;
  OM_REQUIRE(n_grf >= 0 && n_grf <= 64, "om_h1_reset_envs: n_grf %d outside [0,64]", n_grf);
  OM_REQUIRE(!r.obs || r.obs_dim == nobs + n_grf, "om_h1_reset_envs: obs_dim %d, expected %d (2 n_obs_q - 2 + n_grf)",
             r.obs_dim, nobs + n_grf);
  const bool model_draw = r.model_index != nullptr;
  OM_REQUIRE(!model_draw || (r.partial_resets && r.mass && r.masses_host && r.n_models >= 1 &&
                             r.n_models <= RESET_MAX_MODELS),
             "om_h1_reset_envs: the model draw needs partial_resets, mass, masses_host and 1..%d models", RESET_MAX_MODELS);
  if (n == 0) return 0;
  OM_REQUIRE(r.traj_no && r.step_no && r.reset_count && r.xy_off && r.qpos && r.qvel, "om_h1_reset_envs: null state");
  if (!r.mask)
    OM_REQUIRE(r.absorbing && r.episode_step && r.last && r.obs_in && r.obs && r.prev_x_vel,
               "om_h1_reset_envs: auto-reset needs absorbing, episode_step, last, obs_in, obs and prev_x_vel");
  ResetKernel kern = ResetKernels::get(nq);
  OM_REQUIRE(kern, "om_h1_reset_envs: no kernel for n_obs_q %d", nq);
  ResetDev a = {};
  a.t = td; a.seed = seed; a.env_id0 = env_id0; a.n = n; a.ld = ld;
  a.mask = r.mask; a.absorbing = r.absorbing; a.horizon = r.horizon;
  a.forced_traj = r.forced_traj; a.forced_step = r.forced_step; a.x_vel_idx = spec->x_vel_idx;
  a.traj_no = r.traj_no; a.step_no = r.step_no; a.reset_count = r.reset_count; a.xy_off = r.xy_off;
  a.qpos = r.qpos; a.qvel = r.qvel; a.obs_in = r.obs_in; a.obs = r.obs;
  a.prev_x_vel = r.prev_x_vel; a.episode_step = r.episode_step; a.last = r.last;
  a.grf = r.grf; a.n_grf = n_grf;
  if (model_draw) {
    a.partial_resets = r.partial_resets; a.model_index = r.model_index; a.mass = r.mass;
    a.n_models = r.n_models; a.random = r.random ? 1 : 0;
    for (int k = 0; k < r.n_models; ++k) a.masses[k] = (float)r.masses_host[k];
  }
  bool qcov[MAXQ] = {}, vcov[MAXQ] = {};
  for (int k = 0; k < nq; ++k) {
    const int p = spec->obs_perm[k];
    OM_REQUIRE(p >= 0 && p < m->host.nq && p < m->host.nv, "om_h1_reset_envs: OmH1Spec.obs_perm[%d] = %d out of range", k, p);
    a.perm[k] = p;
    qcov[p] = vcov[p] = true;
  }
  for (int i = 0; i < m->host.nq; ++i)
    if (!qcov[i]) { a.xq_row[a.n_xq] = (uint8_t)i; a.xq_val[a.n_xq] = m->host.qpos0[i]; ++a.n_xq; }
  for (int i = 0; i < m->host.nv; ++i)
    if (!vcov[i]) a.xv_row[a.n_xv++] = (uint8_t)i;
  kern<<<ceil_div(n, RESET_BLOCK), RESET_BLOCK, 0, (cudaStream_t)stream>>>(a);
  OM_LAUNCHED();
  return 0;
}
