// Model handle: uploads the mjModel-like tables and decides which kernel family serves them.
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "om_common.cuh"
#include "gen/tables_unitree_h1.h"
#include "gen/tables_stick_figure_a3.h"
#include "gen/h1v/list.h"
#include "gen/h1v/tables.h"

namespace om {

std::string& last_error() {
  static thread_local std::string e;
  return e;
}
int fail(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  last_error() = buf;
  return 1;
}
std::atomic<long long> g_launches{0};

static int env_int(const char* name, int dflt) {
  const char* f = getenv(name);
  return f ? atoi(f) : dflt;
}
Knobs g_knobs = [] {
  Knobs k;
  k.play_chunk = env_int("OM_PLAY_CHUNK", 0);
  k.h1_split = env_int("OM_H1_SPLIT", -1);
  k.a3_split = env_int("OM_A3_SPLIT", -1);
  k.serial_scan = env_int("OM_SERIAL_SCAN", 0);
  k.disc_vail2 = env_int("OM_DISC_VAIL2", -1);
  k.disc_pg2 = env_int("OM_DISC_PG2", -1);
  k.a3_feat_minb = env_int("OM_A3_FEAT_MINB", 0);
  return k;
}();

template <class T>
static bool same_i(const int* a, const T* b, int n) {
  for (int i = 0; i < n; ++i)
    if (a[i] != (int)b[i]) return false;
  return true;
}
static bool same_f(const float* a, const float* b, int n) {
  for (int i = 0; i < n; ++i)
    if (a[i] != b[i]) return false;
  return true;
}

#define OM_MATCH(prefix, t)                                                                              \
  (t.nbody == prefix##_nbody && t.njnt == prefix##_njnt && t.nsite == prefix##_nsite &&                  \
   t.nq == prefix##_nq && t.nv == prefix##_nv && same_i(t.body_parent, prefix##_body_parentid, t.nbody) && \
   same_i(t.body_jntadr, prefix##_body_jntadr, t.nbody) && same_i(t.body_jntnum, prefix##_body_jntnum, t.nbody) && \
   same_i(t.jnt_type, prefix##_jnt_type, t.njnt) && same_i(t.jnt_qposadr, prefix##_jnt_qposadr, t.njnt) && \
   same_i(t.site_body, prefix##_site_bodyid, t.nsite) && same_f(t.body_pos, prefix##_body_pos, 3 * t.nbody) && \
   same_f(t.body_quat, prefix##_body_quat, 4 * t.nbody) && same_f(t.body_ipos, prefix##_body_ipos, 3 * t.nbody) && \
   same_f(t.body_mass, prefix##_body_mass, t.nbody) && same_f(t.jnt_axis, prefix##_jnt_axis, 3 * t.njnt) && \
   same_f(t.jnt_pos, prefix##_jnt_pos, 3 * t.njnt) && same_f(t.qpos0, prefix##_qpos0, t.nq) &&          \
   same_f(t.site_pos, prefix##_site_pos, 3 * t.nsite) && same_f(t.site_quat, prefix##_site_quat, 4 * t.nsite))

}  // namespace om

using namespace om;

extern "C" const char* om_last_error(void) { return om::last_error().c_str(); }
extern "C" int om_abi_version(void) { return OM_ABI_VERSION; }
extern "C" long long om_launch_count(void) { return om::g_launches.load(); }
extern "C" void om_reset_launch_count(void) { om::g_launches.store(0); }

extern "C" int om_debug_set(const char* knob, int value) {
  OM_REQUIRE(knob, "om_debug_set: null knob");
  const std::string k(knob);
  if (k == "play_chunk") g_knobs.play_chunk = value > 0 ? value : 0;
  else if (k == "h1_split") g_knobs.h1_split = value;
  else if (k == "a3_split") g_knobs.a3_split = value;
  else if (k == "serial_scan") g_knobs.serial_scan = value;
  else if (k == "disc_vail2") g_knobs.disc_vail2 = value;
  else if (k == "disc_pg2") g_knobs.disc_pg2 = value;
  else if (k == "a3_feat_minb") g_knobs.a3_feat_minb = value;
  else return fail("om_debug_set: unknown knob '%s'", knob);
  return 0;
}

extern "C" int om_model_create(const OmModelDesc* d, OmModel** out) {
  OM_REQUIRE(d && out, "om_model_create: null argument");
  OM_REQUIRE(d->nbody >= 2 && d->nbody <= MAXB, "om_model_create: nbody %d outside [2,%d]", d->nbody, MAXB);
  OM_REQUIRE(d->njnt >= 0 && d->njnt <= MAXJ, "om_model_create: njnt %d > %d", d->njnt, MAXJ);
  OM_REQUIRE(d->nsite >= 0 && d->nsite <= MAXS, "om_model_create: nsite %d > %d", d->nsite, MAXS);
  OM_REQUIRE(d->nq <= MAXQ && d->nv <= MAXQ, "om_model_create: nq/nv > %d", MAXQ);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail("om_model_create: no CUDA device (this library has no CPU path)");
  OmModel* m = new OmModel();
  ModelTab& t = m->host;
  std::memset(&t, 0, sizeof t);
  t.nbody = d->nbody; t.njnt = d->njnt; t.nsite = d->nsite; t.nq = d->nq; t.nv = d->nv;
  for (int i = 0; i < d->nbody; ++i) {
    t.body_parent[i] = d->body_parentid[i];
    t.body_root[i] = d->body_rootid[i];
    t.body_jntadr[i] = d->body_jntadr[i];
    t.body_jntnum[i] = d->body_jntnum[i];
    t.body_mass[i] = (float)d->body_mass[i];
    for (int k = 0; k < 3; ++k) t.body_pos[3 * i + k] = (float)d->body_pos[3 * i + k];
    for (int k = 0; k < 4; ++k) t.body_quat[4 * i + k] = (float)d->body_quat[4 * i + k];
    for (int k = 0; k < 3; ++k) t.body_ipos[3 * i + k] = (float)d->body_ipos[3 * i + k];
    if (i > 0 && (t.body_parent[i] < 0 || t.body_parent[i] >= i)) {
      delete m;
      return fail("om_model_create: body %d has parent %d (bodies must be in depth-first order)", i, t.body_parent[i]);
    }
    if (t.body_jntnum[i] > 8) {
      delete m;
      return fail("om_model_create: body %d has %d joints (max 8)", i, t.body_jntnum[i]);
    }
  }
  double tree_mass[MAXB] = {0};
  for (int i = 1; i < d->nbody; ++i) tree_mass[t.body_root[i]] += d->body_mass[i];
  for (int i = 0; i < d->nbody; ++i) t.tree_inv_mass[i] = tree_mass[i] > 1e-15 ? (float)(1.0 / tree_mass[i]) : 0.f;
  for (int j = 0; j < d->njnt; ++j) {
    t.jnt_type[j] = d->jnt_type[j];
    t.jnt_qposadr[j] = d->jnt_qposadr[j];
    t.jnt_dofadr[j] = d->jnt_dofadr[j];
    for (int k = 0; k < 3; ++k) t.jnt_axis[3 * j + k] = (float)d->jnt_axis[3 * j + k];
    for (int k = 0; k < 3; ++k) t.jnt_pos[3 * j + k] = (float)d->jnt_pos[3 * j + k];
  }
  for (int k = 0; k < d->nq; ++k) t.qpos0[k] = (float)d->qpos0[k];
  for (int s = 0; s < d->nsite; ++s) {
    t.site_body[s] = d->site_bodyid[s];
    for (int k = 0; k < 3; ++k) t.site_pos[3 * s + k] = (float)d->site_pos[3 * s + k];
    for (int k = 0; k < 4; ++k) t.site_quat[4 * s + k] = (float)d->site_quat[4 * s + k];
  }
  if (OM_MATCH(om_tab_h1, t)) m->specialised = SPEC_H1;
  else if (OM_MATCH(om_tab_a3, t)) m->specialised = SPEC_A3;
  // the UnitreeH1 variants with fused playback / live-step kernels; only the default model is `specialised` (om_fk and
  // om_h1_step keep the table-driven FK for the others)
  if (m->specialised == SPEC_H1) m->h1_variant = 1;
#define OM_H1_VARIANT_MATCH(id, name) else if (OM_MATCH(om_tab_h1v_##name, t)) m->h1_variant = id;
  OM_H1_VARIANTS(OM_H1_VARIANT_MATCH)
#undef OM_H1_VARIANT_MATCH
  cudaGetDevice(&m->device);
  cudaError_t e = cudaMalloc(&m->dev, sizeof(ModelTab));
  if (e == cudaSuccess) e = cudaMemcpy(m->dev, &t, sizeof(ModelTab), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    delete m;
    return fail("om_model_create: device upload failed: %s", cudaGetErrorString(e));
  }
  *out = m;
  return 0;
}

extern "C" void om_model_destroy(OmModel* m) {
  if (!m) return;
  if (m->dev) cudaFree(m->dev);
  delete m;
}

extern "C" int om_model_bind_env_body_mass(OmModel* m, int body, const float* mass, int ld) {
  OM_REQUIRE(m && mass, "om_model_bind_env_body_mass: null argument");
  OM_REQUIRE(OM_H1_IS_CARRY(m->h1_variant),
             "om_model_bind_env_body_mass: only the UnitreeH1 carry models take a per-env body mass (h1 variant %d)",
             m->h1_variant);
  OM_REQUIRE(body == OM_H1_CARRY_WEIGHT_BODY, "om_model_bind_env_body_mass: body %d is not the weight body (%d)", body,
             OM_H1_CARRY_WEIGHT_BODY);
  OM_REQUIRE(ld >= 1, "om_model_bind_env_body_mass: ld %d < 1", ld);
  OM_REQUIRE(!m->env_mass || (m->env_mass == mass && m->env_mass_ld == ld),
             "om_model_bind_env_body_mass: the model is already bound to another buffer (a binding is for life)");
  const ModelTab& t = m->host;
  double m0 = 0.0;
  for (int i = 1; i < t.nbody; ++i)
    if (i != body && t.body_root[i] == t.body_root[body]) m0 += t.body_mass[i];
  m->env_mass = mass;
  m->env_mass_body = body;
  m->env_mass_ld = ld;
  m->env_mass_m0 = (float)m0;
  return 0;
}

extern "C" int om_model_is_specialised(const OmModel* m) { return m ? m->specialised : 0; }
extern "C" int om_model_h1_variant(const OmModel* m) { return m ? m->h1_variant : 0; }
