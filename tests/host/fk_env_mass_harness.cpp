// TEST INFRASTRUCTURE: compiles the GENERATED carry-model FK whose weight mass is a runtime argument
// (codegen.generate_fk(..., env_mass_body=...)) as plain host C++, so that it can be checked against the float64 oracle in
// a container without a GPU.  Never shipped, never used by the product (which has no CPU path).
#include <cmath>
#include <cstring>
#define OM_HD inline
static inline float rsqrtf(float x) { return 1.0f / std::sqrt(x); }
#include "om_math.cuh"
#include "fk_h1_carry_env.cuh"

struct HostSink {
  static constexpr bool want_site_xmat = false;
  float *xp, *xq, *sp, *cv, *cm;
  void xpos(int b, float x, float y, float z) { xp[b*3]=x; xp[b*3+1]=y; xp[b*3+2]=z; }
  void xquat(int b, float w, float x, float y, float z) { xq[b*4]=w; xq[b*4+1]=x; xq[b*4+2]=y; xq[b*4+3]=z; }
  void site_xpos(int s, float x, float y, float z) { sp[s*3]=x; sp[s*3+1]=y; sp[s*3+2]=z; }
  void site_xmat(int, float, float, float, float, float, float, float, float, float) {}
  void cvel(int b, float wx, float wy, float wz, float vx, float vy, float vz) {
    float v[6] = {wx,wy,wz,vx,vy,vz}; std::memcpy(cv + 6*b, v, sizeof v); }
  void com(float x, float y, float z) { cm[0]=x; cm[1]=y; cm[2]=z; }
  void vel_p(int, float, float, float, float, float, float) {}
};

// env e: state (q[17 e..], qd[17 e..]) with weight-body mass mass[e]
extern "C" void host_fk_h1_carry_env(const float* q, const float* qd, const float* mass, int n, float* xp, float* xq,
                                     float* sp, float* cv, float* cm) {
  for (int e = 0; e < n; ++e) {
    float qq[17], dd[17];
    std::memcpy(qq, q + 17*e, sizeof qq); std::memcpy(dd, qd + 17*e, sizeof dd);
    HostSink S{xp + 66*e, xq + 88*e, sp + 3*e, cv + 132*e, cm + 3*e};
    om_fk_h1_carry_env(qq, dd, S, mass[e]);
  }
}
