// Device math shared by every kernel: vectors, quaternions (MuJoCo mju_* conventions) and the Philox contract.
// Self-contained on purpose: tests/host/*.cpp compile the kernels' per-env device functions as plain host C++
// (OM_HD pre-defined as `inline`) to check them against the float64 oracle in a container without a GPU.
#pragma once
#include <stdint.h>
#include <math.h>

#ifndef OM_HD
#define OM_HD __device__ __forceinline__
#endif

namespace om {

struct V3 { float x, y, z; };
struct Q4 { float w, x, y, z; };

OM_HD V3 v3(float x, float y, float z) { return V3{x, y, z}; }
OM_HD V3 operator+(V3 a, V3 b) { return V3{a.x + b.x, a.y + b.y, a.z + b.z}; }
OM_HD V3 operator-(V3 a, V3 b) { return V3{a.x - b.x, a.y - b.y, a.z - b.z}; }
OM_HD V3 operator*(V3 a, float s) { return V3{a.x * s, a.y * s, a.z * s}; }
OM_HD V3 cross(V3 a, V3 b) { return V3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
OM_HD float dot(V3 a, V3 b) { return fmaf(a.x, b.x, fmaf(a.y, b.y, a.z * b.z)); }
OM_HD V3 fma3(V3 a, float s, V3 c) { return V3{fmaf(a.x, s, c.x), fmaf(a.y, s, c.y), fmaf(a.z, s, c.z)}; }

// mju_mulQuat
OM_HD Q4 qmul(Q4 a, Q4 b) {
  return Q4{a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z, a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y,
            a.w * b.y - a.x * b.z + a.y * b.w + a.z * b.x, a.w * b.z + a.x * b.y - a.y * b.x + a.z * b.w};
}
// mju_rotVecQuat
OM_HD V3 qrot(Q4 q, V3 v) {
  V3 u{q.x, q.y, q.z};
  V3 t = v * q.w + cross(u, v);
  V3 c = cross(u, t);
  return V3{fmaf(2.0f, c.x, v.x), fmaf(2.0f, c.y, v.y), fmaf(2.0f, c.z, v.z)};
}
// mju_normalize4
OM_HD Q4 qnormalize(Q4 q) {
  float n2 = fmaf(q.w, q.w, fmaf(q.x, q.x, fmaf(q.y, q.y, q.z * q.z)));
  if (n2 < 1e-30f) return Q4{1.f, 0.f, 0.f, 0.f};
  float inv = rsqrtf(n2);
  return Q4{q.w * inv, q.x * inv, q.y * inv, q.z * inv};
}
// mju_quat2Mat (row major)
OM_HD void quat2mat(Q4 q, float* m) {
  float ww = q.w * q.w, xx = q.x * q.x, yy = q.y * q.y, zz = q.z * q.z;
  float xy = q.x * q.y, xz = q.x * q.z, yz = q.y * q.z, wx = q.w * q.x, wy = q.w * q.y, wz = q.w * q.z;
  m[0] = ww + xx - yy - zz; m[1] = 2.f * (xy - wz);   m[2] = 2.f * (xz + wy);
  m[3] = 2.f * (xy + wz);   m[4] = ww - xx + yy - zz; m[5] = 2.f * (yz - wx);
  m[6] = 2.f * (xz - wy);   m[7] = 2.f * (yz + wx);   m[8] = ww - xx - yy + zz;
}

// ---------------------------------------------------------------- bounded-range trigonometry
// The FK evaluates one sin/cos pair per hinge and the task a handful more; libm's sincosf / tanf inline a
// Payne-Hanek slow path at every call site (dead code for joint angles, but it triples the code size of the
// straight-line kernels and their instruction-cache misses).  These keep libm's fast path -- three-term Cody-Waite
// reduction by pi/2 and degree-7/8 minimax polynomials on [-pi/4, pi/4], error <= 2 ulp -- and send anything outside
// its validity range (|x| > 105615, inf, nan) to ONE out-of-line libm call.
#ifdef __CUDACC__
#define OM_NOINLINE static __device__ __noinline__
OM_HD int om_float_bits(float x) { return __float_as_int(x); }
OM_HD float om_bits_float(int i) { return __int_as_float(i); }
#else
#define OM_NOINLINE static inline
#include <string.h>
OM_HD int om_float_bits(float x) { int i; memcpy(&i, &x, 4); return i; }
OM_HD float om_bits_float(int i) { float x; memcpy(&x, &i, 4); return x; }
#endif
struct SinCos { float s, c; };
OM_NOINLINE SinCos om_sincos_libm(float x) { SinCos r; sincosf(x, &r.s, &r.c); return r; }   // by value: no stack traffic
OM_NOINLINE float om_tan_libm(float x) { return tanf(x); }
// 1 / x without the IEEE-division fix-up sequence (MUFU.RCP + one Newton step, <= 1 ulp): a full-precision a / b costs ~20
// instructions with its slow-path check, and four of them were 14 % of the A3 feature kernel
OM_HD float om_rcp(float x) {
#ifdef __CUDA_ARCH__
  return __frcp_rn(x);
#else
  return 1.0f / x;
#endif
}

template <bool GUARD>
OM_HD void om_sincos_t(float x, float* sn, float* cs) {
  if (GUARD && !(fabsf(x) <= 105615.0f)) { const SinCos r = om_sincos_libm(x); *sn = r.s; *cs = r.c; return; }
  const float j = fmaf(x, 0.636619747f, 12582912.0f);           // 1.5 * 2^23: the low mantissa bits hold rint(x * 2/pi)
  const int q = om_float_bits(j);
  const float k = j - 12582912.0f;
  float r = fmaf(k, -1.57079601e+00f, x);
  r = fmaf(k, -3.13916473e-07f, r);
  r = fmaf(k, -5.39030253e-15f, r);
  const float r2 = r * r;
  float ps = fmaf(r2, -1.95152959e-04f, 8.33216087e-03f);
  ps = fmaf(ps, r2, -1.66666546e-01f);
  ps = fmaf(ps * r2, r, r);                                     // sin(r)
  float pc = fmaf(r2, 2.44331571e-05f, -1.38873163e-03f);
  pc = fmaf(pc, r2, 4.16666456e-02f);
  pc = fmaf(pc, r2, -0.5f);
  pc = fmaf(pc, r2, 1.0f);                                      // cos(r)
  const float a = (q & 1) ? pc : ps, b = (q & 1) ? ps : pc;     // quadrant: swap, then signs
  *sn = (q & 2) ? -a : a;
  *cs = ((q + 1) & 2) ? -b : b;
}

OM_HD void om_sincos(float x, float* sn, float* cs) { om_sincos_t<true>(x, sn, cs); }
// Hinge angles only: no range guard.  Beyond 1e5 rad an fp32 angle is quantised to 0.008 rad and the kinematics is
// meaningless anyway; nan stays nan.
OM_HD void om_sincos_hinge(float x, float* sn, float* cs) { om_sincos_t<false>(x, sn, cs); }

// tan on [-pi/4 - eps, pi/4 + eps] (the argument of the foot clock terms, rewards.py:65-102); libm outside
OM_HD float om_tan_q(float x) {
  if (!(fabsf(x) <= 0.7854f)) return om_tan_libm(x);
  const float z = x * x;                                        // odd minimax polynomial, degree 13 (Cephes tanf)
  float p = fmaf(z, 9.38540185543e-3f, 3.11992232697e-3f);
  p = fmaf(p, z, 2.44301354525e-2f);
  p = fmaf(p, z, 5.34112807005e-2f);
  p = fmaf(p, z, 1.33387994085e-1f);
  p = fmaf(p, z, 3.33331568548e-1f);
  return fmaf(p * z, x, x);
}

// atan2 for the goal-step headings: reciprocal instead of libm's IEEE division, degree-8 minimax polynomial of atan(t)/t
// in t^2 on [0, 1] (|error| < 1e-7 in fp32); zeros, denormals, infinities and nan take the out-of-line libm call
OM_NOINLINE float om_atan2_libm(float y, float x) { return atan2f(y, x); }
OM_HD float om_atan2(float y, float x) {
  const float ax = fabsf(x), ay = fabsf(y);
  const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
  if (!(mx > 1e-30f && mx < 1e30f)) return om_atan2_libm(y, x);
  const float t = mn * om_rcp(mx), z = t * t;
  float p = fmaf(z, 2.4567244e-03f, -1.4401359e-02f);
  p = fmaf(p, z, 3.9781228e-02f);
  p = fmaf(p, z, -7.2348580e-02f);
  p = fmaf(p, z, 1.0498947e-01f);
  p = fmaf(p, z, -1.4161229e-01f);
  p = fmaf(p, z, 1.9985907e-01f);
  p = fmaf(p, z, -3.3332598e-01f);
  p = fmaf(p, z, 9.9999988e-01f);
  float r = p * t;
  if (ay > ax) r = 1.57079632679489662f - r;
  if (x < 0.f) r = 3.14159265358979324f - r;
  return copysignf(r, y);
}

// ---------------------------------------------------------------- Philox4x32-10 (contract: oracle/philox.py)
struct U4 { uint32_t x, y, z, w; };
OM_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
OM_HD U4 philox4x32_10(U4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = mulhi32(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    uint32_t hi1 = mulhi32(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = U4{hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0};
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}
OM_HD U4 om_draw(uint64_t seed, uint32_t env, uint32_t count, uint32_t stream) {
  return philox4x32_10(U4{env, count, stream, 0u}, (uint32_t)seed, (uint32_t)(seed >> 32));
}
OM_HD int to_int(uint32_t x, int n) { return (int)mulhi32(x, (uint32_t)n); }
// Streams (third counter word) in use: 0 trajectory resets, 16..30 the A3 reset, 32 the MultiMuJoCo model switch of a whole
// reset() (om_h1_draw_models), 33 the model an env draws at its own partial reset (om_h1_reset_envs), 48 expert minibatches.
constexpr uint32_t STREAM_PARTIAL_MODEL_RESET = 33u;   // utils/philox.py
OM_HD float to_unit(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }

}  // namespace om
