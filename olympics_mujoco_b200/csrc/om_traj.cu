// K3: reference-trajectory table + per-env integer state, and the fused H1 playback kernel.
//
// The fused playback / live-step kernels are templates over a UnitreeH1 variant descriptor V (H1Default below; the other
// variants' descriptors are generated into gen/h1v/):
//   V::NQ      joints in the observation spec (= nq = nv of the model); the trajectory has K = 2 NQ keys
//   V::NBODY, V::NSITE
//   V::perm(k) qpos / qvel address of observation-spec entry k
//   V::fk(q, qd, sink)  the generated FK of the model
//   V::ENV_MASS  fk takes one more argument, the env's mass of the carried weight (a carry model bound to a per-env mass
//                with om_model_bind_env_body_mass: the kernels load it once per thread from PlayArgsEnv / LiveArgs::env_mass)
// build.py compiles this file once more per variant with -DOM_H1_VARIANT=<name>: such a compilation only instantiates the
// fused kernels of that variant (H1Kernels h1k_<name>), in parallel with the rest of the build.
#include <cstdlib>
#include <type_traits>
#include <vector>

#include "om_common.cuh"
#include "om_sinks.cuh"
#include "om_traj.cuh"
#ifdef OM_H1_VARIANT
#include OM_H1_VARIANT_HEADER
#else
#include "gen/fk_unitree_h1.cuh"
#include "gen/h1_perm.h"
#include "gen/h1v/list.h"
#endif

namespace om {

#ifndef OM_H1_VARIANT
// ---------------------------------------------------------------- per-step API kernels
__global__ void __launch_bounds__(128) traj_reset_kernel(TrajDev t, uint64_t seed, uint32_t env_id0,
                                                         const uint8_t* __restrict__ mask,
                                                         const int32_t* __restrict__ forced_traj,
                                                         const int32_t* __restrict__ forced_step,
                                                         int32_t* traj_no, int32_t* step_no, uint32_t* reset_count,
                                                         double* xy_off, float* sample, int n, int ld) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n) return;
  if (mask && !mask[env]) return;
  int tr, st;
  uint32_t rc = reset_count[env];
  traj_draw(t, seed, env_id0 + env, rc, tr, st);
  if (forced_traj && forced_traj[env] >= 0) tr = min(forced_traj[env], t.n_traj - 1);
  if (forced_step && forced_step[env] >= 0) st = min(forced_step[env], t.T - 1);
  reset_count[env] = rc + 1;
  traj_no[env] = tr;
  step_no[env] = st;
  const double ox = t.xy[((size_t)tr * t.T + st) * 2], oy = t.xy[((size_t)tr * t.T + st) * 2 + 1];
  xy_off[env] = ox;
  xy_off[(size_t)ld + env] = oy;
  if (sample) traj_write_sample(t, tr, st, ox, oy, sample, ld, env);
}

__global__ void __launch_bounds__(128) traj_current_kernel(TrajDev t, const int32_t* __restrict__ traj_no,
                                                           const int32_t* __restrict__ step_no,
                                                           const double* __restrict__ xy_off, float* sample, int n,
                                                           int ld) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n) return;
  traj_write_sample(t, traj_no[env], step_no[env], xy_off[env], xy_off[(size_t)ld + env], sample, ld, env);
}

__global__ void __launch_bounds__(128) traj_next_kernel(TrajDev t, uint64_t seed, uint32_t env_id0, int auto_reset,
                                                        int32_t* traj_no, int32_t* step_no, uint32_t* reset_count,
                                                        double* xy_off, float* sample, uint8_t* wrapped, int n, int ld) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n) return;
  int tr = traj_no[env], st = step_no[env] + 1;
  double ox = xy_off[env], oy = xy_off[(size_t)ld + env];
  const bool wrap = st >= t.T;
  if (wrap && !auto_reset) {            // get_next_sample returns None: the index parks at T, sample untouched
    step_no[env] = t.T;
    if (wrapped) wrapped[env] = 1;
    return;
  }
  if (wrap) {
    uint32_t rc = reset_count[env];
    traj_draw(t, seed, env_id0 + env, rc, tr, st);
    reset_count[env] = rc + 1;
    ox = t.xy[((size_t)tr * t.T + st) * 2];
    oy = t.xy[((size_t)tr * t.T + st) * 2 + 1];
    xy_off[env] = ox;
    xy_off[(size_t)ld + env] = oy;
    traj_no[env] = tr;
  }
  step_no[env] = st;
  if (wrapped) wrapped[env] = wrap ? 1 : 0;
  if (sample) traj_write_sample(t, tr, st, ox, oy, sample, ld, env);
}

#endif  // !OM_H1_VARIANT

template <class V>
struct H1Dims {
  static constexpr int NQ = V::NQ, K = 2 * NQ, KPAD = (K + 3) / 4 * 4;
  static constexpr int NOBS = K - 2;          // observation = trajectory keys without root x, y
  static constexpr int PW = 2 * NOBS;         // statistic rows of the observation moments: sum[NOBS], sumsq[NOBS]
};

// ---------------------------------------------------------------- fused playback (sequential in time)
// One thread per env walks its episode step by step (loco_env_base.py:511-552).  Used when the episode is
// short or the caller asks for it; the time-parallel kernel below is the throughput path.
struct PlayArgs {
  TrajDev t;
  uint64_t seed;
  uint32_t env_id0;
  double dt;
  float target;
  int n_steps, end_reset, n, ld;      // (no use_absorbing: the playback loops call _has_fallen whatever the MDP setting,
                                      //  loco_env_base.py:422,541)
  int forced;         // 1 = play_trajectory (the model is forced to each sample), 0 = play_trajectory_from_velocity
  OmPlayState s;      // live carried state (written by the thread that runs the last step)
  OmPlayState snap;   // episode-start snapshot read by every chunk of the time-parallel kernel
  OmPlayOut o;
  double* obs_moments;   // = o.obs_moments (S1 fused into the playback), or null
};
// The playback arguments of a variant whose FK takes the env's weight mass.  A type of its own, so that the kernel parameters
// of every other variant (and with them their code) stay exactly what they were.
struct PlayArgsEnv : PlayArgs {
  const float* env_mass;   // [ld] mass of the carried weight per env
};
template <class V>
using PlayArgsOf = std::conditional_t<V::ENV_MASS, PlayArgsEnv, PlayArgs>;

// observation columns 0-3 (pelvis ty, tilt, list, rotation) are the same root joints in every variant
OM_HD bool h1_fallen_f(float y, float tilt, float lst, float rot) {
  const double PI = 3.141592653589793;
  const double dy = y, dt = tilt, dl = lst, dr = rot;
  return (dy < -0.3) || (dy > 0.1) || (dt < (-PI / 4.5)) || (dt > (PI / 12)) || (dl < -PI / 12) || (dl > PI / 8) ||
         (dr < (-PI / 8)) || (dr > (PI / 8));
}

// the variant's FK, with the env's body mass when the variant takes one
template <class V, class Sink>
OM_HD void v_fk(const float (&q)[V::NQ], const float (&qd)[V::NQ], Sink& S, float mass) {
  if constexpr (V::ENV_MASS) V::fk(q, qd, S, mass);
  else V::fk(q, qd, S);
}

// the env's mass of the carried weight, loaded once per thread (0 and no load for a variant without one)
template <class V, class A>
OM_HD float v_env_mass(const A& a, size_t env) {
  if constexpr (V::ENV_MASS) return a.env_mass[env];
  else return 0.f;
}

// One playback step given the sim state; shared by both playback kernels.
//   qs[NQ] (spec order, double) , dq[NQ] (spec order) -> FK outputs at time slot `slot`
// STREAM: streaming stores -- the time-parallel kernel (few envs, many steps: +2.5 % there); with 10^6 envs in the
// one-thread-per-env kernel they measured 1.5 % slower.
template <class V, bool STREAM>
OM_HD void play_fk(const double (&qs)[V::NQ], const float (&dq)[V::NQ], const OmPlayOut& o, size_t slot, size_t ld,
                   size_t env, float mass) {
  float q[V::NQ], qd[V::NQ];
#pragma unroll
  for (int k = 0; k < V::NQ; ++k) {
    q[V::perm(k)] = (float)qs[k];
    qd[V::perm(k)] = dq[k];
  }
  SoaSink<false, STREAM> S{o.xpos ? o.xpos + slot * (V::NBODY * 3) * ld : nullptr,
                           o.xquat ? o.xquat + slot * (V::NBODY * 4) * ld : nullptr,
                           o.site_xpos ? o.site_xpos + slot * (V::NSITE * 3) * ld : nullptr, nullptr,
                           o.cvel ? o.cvel + slot * (V::NBODY * 6) * ld : nullptr, nullptr, ld, env};
  v_fk<V>(q, qd, S, mass);
}

// obs / fallen / reward / integer state of one step from the freshly gathered sample row
constexpr int PLAY_BLOCK = 128;
template <class V, bool STREAM>
OM_HD void play_emit(const float (&samp)[H1Dims<V>::KPAD], float prev_x_vel, const PlayArgs& a, size_t slot, size_t env,
                     int tr, int st) {
  constexpr int NOBS = H1Dims<V>::NOBS;
  const size_t ld = a.ld;
  if (a.o.obs) {
    float* ob = a.o.obs + slot * NOBS * ld + env;
#pragma unroll
    for (int k = 0; k < NOBS; ++k) {
#ifdef __CUDA_ARCH__
      if (STREAM) __stcs(ob + k * ld, samp[k + 2]);   // written once, not read back by this call (the moments come from the prefix sums)
      else ob[k * ld] = samp[k + 2];
#else
      ob[k * ld] = samp[k + 2];
#endif
    }
  }
  if (a.o.fallen) a.o.fallen[slot * ld + env] = h1_fallen_f(samp[2], samp[3], samp[4], samp[5]) ? 1 : 0;
  if (a.o.reward) {
    const float d = prev_x_vel - a.target;
    a.o.reward[slot * ld + env] = expf(-(d * d));
  }
  if (a.o.traj_no_t) a.o.traj_no_t[slot * ld + env] = tr;
  if (a.o.step_no_t) a.o.step_no_t[slot * ld + env] = st;
}

// S1 of the playback WITHOUT touching the observation buffer: every observation a playback call emits is a row of the
// (L2-resident) trajectory table, and an env walks the table in contiguous runs -- rows st0+1 .. T-1 of its trajectory, then
// after each wrap reset rows st' .. of the drawn one.  With float64 prefix sums of the rows and of their squares
// (TrajDev::psum, 1 MB for 4 x 500 samples of the default model) the moment sums of a whole call are a few prefix differences
// per env and channel: one small kernel instead of a second pass over the [T][NOBS][n] observation buffer (262 MB re-read per
// 4096 x 500 rollout of the default model; an in-kernel accumulation through shared memory cost the playback kernel 75 us of
// LSU bandwidth).  Layout of the result: om_moments' [sum[NOBS], sumsq[NOBS], count] (Standardizer networks.py:76-81,
// RunningMeanStd normalize.py:190-208).
constexpr int PM_ENVS = 4;     // envs per warp
template <class V>
__global__ void __launch_bounds__(256) play_moments_kernel(PlayArgs a, OmPlayState start, int start_reset) {
  // a warp takes PM_ENVS envs one after the other with its LANES ON THE PW STATISTIC ROWS (lane l: rows l, l + 32, ...), so
  // that every prefix-table access is one coalesced read and no cross-lane reduction is needed; the 8 warps of the CTA meet
  // in shared memory: PW atomics per 32 envs.  (One thread per env with 64 accumulators each made every load a 32-way
  // scattered access: 34 us for 4096 envs; per-warp atomics queued 2048 same-line float64 updates: 12 us.)
  constexpr int PW = H1Dims<V>::PW, R = (PW + 31) / 32;
  __shared__ double part[8][PW];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int env0 = (blockIdx.x * 8 + w) * PM_ENVS;
  const int T = a.t.T;
  int tr_[PM_ENVS], st_[PM_ENVS];
  uint32_t rc_[PM_ENVS];
#pragma unroll
  for (int u = 0; u < PM_ENVS; ++u) {                  // the state loads of all envs first (independent round trips)
    const int env = env0 + u;
    const bool live = env < a.n;
    tr_[u] = live ? start.traj_no[env] : 0;
    st_[u] = live ? start.step_no[env] : 0;
    rc_[u] = live ? start.reset_count[env] : 0u;
  }
  // row 32 r + lane exists for every lane of a full group of 32 rows; the last group may be partial (e.g. 60 rows)
#define OM_PM_ROW_OK(r) (32 * (r) + 32 <= PW || lane + 32 * (r) < PW)
  double s[R];
#pragma unroll
  for (int r = 0; r < R; ++r) s[r] = 0.0;
#pragma unroll
  for (int u = 0; u < PM_ENVS; ++u) {
    const int env = env0 + u;
    if (env >= a.n) break;
    int tr = tr_[u], st = st_[u];
    uint32_t rc = rc_[u];
    if (start_reset) { traj_draw(a.t, a.seed, a.env_id0 + env, rc, tr, st); ++rc; }
    int left = a.n_steps;
    int lo = st + 1;                                   // the start row itself was emitted by the previous step / by reset()
    while (left > 0) {
      if (lo >= T) {                                   // wrap -> reset: the drawn sample itself is the next observation
        traj_draw(a.t, a.seed, a.env_id0 + env, rc, tr, st);
        ++rc;
        lo = st;
      }
      const int hi = min(T, lo + left);                // rows lo .. hi-1
      const double* p_lo = a.t.psum + ((size_t)tr * (T + 1) + lo) * PW + lane;
      const double* p_hi = a.t.psum + ((size_t)tr * (T + 1) + hi) * PW + lane;
      double h[R], l[R];
#pragma unroll
      for (int r = 0; r < R; ++r) h[r] = OM_PM_ROW_OK(r) ? __ldg(p_hi + 32 * r) : 0.0;
#pragma unroll
      for (int r = 0; r < R; ++r) l[r] = OM_PM_ROW_OK(r) ? __ldg(p_lo + 32 * r) : 0.0;
#pragma unroll
      for (int r = 0; r < R; ++r) s[r] += h[r] - l[r];
      left -= hi - lo;
      lo = hi;
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r)
    if (OM_PM_ROW_OK(r)) part[w][lane + 32 * r] = s[r];
#undef OM_PM_ROW_OK
  __syncthreads();
  if (threadIdx.x < PW) {
    double v = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) v += part[k][threadIdx.x];
    if (v != 0.0) atomicAdd(a.obs_moments + threadIdx.x, v);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(a.obs_moments + PW, (double)a.n * (double)a.n_steps);
}

template <class V, int BLOCK>
__global__ void __launch_bounds__(BLOCK) play_h1_seq_kernel(PlayArgsOf<V> a) {
  constexpr int NQ = V::NQ, K = H1Dims<V>::K, KPAD = H1Dims<V>::KPAD;
  const int env = blockIdx.x * BLOCK + threadIdx.x;
  if (env >= a.n) return;
  const size_t ld = a.ld, e = env;
  int tr = a.s.traj_no[e], st = a.s.step_no[e];
  uint32_t rc = a.s.reset_count[e];
  double ox = a.s.xy_off[e], oy = a.s.xy_off[ld + e];
  double cq[NQ];
  float dq[NQ];
#pragma unroll
  for (int k = 0; k < NQ; ++k) {
    cq[k] = a.s.curr_qpos ? a.s.curr_qpos[k * ld + e] : 0.0;
    dq[k] = a.s.pending[(NQ + k) * ld + e];
  }
  float pxv = a.s.prev_x_vel[e];
  const float mass = v_env_mass<V>(a, e);
  float samp[KPAD];
  bool have_samp = false;
  if (a.forced) {
#pragma unroll
    for (int k = 0; k < NQ; ++k) cq[k] = a.s.pending[k * ld + e];                    // play_trajectory: q = sample (:408)
  }
  for (int s = 0; s < a.n_steps; ++s) {
    if (!a.forced) {
#pragma unroll
      for (int k = 0; k < NQ; ++k) cq[k] = fma(a.dt, (double)dq[k], cq[k]);          // :515-519
    }
    play_fk<V, false>(cq, dq, a.o, (size_t)s, ld, e, mass);                            // :521-525 / :408-410
    ++st;                                                                            // :532
    const bool wrap = st >= a.t.T;
    if (wrap) {                                                                      // :534-537
      traj_draw(a.t, a.seed, a.env_id0 + env, rc, tr, st);
      ++rc;
      ox = a.t.xy[((size_t)tr * a.t.T + st) * 2];
      oy = a.t.xy[((size_t)tr * a.t.T + st) * 2 + 1];
    }
    traj_load_row(a.t, tr, st, samp);
    have_samp = true;
    if (a.forced) {                   // the next step is forced to this sample (x, y re-centred in double, then fp32)
      cq[0] = (float)(a.t.xy[((size_t)tr * a.t.T + st) * 2] - ox);
      cq[1] = (float)(a.t.xy[((size_t)tr * a.t.T + st) * 2 + 1] - oy);
#pragma unroll
      for (int k = 2; k < NQ; ++k) cq[k] = samp[k];
    } else if (wrap) {
      cq[0] = 0.0; cq[1] = 0.0;       // x - x_off and y - y_off are exactly zero at the reset sample
#pragma unroll
      for (int k = 2; k < NQ; ++k) cq[k] = samp[k];
    }
#pragma unroll
    for (int k = 0; k < NQ; ++k) dq[k] = samp[NQ + k];
    play_emit<V, false>(samp, pxv, a, (size_t)s, e, tr, st);                           // :539-541
    pxv = samp[NQ];                                                                  // dq_pelvis_tx
  }
  // write the loop's `sample` variable back (x, y re-centred) before the end-of-episode reset
  if (have_samp) {
    a.s.pending[e] = (float)(a.t.xy[((size_t)tr * a.t.T + st) * 2] - ox);
    a.s.pending[ld + e] = (float)(a.t.xy[((size_t)tr * a.t.T + st) * 2 + 1] - oy);
#pragma unroll
    for (int k = 2; k < K; ++k) a.s.pending[k * ld + e] = samp[k];
  }
  if (a.end_reset) {                                                                 // :555-557
    traj_draw(a.t, a.seed, a.env_id0 + env, rc, tr, st);
    ++rc;
    ox = a.t.xy[((size_t)tr * a.t.T + st) * 2];
    oy = a.t.xy[((size_t)tr * a.t.T + st) * 2 + 1];
    traj_load_row(a.t, tr, st, samp);
    cq[0] = 0.0; cq[1] = 0.0;
#pragma unroll
    for (int k = 2; k < NQ; ++k) cq[k] = samp[k];
    pxv = samp[NQ];
  }
  a.s.traj_no[e] = tr;
  a.s.step_no[e] = st;
  a.s.reset_count[e] = rc;
  a.s.xy_off[e] = ox;
  a.s.xy_off[ld + e] = oy;
#pragma unroll
  for (int k = 0; k < NQ; ++k) if (a.s.curr_qpos) a.s.curr_qpos[k * ld + e] = cq[k];
  a.s.prev_x_vel[e] = pxv;
}

// ---------------------------------------------------------------- fused playback, time-parallel
// reset() at the START of a playback call (loco_env_base.py:481 / :377: every call begins with self.reset();
// sample = get_current_sample(); curr_qpos = sample[:len_qpos]) for one env: the draw, then the carried state is written
// to `dst` (the live state for the sequential kernel, the episode-start snapshot for the time-parallel one).
template <class V>
OM_HD void play_start_reset(const PlayArgs& a, const OmPlayState& src, const OmPlayState& dst, int env) {
  constexpr int NQ = V::NQ, K = H1Dims<V>::K;
  const size_t ld = a.ld, e = env;
  int tr, st;
  const uint32_t rc = src.reset_count[e];
  traj_draw(a.t, a.seed, a.env_id0 + env, rc, tr, st);
  float samp[H1Dims<V>::KPAD];
  traj_reset_row(a.t, tr, st, samp);
  dst.traj_no[e] = tr;
  dst.step_no[e] = st;
  dst.reset_count[e] = rc + 1;
  dst.xy_off[e] = a.t.xy[((size_t)tr * a.t.T + st) * 2];
  dst.xy_off[ld + e] = a.t.xy[((size_t)tr * a.t.T + st) * 2 + 1];
#pragma unroll
  for (int k = 0; k < K; ++k) dst.pending[k * ld + e] = samp[k];
  if (dst.curr_qpos) {
#pragma unroll
    for (int k = 0; k < NQ; ++k) dst.curr_qpos[k * ld + e] = (double)samp[k];
  }
  dst.prev_x_vel[e] = samp[NQ];
}

template <class V>
__global__ void __launch_bounds__(256) play_start_reset_kernel(PlayArgs a) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < a.n) play_start_reset<V>(a, a.s, a.s, e);
}

template <class V, bool RESET>
__global__ void __launch_bounds__(256) play_snapshot_kernel(PlayArgs a, OmPlayState live, OmPlayState snap, int n, int ld) {
  constexpr int NQ = V::NQ, K = H1Dims<V>::K;
  pdl_trigger();                                 // a few CTAs: the playback kernel's first wave may become resident now
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  if (RESET) {                                   // the call starts with reset(): the snapshot IS the reset state
    play_start_reset<V>(a, live, snap, e);
    return;
  }
  // all loads first (the pointers may alias as far as the compiler knows: a load-store-load chain costs K round trips)
  double cq[NQ], xo[2];
  float pd[K];
#pragma unroll
  for (int k = 0; k < NQ; ++k) cq[k] = live.curr_qpos ? live.curr_qpos[(size_t)k * ld + e] : 0.0;
#pragma unroll
  for (int k = 0; k < K; ++k) pd[k] = live.pending[(size_t)k * ld + e];
  xo[0] = live.xy_off[e];
  xo[1] = live.xy_off[(size_t)ld + e];
  const int32_t tr = live.traj_no[e], st = live.step_no[e];
  const uint32_t rc = live.reset_count[e];
  const float pxv = live.prev_x_vel[e];
  snap.traj_no[e] = tr;
  snap.step_no[e] = st;
  snap.reset_count[e] = rc;
  snap.xy_off[e] = xo[0];
  snap.xy_off[(size_t)ld + e] = xo[1];
  snap.prev_x_vel[e] = pxv;
#pragma unroll
  for (int k = 0; k < NQ; ++k) snap.curr_qpos[(size_t)k * ld + e] = cq[k];
#pragma unroll
  for (int k = 0; k < K; ++k) snap.pending[(size_t)k * ld + e] = pd[k];
}

// The per-env recurrences of the playback loop are (a) the integer trajectory index, which only changes
// non-trivially at wrap resets whose draws depend on (seed, env, reset_count) alone, and (b) the Euler sum
// q_j = q_0 + dt * sum(dq), which telescopes through the float64 prefix table cdq.  A thread can therefore
// reconstruct the loop state in front of ANY step j0 in O(#resets) and then walk `chunk` steps exactly like
// the sequential kernel.  grid = (env tiles, time chunks): 4096 envs x 500 steps become ~300k threads
// instead of 4096, which is what lets a 4096-env rollout fill the 148 SMs.
template <class V, int BLOCK>
__global__ void __launch_bounds__(BLOCK) play_h1_tp_kernel(PlayArgsOf<V> a, int chunk) {
  constexpr int NQ = V::NQ, K = H1Dims<V>::K, KPAD = H1Dims<V>::KPAD;
  pdl_wait();                                    // launched while the snapshot kernel drains
  const int env = blockIdx.x * BLOCK + threadIdx.x;
  if (env >= a.n) return;
  const int j0 = blockIdx.y * chunk, j1 = min(j0 + chunk, a.n_steps);
  const size_t ld = a.ld, e = env;
  const int T = a.t.T;
  int tr = a.snap.traj_no[e], st = a.snap.step_no[e];
  uint32_t rc = a.snap.reset_count[e];
  const float mass = v_env_mass<V>(a, e);               // after pdl_wait: the draw of the preceding reset is visible
  // ---- replay the wrap resets that happen before step j0
  int seg_start = 0;
  bool first = true;
  while (seg_start + (T - st) <= j0) {
    seg_start += T - st;
    traj_draw(a.t, a.seed, a.env_id0 + env, rc, tr, st);
    ++rc;
    first = false;
  }
  const int m = j0 - seg_start;                  // steps already taken inside this segment
  double ox, oy;
  double cq[NQ];
  float dq[NQ];
  float pxv;
  float samp[KPAD];
  const double* c_hi = a.t.cdq + ((size_t)tr * (T + 1) + st + m) * NQ;
  if (a.forced) {
    // play_trajectory: the sim state of step j0 IS the pending sample -- the carried one when nothing happened yet,
    // else row (tr, st + m) re-centred with the offsets of the reset that opened this segment
    if (first) { ox = a.snap.xy_off[e]; oy = a.snap.xy_off[ld + e]; }
    else { ox = a.t.xy[((size_t)tr * T + st) * 2]; oy = a.t.xy[((size_t)tr * T + st) * 2 + 1]; }
    if (first && m == 0) {
#pragma unroll
      for (int k = 0; k < NQ; ++k) { cq[k] = a.snap.pending[k * ld + e]; dq[k] = a.snap.pending[(NQ + k) * ld + e]; }
      pxv = a.snap.prev_x_vel[e];
    }
  } else if (first) {
    ox = a.snap.xy_off[e]; oy = a.snap.xy_off[ld + e];
    const double* c_lo = a.t.cdq + ((size_t)tr * (T + 1) + st + 1) * NQ;
#pragma unroll
    for (int k = 0; k < NQ; ++k) {
      const double q0 = a.snap.curr_qpos[k * ld + e];
      const float p0 = a.snap.pending[(NQ + k) * ld + e];
      cq[k] = (m == 0) ? q0 : fma(a.dt, (double)p0 + (c_hi[k] - c_lo[k]), q0);
      dq[k] = p0;
    }
    pxv = a.snap.prev_x_vel[e];
  } else {
    ox = a.t.xy[((size_t)tr * T + st) * 2];
    oy = a.t.xy[((size_t)tr * T + st) * 2 + 1];
    traj_load_row(a.t, tr, st, samp);
    const double* c_lo = a.t.cdq + ((size_t)tr * (T + 1) + st) * NQ;
    cq[0] = fma(a.dt, c_hi[0] - c_lo[0], 0.0);
    cq[1] = fma(a.dt, c_hi[1] - c_lo[1], 0.0);
#pragma unroll
    for (int k = 2; k < NQ; ++k) cq[k] = fma(a.dt, c_hi[k] - c_lo[k], (double)samp[k]);
  }
  st += m;
  if (!first || m > 0) {                         // the pending sample is row (tr, st)
    traj_load_row(a.t, tr, st, samp);
#pragma unroll
    for (int k = 0; k < NQ; ++k) dq[k] = samp[NQ + k];
    pxv = samp[NQ];
    if (a.forced) {
      cq[0] = (float)(a.t.xy[((size_t)tr * T + st) * 2] - ox);
      cq[1] = (float)(a.t.xy[((size_t)tr * T + st) * 2 + 1] - oy);
#pragma unroll
      for (int k = 2; k < NQ; ++k) cq[k] = samp[k];
    }
  }
  // ---- walk the chunk (identical to the sequential kernel's loop body)
  for (int s = j0; s < j1; ++s) {
    if (!a.forced) {
#pragma unroll
      for (int k = 0; k < NQ; ++k) cq[k] = fma(a.dt, (double)dq[k], cq[k]);
    }
    play_fk<V, true>(cq, dq, a.o, (size_t)s, ld, e, mass);
    ++st;
    const bool wrap = st >= T;
    if (wrap) {
      traj_draw(a.t, a.seed, a.env_id0 + env, rc, tr, st);
      ++rc;
      ox = a.t.xy[((size_t)tr * T + st) * 2];
      oy = a.t.xy[((size_t)tr * T + st) * 2 + 1];
    }
    traj_load_row(a.t, tr, st, samp);
    if (a.forced) {
      cq[0] = (float)(a.t.xy[((size_t)tr * T + st) * 2] - ox);
      cq[1] = (float)(a.t.xy[((size_t)tr * T + st) * 2 + 1] - oy);
#pragma unroll
      for (int k = 2; k < NQ; ++k) cq[k] = samp[k];
    } else if (wrap) {
      cq[0] = 0.0; cq[1] = 0.0;
#pragma unroll
      for (int k = 2; k < NQ; ++k) cq[k] = samp[k];
    }
#pragma unroll
    for (int k = 0; k < NQ; ++k) dq[k] = samp[NQ + k];
    play_emit<V, true>(samp, pxv, a, (size_t)s, e, tr, st);
    pxv = samp[NQ];
  }
  if (j1 != a.n_steps) return;
  // ---- the thread that ran the last step owns the carried state
  a.s.pending[e] = (float)(a.t.xy[((size_t)tr * T + st) * 2] - ox);
  a.s.pending[ld + e] = (float)(a.t.xy[((size_t)tr * T + st) * 2 + 1] - oy);
#pragma unroll
  for (int k = 2; k < K; ++k) a.s.pending[k * ld + e] = samp[k];
  if (a.end_reset) {
    traj_draw(a.t, a.seed, a.env_id0 + env, rc, tr, st);
    ++rc;
    ox = a.t.xy[((size_t)tr * T + st) * 2];
    oy = a.t.xy[((size_t)tr * T + st) * 2 + 1];
    traj_load_row(a.t, tr, st, samp);
    cq[0] = 0.0; cq[1] = 0.0;
#pragma unroll
    for (int k = 2; k < NQ; ++k) cq[k] = samp[k];
    pxv = samp[NQ];
  }
  a.s.traj_no[e] = tr;
  a.s.step_no[e] = st;
  a.s.reset_count[e] = rc;
  a.s.xy_off[e] = ox;
  a.s.xy_off[ld + e] = oy;
#pragma unroll
  for (int k = 0; k < NQ; ++k) if (a.s.curr_qpos) a.s.curr_qpos[k * ld + e] = cq[k];
  a.s.prev_x_vel[e] = pxv;
}

// ---------------------------------------------------------------- fused live step
// One env step of a trajectory-driven rollout in ONE kernel (was traj_next -> set_sim_state -> h1_step, the sample and
// qpos / qvel round-tripping through HBM between three launches): advance the trajectory index (wrap -> reset,
// loco_env_base.py:534-537), gather the sample row (get_next_sample, trajectory.py:389-401), scatter it into qpos / qvel
// (set_sim_state :659-684; only written when the caller wants the MjData mirrors), K1 on it, observation
// (_create_observation :737-767), has_fallen, TargetVelocityReward on the PREVIOUS observation (mushroom MuJoCo.step:
// reward(self._obs, action, cur_obs, absorbing); self._obs = cur_obs).
struct LiveArgs {
  TrajDev t;
  uint64_t seed;
  uint32_t env_id0;
  float target;
  int use_absorbing, n, ld;
  int32_t* traj_no; int32_t* step_no; uint32_t* reset_count; double* xy_off; float* prev_x_vel;
  float* qpos; float* qvel;
  float* xpos; float* xquat; float* site_xpos; float* cvel;
  float* obs; float* reward; uint8_t* absorbing; uint8_t* wrapped;
  const float* env_mass;   // [ld] mass of the carried weight per env (V::ENV_MASS), else unused
};

// STREAM: streaming stores for the FK outputs (131 072 envs: 34.9 -> 31.8 us = 0.97 of HBM; 1 048 576 envs: 0.261 -> 0.266 ms,
// so the host picks by batch size)
template <class V, int BLOCK, bool STREAM>
__global__ void __launch_bounds__(BLOCK) h1_live_step_kernel(LiveArgs a) {
  constexpr int NQ = V::NQ, NOBS = H1Dims<V>::NOBS;
  pdl_wait();                                    // consecutive live steps: this launch overlaps the previous step's drain
  const int env = blockIdx.x * BLOCK + threadIdx.x;
  if (env >= a.n) return;
  const size_t ld = a.ld, e = env;
  const int T = a.t.T;
  int tr = a.traj_no[e], st = a.step_no[e] + 1;
  double ox = a.xy_off[e], oy = a.xy_off[ld + e];
  const float pxv = a.prev_x_vel[e];
  const bool wrap = st >= T;
  if (wrap) {
    const uint32_t rc = a.reset_count[e];
    traj_draw(a.t, a.seed, a.env_id0 + env, rc, tr, st);
    a.reset_count[e] = rc + 1;
    ox = a.t.xy[((size_t)tr * T + st) * 2];
    oy = a.t.xy[((size_t)tr * T + st) * 2 + 1];
    a.xy_off[e] = ox;
    a.xy_off[ld + e] = oy;
    a.traj_no[e] = tr;
  }
  a.step_no[e] = st;
  if (a.wrapped) a.wrapped[e] = wrap ? 1 : 0;
  float samp[H1Dims<V>::KPAD];
  traj_load_row(a.t, tr, st, samp);
  samp[0] = (float)(a.t.xy[((size_t)tr * T + st) * 2] - ox);
  samp[1] = (float)(a.t.xy[((size_t)tr * T + st) * 2 + 1] - oy);
  float q[NQ], qd[NQ];
#pragma unroll
  for (int k = 0; k < NQ; ++k) {
    q[V::perm(k)] = samp[k];
    qd[V::perm(k)] = samp[NQ + k];
  }
  if (a.qpos) {
#pragma unroll
    for (int k = 0; k < NQ; ++k) a.qpos[k * ld + e] = q[k];
  }
  if (a.qvel) {
#pragma unroll
    for (int k = 0; k < NQ; ++k) a.qvel[k * ld + e] = qd[k];
  }
  if (a.obs) {
#pragma unroll
    for (int k = 0; k < NOBS; ++k) a.obs[k * ld + e] = samp[k + 2];
  }
  if (a.absorbing) a.absorbing[e] = (a.use_absorbing && h1_fallen_f(samp[2], samp[3], samp[4], samp[5])) ? 1 : 0;
  if (a.reward) {
    const float d = pxv - a.target;
    a.reward[e] = expf(-(d * d));
  }
  a.prev_x_vel[e] = samp[NQ];                     // dq_pelvis_tx: emitted row NQ - 2 of UnitreeH1's own spec (checked on the host)
  if (a.xpos || a.xquat || a.site_xpos || a.cvel) {
    SoaSink<false, STREAM> S{a.xpos, a.xquat, a.site_xpos, nullptr, a.cvel, nullptr, ld, e};
    v_fk<V>(q, qd, S, v_env_mass<V>(a, e));      // after pdl_wait (top of the kernel)
  }
}

}  // namespace om

using namespace om;

#ifndef OM_H1_VARIANT
extern "C" int om_traj_create(const double* table, int K, int n_traj, int T, OmTraj** out) {
  OM_REQUIRE(table && out, "om_traj_create: null argument");
  OM_REQUIRE(K >= 2 && K <= 64 && n_traj >= 1 && T >= 1, "om_traj_create: bad shape K=%d n_traj=%d T=%d", K, n_traj, T);
  const int kpad = (K + 3) / 4 * 4;
  std::vector<float> rows((size_t)n_traj * T * kpad, 0.f);
  std::vector<double> xy((size_t)n_traj * T * 2);
  for (int k = 0; k < K; ++k)
    for (int tr = 0; tr < n_traj; ++tr)
      for (int s = 0; s < T; ++s) {
        const double v = table[((size_t)k * n_traj + tr) * T + s];
        rows[((size_t)tr * T + s) * kpad + k] = (float)v;
        if (k < 2) xy[((size_t)tr * T + s) * 2 + k] = v;
      }
  // exclusive prefix sums of the (fp32-rounded, as stored) velocity channels, accumulated in float64
  const int nq = K / 2;
  std::vector<double> cdq((size_t)n_traj * (T + 1) * nq, 0.0);
  for (int tr = 0; tr < n_traj; ++tr)
    for (int s = 0; s < T; ++s)
      for (int k = 0; k < nq; ++k)
        cdq[((size_t)tr * (T + 1) + s + 1) * nq + k] =
            cdq[((size_t)tr * (T + 1) + s) * nq + k] + (double)rows[((size_t)tr * T + s) * kpad + nq + k];
  // exclusive prefix sums of the emitted observation rows (channels 2 .. K-1, fp32-rounded as stored) and of their squares,
  // float64, for the key counts of the UnitreeH1 models with fused playback (no back joint 32, default and carry 34, arms
  // without / with the back joint 48 / 50):  psum[tr][i][c] = sum_{j<i} row_j[c+2], psum[tr][i][nobs+c] = sum_{j<i} row_j[c+2]^2
  std::vector<double> psum;
  if (K == 32 || K == 34 || K == 48 || K == 50) {
    const int nobs = K - 2, pw = 2 * nobs;
    psum.assign((size_t)n_traj * (T + 1) * pw, 0.0);
    for (int tr = 0; tr < n_traj; ++tr)
      for (int s = 0; s < T; ++s)
        for (int c = 0; c < nobs; ++c) {
          const double v = (double)rows[((size_t)tr * T + s) * kpad + c + 2];
          const size_t at = ((size_t)tr * (T + 1) + s) * pw;
          psum[at + pw + c] = psum[at + c] + v;
          psum[at + pw + nobs + c] = psum[at + nobs + c] + v * v;
        }
  }
  OmTraj* t = new OmTraj();
  t->d.K = K; t->d.kpad = kpad; t->d.n_traj = n_traj; t->d.T = T;
  float* drows = nullptr;
  double* dxy = nullptr;
  double* dcdq = nullptr;
  double* dpsum = nullptr;
  cudaError_t e = cudaMalloc(&drows, rows.size() * sizeof(float));
  if (e == cudaSuccess && !psum.empty()) e = cudaMalloc(&dpsum, psum.size() * sizeof(double));
  if (e == cudaSuccess && !psum.empty()) e = cudaMemcpy(dpsum, psum.data(), psum.size() * sizeof(double), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMalloc(&dxy, xy.size() * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&dcdq, cdq.size() * sizeof(double));
  if (e == cudaSuccess) e = cudaMemcpy(drows, rows.data(), rows.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(dxy, xy.data(), xy.size() * sizeof(double), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(dcdq, cdq.data(), cdq.size() * sizeof(double), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    if (drows) cudaFree(drows);
    if (dxy) cudaFree(dxy);
    if (dcdq) cudaFree(dcdq);
    if (dpsum) cudaFree(dpsum);
    delete t;
    return fail("om_traj_create: device upload failed: %s (no CPU path)", cudaGetErrorString(e));
  }
  t->d.rows = drows;
  t->d.xy = dxy;
  t->d.cdq = dcdq;
  t->d.psum = dpsum;
  *out = t;
  return 0;
}

extern "C" void om_traj_destroy(OmTraj* t) {
  if (!t) return;
  cudaFree((void*)t->d.rows);
  cudaFree((void*)t->d.xy);
  cudaFree((void*)t->d.cdq);
  if (t->d.psum) cudaFree((void*)t->d.psum);
  if (t->scratch) cudaFree(t->scratch);
  if (t->ev_fork) cudaEventDestroy(t->ev_fork);
  if (t->ev_join) cudaEventDestroy(t->ev_join);
  if (t->side) cudaStreamDestroy(t->side);
  delete t;
}

extern "C" int om_traj_reset(const OmTraj* t, uint64_t seed, uint32_t env_id0, const uint8_t* mask,
                             const int32_t* forced_traj, const int32_t* forced_step, int32_t* traj_no, int32_t* step_no,
                             uint32_t* reset_count, double* xy_off, float* sample, int n, int ld, void* stream) {
  OM_REQUIRE(t, "om_traj_reset: null table");
  OM_REQUIRE(n >= 0 && ld >= n, "om_traj_reset: need 0 <= n <= ld");
  if (n == 0) return 0;
  OM_REQUIRE(traj_no && step_no && reset_count && xy_off, "om_traj_reset: null state");
  traj_reset_kernel<<<ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(t->d, seed, env_id0, mask, forced_traj, forced_step,
                                                                         traj_no, step_no, reset_count, xy_off, sample, n, ld);
  OM_LAUNCHED();
  return 0;
}

extern "C" int om_traj_current(const OmTraj* t, const int32_t* traj_no, const int32_t* step_no, const double* xy_off,
                               float* sample, int n, int ld, void* stream) {
  OM_REQUIRE(t, "om_traj_current: null table");
  OM_REQUIRE(n >= 0 && ld >= n, "om_traj_current: need 0 <= n <= ld");
  if (n == 0) return 0;
  OM_REQUIRE(traj_no && step_no && xy_off && sample, "om_traj_current: null argument");
  traj_current_kernel<<<ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(t->d, traj_no, step_no, xy_off, sample, n, ld);
  OM_LAUNCHED();
  return 0;
}

extern "C" int om_traj_next(const OmTraj* t, uint64_t seed, uint32_t env_id0, int auto_reset, int32_t* traj_no,
                            int32_t* step_no, uint32_t* reset_count, double* xy_off, float* sample, uint8_t* wrapped,
                            int n, int ld, void* stream) {
  OM_REQUIRE(t, "om_traj_next: null table");
  OM_REQUIRE(n >= 0 && ld >= n, "om_traj_next: need 0 <= n <= ld");
  if (n == 0) return 0;
  OM_REQUIRE(traj_no && step_no && reset_count && xy_off, "om_traj_next: null state");
  traj_next_kernel<<<ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(t->d, seed, env_id0, auto_reset, traj_no, step_no, reset_count,
                                                                        xy_off, sample, wrapped, n, ld);
  OM_LAUNCHED();
  return 0;
}

namespace om {
// The model switch of a MultiMuJoCo reset() (loco_env_base.py:586-599), drawn per env: env i takes model
// Philox(seed; env_id0 + i, count, STREAM_MODEL_RESET) mod n_models, or (env_id0 + i + count + 1) mod n_models in round
// robin, and the mass its carried weight has in that model.
constexpr uint32_t STREAM_MODEL_RESET = 32u;      // utils/philox.py
constexpr int DRAW_MAX_MODELS = 16;
struct DrawMasses { float m[DRAW_MAX_MODELS]; };

__global__ void __launch_bounds__(256) h1_draw_models_kernel(uint64_t seed, uint32_t env_id0, uint32_t count, int n_models,
                                                             int random, DrawMasses masses, int32_t* idx, float* mass, int n) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const uint32_t env = env_id0 + (uint32_t)e;
  const int k = random ? to_int(om_draw(seed, env, count, STREAM_MODEL_RESET).x, n_models)
                       : (int)(((uint64_t)env + count + 1u) % (uint64_t)n_models);
  idx[e] = k;
  mass[e] = masses.m[k];
}
}  // namespace om

extern "C" int om_h1_draw_models(uint64_t seed, uint32_t env_id0, uint32_t count, int n_models, int random,
                                 const double* body_mass_host, int32_t* idx, float* mass, int n, void* stream) {
  OM_REQUIRE(n_models >= 1 && n_models <= DRAW_MAX_MODELS, "om_h1_draw_models: n_models %d outside [1,%d]", n_models,
             DRAW_MAX_MODELS);
  OM_REQUIRE(body_mass_host, "om_h1_draw_models: null body_mass_host");
  OM_REQUIRE(n >= 0, "om_h1_draw_models: n < 0");
  if (n == 0) return 0;
  OM_REQUIRE(idx && mass, "om_h1_draw_models: null output");
  DrawMasses dm = {};
  for (int k = 0; k < n_models; ++k) dm.m[k] = (float)body_mass_host[k];
  h1_draw_models_kernel<<<ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(seed, env_id0, count, n_models, random ? 1 : 0,
                                                                            dm, idx, mass, n);
  OM_LAUNCHED();
  return 0;
}

#endif  // !OM_H1_VARIANT

namespace om {

// ---------------------------------------------------------------- host launchers of one variant
// The C entry points validate the arguments against the model, then launch through the model's entry.
struct H1Kernels {
  int nq;                      // observation-spec joints; the trajectory has 2 nq keys
  const int* perm_host;        // [nq] qpos/qvel address of observation-spec entry k
  int (*play)(const OmTraj* t, const PlayArgs& a, bool start_reset, void* stream, const float* env_mass);
  int (*live)(const LiveArgs& a, void* stream);
};

template <class V>
int play_launch(const OmTraj* t, const PlayArgs& args, bool start_reset, void* stream, const float* env_mass) {
  constexpr int BLOCK = PLAY_BLOCK;
  PlayArgsOf<V> a;
  static_cast<PlayArgs&>(a) = args;
  if constexpr (V::ENV_MASS) a.env_mass = env_mass;
  const int n = a.n, n_steps = a.n_steps, ld = a.ld;
  const bool mom = a.obs_moments != nullptr;
  // time-parallel when the env count alone cannot fill the machine (148 SMs x 2048 threads)
  const long long target_threads = 148LL * 2048;
  const long long chunks_wanted = target_threads / n > 0 ? target_threads / n : 1;
  int chunk = ceil_div(n_steps, chunks_wanted);
  if (g_knobs.play_chunk > 0) chunk = g_knobs.play_chunk;            // tuning / test hook (om_debug_set)
  if (chunk < 1) chunk = 1;
  if (chunk >= n_steps) {
    if (mom) {                                      // reads the START state: before anything below touches it
      play_moments_kernel<V><<<ceil_div(n, 8 * PM_ENVS), 256, 0, (cudaStream_t)stream>>>(a, a.s, start_reset ? 1 : 0);
      OM_LAUNCHED();
    }
    if (start_reset) {
      play_start_reset_kernel<V><<<ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(a);
      OM_LAUNCHED();
    }
    play_h1_seq_kernel<V, BLOCK><<<ceil_div(n, BLOCK), BLOCK, 0, (cudaStream_t)stream>>>(a);
    OM_LAUNCHED();
    return 0;
  }
  // the carried state is read by every chunk and overwritten by the last one: snapshot the episode-start
  // state (stream-ordered scratch) so that no thread can observe another's end-of-episode write
  constexpr int NQ = V::NQ, K = H1Dims<V>::K;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t L = (size_t)ld;
  const size_t bytes = L * (4 + 4 + 4 + 16 + 4 + NQ * 8 + K * 4) + 256;
  if (t->scratch_bytes < bytes) {
    if (t->scratch) OM_CUDA_OK(cudaFree(t->scratch));       // synchronises: no earlier call still reads it
    t->scratch = nullptr;
    t->scratch_bytes = 0;
    OM_CUDA_OK(cudaMalloc((void**)&t->scratch, bytes));
    t->scratch_bytes = bytes;
  }
  char* p = t->scratch;
  a.snap.curr_qpos = (double*)p; p += L * NQ * 8;
  a.snap.xy_off = (double*)p; p += L * 16;
  a.snap.pending = (float*)p; p += L * K * 4;
  a.snap.prev_x_vel = (float*)p; p += L * 4;
  a.snap.traj_no = (int32_t*)p; p += L * 4;
  a.snap.step_no = (int32_t*)p; p += L * 4;
  a.snap.reset_count = (uint32_t*)p;
  if (start_reset) play_snapshot_kernel<V, true><<<ceil_div(n, 256), 256, 0, st>>>(a, a.s, a.snap, n, ld);
  else play_snapshot_kernel<V, false><<<ceil_div(n, 256), 256, 0, st>>>(a, a.s, a.snap, n, ld);
  OM_LAUNCHED();
  dim3 grid(ceil_div(n, BLOCK), ceil_div(n_steps, chunk));
  if (mom) {
    // The moments kernel (L2-bound: prefix-table reads) runs BESIDE the playback kernel (DRAM-bound) on a side stream:
    // both only read the snapshot, which now holds the state after the call's start reset.  Plain fork / join with two
    // events, legal under stream capture.
    if (!t->side) {
      OM_CUDA_OK(cudaStreamCreateWithFlags(&t->side, cudaStreamNonBlocking));
      OM_CUDA_OK(cudaEventCreateWithFlags(&t->ev_fork, cudaEventDisableTiming));
      OM_CUDA_OK(cudaEventCreateWithFlags(&t->ev_join, cudaEventDisableTiming));
    }
    OM_CUDA_OK(cudaEventRecord(t->ev_fork, st));
    OM_CUDA_OK(cudaStreamWaitEvent(t->side, t->ev_fork, 0));
    play_moments_kernel<V><<<ceil_div(n, 8 * PM_ENVS), 256, 0, t->side>>>(a, a.snap, 0);
    OM_LAUNCHED();
    OM_CUDA_OK(cudaEventRecord(t->ev_join, t->side));
  }
  OM_CUDA_OK(launch_pdl(play_h1_tp_kernel<V, BLOCK>, grid, dim3(BLOCK), 0, st, a, chunk));
  OM_LAUNCHED();
  if (mom) OM_CUDA_OK(cudaStreamWaitEvent(st, t->ev_join, 0));
  return 0;
}

template <class V>
int live_launch(const LiveArgs& a, void* stream) {
  constexpr int BLOCK = 128;
  const int n = a.n;
  if (n <= 524288) OM_CUDA_OK(launch_pdl(h1_live_step_kernel<V, BLOCK, true>, dim3(ceil_div(n, BLOCK)), dim3(BLOCK), 0, (cudaStream_t)stream, a));
  else OM_CUDA_OK(launch_pdl(h1_live_step_kernel<V, BLOCK, false>, dim3(ceil_div(n, BLOCK)), dim3(BLOCK), 0, (cudaStream_t)stream, a));
  OM_LAUNCHED();
  return 0;
}

}  // namespace om

#ifndef OM_H1_VARIANT
namespace om {

// ---------------------------------------------------------------- the default model's kernels
// UnitreeH1 with the arms disabled and the back joint kept (variant id 1): one instantiation of the kernels above.  The
// other variants are instantiated by the -DOM_H1_VARIANT compilations of this file.
struct H1Default {
  static constexpr int ID = 1, NQ = 17, NBODY = 21, NSITE = 1;
  static constexpr bool ENV_MASS = false;
  static OM_HD int perm(int k) { return OM_H1_PERM[k]; }
  template <class Sink>
  static OM_HD void fk(const float (&q)[NQ], const float (&qd)[NQ], Sink& S) { om_fk_unitree_h1(q, qd, S); }
};

static const H1Kernels h1k_default = {H1Default::NQ, OM_H1_PERM_HOST, &play_launch<H1Default>, &live_launch<H1Default>};
#define OM_H1_VARIANT_DECL(id, name) extern const H1Kernels h1k_##name;
OM_H1_VARIANTS(OM_H1_VARIANT_DECL)
#undef OM_H1_VARIANT_DECL
extern const H1Kernels h1k_carry_env;    // the carry model with a per-env weight mass (gen/h1v/carry_env.cuh)

// the fused kernels of the model's variant (OmModel::h1_variant), or null; a carry model bound to a per-env weight mass
// launches the carry_env kernels instead
static const H1Kernels* h1_kernels(const OmModel* m) {
  if (m->env_mass) return &h1k_carry_env;
  switch (m->h1_variant) {
    case H1Default::ID: return &h1k_default;
#define OM_H1_VARIANT_CASE(id, name) case id: return &h1k_##name;
    OM_H1_VARIANTS(OM_H1_VARIANT_CASE)
#undef OM_H1_VARIANT_CASE
    default: return nullptr;
  }
}

}  // namespace om

static int play_impl(const OmModel* m, const OmH1Spec* spec, const OmTraj* t, uint64_t seed, uint32_t env_id0, double dt,
                     int n_steps, int end_episode_reset, const OmPlayState* state, const OmPlayOut* out, int n, int ld,
                     void* stream, int forced) {
  OM_REQUIRE(m && spec && t && state && out, "om_h1_play_from_velocity: null argument");
  OM_REQUIRE(n >= 0 && ld >= n && n_steps >= 0, "om_h1_play_from_velocity: bad sizes");
  const H1Kernels* hk = h1_kernels(m);
  OM_REQUIRE(hk, "om_h1_play_from_velocity: model is not a UnitreeH1 model with fused kernels");
  OM_REQUIRE(spec->n_obs_q == hk->nq && t->d.K == 2 * hk->nq,
             "om_h1_play_from_velocity: expects the %d-key trajectory of this UnitreeH1 model", 2 * hk->nq);
  for (int k = 0; k < hk->nq; ++k)
    OM_REQUIRE(spec->obs_perm[k] == hk->perm_host[k], "om_h1_play_from_velocity: observation spec differs from UnitreeH1's");
  if (n == 0) return 0;
  OM_REQUIRE(state->traj_no && state->step_no && state->reset_count && state->xy_off && (forced || state->curr_qpos) &&
                 state->pending && state->prev_x_vel, "om_h1_play_from_velocity: incomplete state");
  PlayArgs a;
  a.t = t->d; a.seed = seed; a.env_id0 = env_id0; a.dt = dt; a.target = spec->target_velocity;
  a.n_steps = n_steps; a.end_reset = end_episode_reset & 1;
  const bool start_reset = (end_episode_reset & 2) != 0;          // OM_PLAY_START_RESET
  a.n = n; a.ld = ld; a.s = *state; a.snap = *state; a.o = *out; a.forced = forced;
  a.obs_moments = out->obs_moments;
  OM_REQUIRE(!m->env_mass || n <= m->env_mass_ld, "om_h1_play_from_velocity: %d envs, but the bound body mass holds %d",
             n, m->env_mass_ld);
  OM_REQUIRE(!a.obs_moments || t->d.psum, "om_h1_play_from_velocity: this trajectory handle has no prefix tables");
  return hk->play(t, a, start_reset, stream, m->env_mass);
}

extern "C" int om_h1_play_from_velocity(const OmModel* m, const OmH1Spec* spec, const OmTraj* t, uint64_t seed,
                                        uint32_t env_id0, double dt, int n_steps, int end_episode_reset,
                                        const OmPlayState* state, const OmPlayOut* out, int n, int ld, void* stream) {
  return play_impl(m, spec, t, seed, env_id0, dt, n_steps, end_episode_reset, state, out, n, ld, stream, 0);
}

extern "C" int om_h1_play_trajectory(const OmModel* m, const OmH1Spec* spec, const OmTraj* t, uint64_t seed, uint32_t env_id0,
                                     int n_steps, int end_episode_reset, const OmPlayState* state, const OmPlayOut* out, int n,
                                     int ld, void* stream) {
  return play_impl(m, spec, t, seed, env_id0, 0.0, n_steps, end_episode_reset, state, out, n, ld, stream, 1);
}

extern "C" int om_h1_live_step(const OmModel* m, const OmH1Spec* spec, const OmTraj* t, uint64_t seed, uint32_t env_id0,
                               const OmLiveState* state, const OmLiveOut* out, int n, int ld, void* stream) {
  OM_REQUIRE(m && spec && t && state && out, "om_h1_live_step: null argument");
  OM_REQUIRE(n >= 0 && ld >= n, "om_h1_live_step: need 0 <= n <= ld (n=%d ld=%d)", n, ld);
  const H1Kernels* hk = h1_kernels(m);
  OM_REQUIRE(hk, "om_h1_live_step: model is not a UnitreeH1 model with fused kernels");
  OM_REQUIRE(spec->n_obs_q == hk->nq && t->d.K == 2 * hk->nq,
             "om_h1_live_step: expects the %d-key trajectory of this UnitreeH1 model", 2 * hk->nq);
  OM_REQUIRE(spec->x_vel_idx == hk->nq - 2, "om_h1_live_step: x_vel_idx must be %d (dq_pelvis_tx of UnitreeH1's own spec)",
             hk->nq - 2);
  for (int k = 0; k < hk->nq; ++k)
    OM_REQUIRE(spec->obs_perm[k] == hk->perm_host[k], "om_h1_live_step: observation spec differs from UnitreeH1's");
  if (n == 0) return 0;
  OM_REQUIRE(state->traj_no && state->step_no && state->reset_count && state->xy_off && state->prev_x_vel,
             "om_h1_live_step: incomplete state");
  LiveArgs a;
  a.t = t->d; a.seed = seed; a.env_id0 = env_id0; a.target = spec->target_velocity;
  a.use_absorbing = spec->use_absorbing_states; a.n = n; a.ld = ld;
  a.traj_no = state->traj_no; a.step_no = state->step_no; a.reset_count = state->reset_count; a.xy_off = state->xy_off;
  a.prev_x_vel = state->prev_x_vel;
  a.qpos = out->qpos; a.qvel = out->qvel; a.xpos = out->xpos; a.xquat = out->xquat; a.site_xpos = out->site_xpos;
  a.cvel = out->cvel; a.obs = out->obs; a.reward = out->reward; a.absorbing = out->absorbing; a.wrapped = out->wrapped;
  a.env_mass = m->env_mass;
  OM_REQUIRE(!m->env_mass || n <= m->env_mass_ld, "om_h1_live_step: %d envs, but the bound body mass holds %d", n,
             m->env_mass_ld);
  return hk->live(a, stream);
}
#else
#define OM_PASTE2(a, b) a##b
#define OM_PASTE(a, b) OM_PASTE2(a, b)
namespace om {
extern const H1Kernels OM_PASTE(h1k_, OM_H1_VARIANT) = {OM_PASTE(H1V_, OM_H1_VARIANT)::NQ,
                                                        OM_PASTE(H1V_, OM_H1_VARIANT)::perm_host(),
                                                        &play_launch<OM_PASTE(H1V_, OM_H1_VARIANT)>,
                                                        &live_launch<OM_PASTE(H1V_, OM_H1_VARIANT)>};
}  // namespace om
#endif  // !OM_H1_VARIANT
