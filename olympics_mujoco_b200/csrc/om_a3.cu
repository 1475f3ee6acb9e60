// K2 (A3 flavour) kernels and C ABI: StickFigureA3 RL step tail (FK fused, not materialised unless asked for),
// multi-step replay of recorded sim states, and the randomised reset.  Per-env arithmetic: om_a3_task.cuh.
#include <cmath>
#include <cstdlib>
#include <vector>

#include "om_common.cuh"
#include "om_sinks.cuh"
#include "om_a3_task.cuh"

namespace om {

struct A3Args {
  A3TaskConst C;
  const float* qpos;      // [T][25][ld]
  const float* qvel;      // [T][24][ld]
  const float* contact;   // [T][4][ld]: l_grf, r_grf, min contact z, flags (1 = foot-floor contact, 2 = bad collision)
  int32_t* ints;          // [7][ld]
  float* sequence;        // [80][ld]
  OmA3Out o;
  int T, n, ld;
};

struct SeqGlobal {
  const float* base; size_t ld;
  OM_HD float operator()(int t, int c) const { return base[(unsigned)(t * 4 + c) * (unsigned)ld]; }     // 80 rows: 32-bit offsets
};
struct SeqStore {
  float* base; size_t ld;
  OM_HD void operator()(int t, int c, float v) const { base[(size_t)(t * 4 + c) * ld] = v; }
};

// One thread per env walks its T recorded steps; the integer task state lives in registers across steps and the
// next step's 53 inputs are requested before the current step's FK so that the loads overlap the arithmetic.
template <int BLOCK, bool WRITE_FK>
__global__ void __launch_bounds__(BLOCK) a3_task_kernel(A3Args a) {
  const int env = blockIdx.x * BLOCK + threadIdx.x;
  if (env >= a.n) return;
  const size_t ld = a.ld, e = env;
  A3TaskRegs s{a.ints[A3I_PHASE * ld + e], a.ints[A3I_T1 * ld + e], a.ints[A3I_T2 * ld + e], a.ints[A3I_FRAMES * ld + e],
               a.ints[A3I_MODE * ld + e], a.ints[A3I_SEQLEN * ld + e], a.ints[A3I_REACHED * ld + e]};
  const SeqGlobal seq{a.sequence + e, ld};
  float q[A3_NQ], qd[A3_NV], con[4];
  auto load = [&](int t, float (&q_)[A3_NQ], float (&qd_)[A3_NV], float (&c_)[4]) {
    const float* qp = a.qpos + (size_t)t * A3_NQ * ld + e;
    const float* vp = a.qvel + (size_t)t * A3_NV * ld + e;
    const float* cp = a.contact + (size_t)t * 4 * ld + e;
#pragma unroll
    for (int k = 0; k < A3_NQ; ++k) q_[k] = qp[k * ld];
#pragma unroll
    for (int k = 0; k < A3_NV; ++k) qd_[k] = vp[k * ld];
#pragma unroll
    for (int k = 0; k < 4; ++k) c_[k] = cp[k * ld];
  };
  load(0, q, qd, con);
  A3Targets tc = a3_targets_load(s, seq);
  for (int t = 0; t < a.T; ++t) {
    float qn[A3_NQ], qdn[A3_NV], conn[4];
    if (t + 1 < a.T) load(t + 1, qn, qdn, conn);
    float obs[A3_NOBS], terms[6], total;
    bool done;
    a3_obs_robot(q, qd, obs);
    A3TaskIn in;
    if (WRITE_FK) {
      const size_t slot = (size_t)t;
      A3Sink<SoaSink<true>> S{{a.o.xpos ? a.o.xpos + slot * 51 * ld : nullptr, a.o.xquat ? a.o.xquat + slot * 68 * ld : nullptr,
                               a.o.site_xpos ? a.o.site_xpos + slot * 6 * ld : nullptr,
                               a.o.site_xmat ? a.o.site_xmat + slot * 18 * ld : nullptr,
                               a.o.cvel ? a.o.cvel + slot * 102 * ld : nullptr, nullptr, ld, e}, {}};
      om_fk_stick_figure_a3(q, qd, S);
      in = a3_task_in(S.f);
    } else {
      A3Sink<NullFkSink> S{};
      om_fk_pos_stick_figure_a3(q, qd, S);       // matrix-chain variant: no body orientations needed
      in = a3_task_in(S.f);
    }
    const int fl = (int)con[3];
    a3_task_step(a.C, A3Exact{a.qpos + (size_t)t * A3_NQ * ld + e, ld, false, false}, in, s, tc, seq, con[0], con[1], con[2], (fl & 1) != 0, (fl & 2) != 0, obs, terms, total, done);
    if (a.o.obs) {
      float* ob = a.o.obs + (size_t)t * A3_NOBS * ld + e;
#pragma unroll
      for (int k = 0; k < A3_NOBS; ++k) ob[k * ld] = obs[k];
    }
    if (a.o.terms) {
      float* tp = a.o.terms + (size_t)t * 6 * ld + e;
#pragma unroll
      for (int k = 0; k < 6; ++k) tp[k * ld] = terms[k];
    }
    if (a.o.reward) a.o.reward[(size_t)t * ld + e] = total;
    if (a.o.done) a.o.done[(size_t)t * ld + e] = done ? 1 : 0;
    if (t + 1 < a.T) {
#pragma unroll
      for (int k = 0; k < A3_NQ; ++k) q[k] = qn[k];
#pragma unroll
      for (int k = 0; k < A3_NV; ++k) qd[k] = qdn[k];
#pragma unroll
      for (int k = 0; k < 4; ++k) con[k] = conn[k];
    }
  }
  a.ints[A3I_PHASE * ld + e] = s.phase; a.ints[A3I_T1 * ld + e] = s.t1; a.ints[A3I_T2 * ld + e] = s.t2;
  a.ints[A3I_FRAMES * ld + e] = s.frames; a.ints[A3I_REACHED * ld + e] = s.reached;
}

// ---------------------------------------------------------------- time-parallel replay (few envs, many steps)
// The only recurrence over time is the task's footstep-target state machine; everything expensive (FK, the
// state-independent 33 observation rows, four reward terms) depends on (env, t) alone.
//   a3_feat_kernel  one thread per (env, t): FK + a3_task_pre; leaves a 16-float record per env-step plus one byte of
//                   "a foot is near candidate target j" bits (om_a3_task.cuh: a3_near_bits).  ~1900 instructions and
//                   660 B of HBM traffic per env-step: issue time and memory time are of the same size.  (Measured and
//                   rejected: persistent CTAs staging the next tile's inputs in shared memory with cp.async or
//                   cp.async.bulk -- the CTAs fall into lockstep, load, compute and store phases stop overlapping
//                   across CTAs, 112 us instead of 90 us.)
//   a3_walk_kernel  one thread per env: the integer state machine over the T bytes (a few instructions per step),
//                   leaves a one-byte (advances, reached) code per env-step and the final task state.  (Measured and
//                   rejected: running it in the last-finishing feat CTA of each env block -- 147 us instead of 142; and
//                   as the first `env_blocks` CTAs of the post kernel -- the float64 re-decision's registers become the
//                   post kernel's: 128 registers, or 64 with spills, 150 us instead of 121.)
//   a3_post_kernel  one thread per (env, t) again: goal steps, orientation and step terms, total.  Starts while the walk
//                   runs, each thread waiting for its own state code (see a3_walk_kernel): the walk costs 2 us of the
//                   call instead of 17.
struct A3Scratch {
  float* feat;          // [T][16][ld]
  // ONE byte per env-step, ENV-major ([ld][tp], tp = T rounded up to 16), written twice:
  //   by the feat pass   candidate bits 0..5 | 0x40 if a decision has to be re-taken in float64    (bit 7 clear)
  //   by the walk pass   advances since the call started | reached << 3 | 0x80, after the step's update
  // The sequential pass reads and rewrites an env's bytes in place as 16-byte vectors (4 loads per 64 steps instead of 64
  // with their address arithmetic -- it runs one warp per scheduler, every instruction's latency is exposed); the
  // (env, t)-parallel passes touch one byte per thread.  Bit 7 is what the post pass, which starts while the walk runs,
  // waits for.
  uint8_t* step;
  int tp;
  int32_t* start;       // [2][ld]   t1, t2 at the start of the call
  float* trig;          // [A3_MAX_CAND + 1][4][ld]   sin, cos of candidate j's heading and of half of it (feat t = 0 -> post)
};

// Row k of a per-(env, t) SoA block: ONE 64-bit base pointer per array (it carries t and the env), rows addressed by the
// 32-bit, warp-uniform offset k * ld -- one IMAD.WIDE per access.  Written as (t * C + k) * ld + e in size_t the compiler
// spent five integer instructions on every one of the ~120 loads and stores of this kernel: a third of its instructions.
// (om_a3_task_step checks that rows * ld fits 32 bits.)
__device__ __forceinline__ const float* row(const float* base, unsigned k, unsigned ld) { return base + k * ld; }
__device__ __forceinline__ float* row(float* base, unsigned k, unsigned ld) { return base + k * ld; }

// one env-step of the (env, t)-parallel pass
__device__ __forceinline__ void a3_feat_item(const A3Args& a, const A3Scratch& w, int ncand, int t, size_t e) {
  const size_t ld = a.ld;
  const unsigned lu = (unsigned)a.ld;
  float q[A3_NQ], qd[A3_NV], con[4];
  const float* qp = a.qpos + (size_t)t * A3_NQ * ld + e;
  const float* vp = a.qvel + (size_t)t * A3_NV * ld + e;
  const float* cp = a.contact + (size_t)t * 4 * ld + e;
#pragma unroll
  // inputs are read once and the observations written once: streaming accesses (evict-first), so that the 64 MB of
  // records this pass leaves for the post pass have a chance to stay in the 126 MB L2
  for (int k = 0; k < A3_NQ; ++k) q[k] = __ldcs(row(qp, k, lu));
#pragma unroll
  for (int k = 0; k < A3_NV; ++k) qd[k] = __ldcs(row(vp, k, lu));
#pragma unroll
  for (int k = 0; k < 4; ++k) con[k] = __ldcs(row(cp, k, lu));
  int phase = a.ints[A3I_PHASE * ld + e] + (t + 1) % a.C.period;            // walking_task.py:248-250, t + 1 increments;
  if (phase >= a.C.period) phase -= a.C.period;                            // the modulo is warp-uniform, the wrap a select
  const int mode = a.ints[A3I_MODE * ld + e];
  const int t1_0 = a.ints[A3I_T1 * ld + e], t2_0 = a.ints[A3I_T2 * ld + e], seq_len = a.ints[A3I_SEQLEN * ld + e];
  const int frames0 = a.ints[A3I_FRAMES * ld + e];
  // The candidate targets' rows are a SECOND level of dependent loads (ints -> row index -> row), consumed only after the
  // forward pass: ask for their lines now, without registers, so that they arrive under the FK arithmetic.
  const int nc = a3_cand_needed(t, frames0, a.C.delay_frames, ncand);      // later targets are out of reach
#pragma unroll 1
  for (int j = 0; j < nc; ++j) {
    const float* p = a.sequence + e + (unsigned)(a3_cand(j, t1_0, t2_0, seq_len) * 4) * lu;
    asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(row(p, 1, lu)));
    asm volatile("prefetch.global.L1 [%0];" ::"l"(row(p, 2, lu)));
  }
  if (t == 0) {                                                            // start state of the call for the post pass
    w.start[e] = t1_0;
    w.start[ld + e] = t2_0;
    for (int j = 0; j <= ncand; ++j) {             // headings of every target the call can reach, and of the one after
      const float th = a.sequence[(size_t)(a3_cand(j, t1_0, t2_0, seq_len) * 4 + 3) * ld + e];
      float sn, cs, sh, ch;
      om_sincos(th, &sn, &cs);
      om_sincos(0.5f * th, &sh, &ch);
      float* tr = w.trig + (size_t)j * 4 * ld + e;
      tr[0] = sn; tr[ld] = cs; tr[2 * ld] = sh; tr[3 * ld] = ch;
    }
  }
  float obs[A3_NOBS], terms[6];
  a3_obs_robot(q, qd, obs);
  A3Sink<NullFkSink> S{};
  om_fk_pos_stick_figure_a3(q, qd, S);           // matrix-chain variant: no body orientations needed
  bool done;
  const int fl = (int)con[3];
  A3Exact ex{qp, ld, true, false};               // decisions within A3_BAND of a threshold are only NOTED here (bit 6 below)
  const A3Rec rec = a3_task_pre(a.C, a3_task_in(S.f), phase, mode, con[0], con[1], con[2], (fl & 1) != 0, (fl & 2) != 0, terms,
                                obs[31], obs[32], done, ex);
  a3_rec_store(rec, w.feat + (size_t)t * A3_NREC * ld + e, lu);
  const uint32_t bits = a3_near_bits(a.C, rec.lsite, rec.rsite, nc, t1_0, t2_0, seq_len, SeqGlobal{a.sequence + e, ld}, ex);
  // bit 6: a decision of this env-step (done, or one of the candidate bits) is within A3_BAND of its threshold; the
  // sequential pass re-takes it in float64 (a3_refix) before it consumes the byte -- about one env-step in 10^4
  w.step[e * w.tp + t] = (uint8_t)(bits | (ex.unsure ? 0x40u : 0u));
  if (a.o.obs) {
    float* ob = a.o.obs + (size_t)t * A3_NOBS * ld + e;
#pragma unroll
    for (int k = 0; k < 33; ++k) __stcs(row(ob, k, lu), obs[k]);
  }
  if (a.o.terms) {
    float* tp = a.o.terms + (size_t)t * 6 * ld + e;
    __stcs(tp, terms[0]); __stcs(row(tp, 1, lu), terms[1]); __stcs(row(tp, 3, lu), terms[3]); __stcs(row(tp, 5, lu), terms[5]);
  }
  if (a.o.done) a.o.done[(size_t)t * ld + e] = done ? 1 : 0;
}

// Re-takes, in float64, the threshold decisions of ONE env-step that the (env, t)-parallel pass could not settle in fp32
// (margin below A3_BAND): rewrites its `done` flag and returns its exact candidate bits.  Out of line: it is called by the
// sequential pass for about one env-step in 10^4.
__device__ __noinline__ uint32_t a3_refix(const A3Args& a, int ncand, int t, size_t e) {
  const size_t ld = a.ld;
  const float* qp = a.qpos + (size_t)t * A3_NQ * ld + e;
  const A3SitesF64 s = a3_sites_f64(qp, ld);
  if (a.o.done) {
    const int fl = (int)a.contact[((size_t)t * 4 + 3) * ld + e];
    a.o.done[(size_t)t * ld + e] = ((double)qp[2 * ld] - fmin(s.ls[2], s.rs[2]) < 0.6 || (fl & 2) != 0) ? 1 : 0;
  }
  const int t1_0 = a.ints[A3I_T1 * ld + e], t2_0 = a.ints[A3I_T2 * ld + e], seq_len = a.ints[A3I_SEQLEN * ld + e];
  const int nc = a3_cand_needed(t, a.ints[A3I_FRAMES * ld + e], a.C.delay_frames, ncand);
  uint32_t bits = 0;
  for (int j = 0; j < nc; ++j) {
    const int k = a3_cand(j, t1_0, t2_0, seq_len);
    const double px = (double)a.sequence[(size_t)(k * 4) * ld + e], py = (double)a.sequence[(size_t)(k * 4 + 1) * ld + e];
    const double pz = (double)a.sequence[(size_t)(k * 4 + 2) * ld + e];
    const double lx = s.ls[0] - px, ly = s.ls[1] - py, lz = s.ls[2] - pz;
    const double rx = s.rs[0] - px, ry = s.rs[1] - py, rz = s.rs[2] - pz;
    if (sqrt(lx * lx + ly * ly + lz * lz) < a.C.target_radius || sqrt(rx * rx + ry * ry + rz * rz) < a.C.target_radius)
      bits |= 1u << j;
  }
  return bits;
}

// The integer state machine over the T candidate bytes of one env (a few instructions per step); leaves a one-byte
// (advances, reached) code per env-step and the final task state.
__device__ __forceinline__ void a3_walk(const A3Args& a, const A3Scratch& w, int ncand, size_t e) {
  const size_t ld = a.ld;
  const int t1_0 = a.ints[A3I_T1 * ld + e], t2_0 = a.ints[A3I_T2 * ld + e], seq_len = a.ints[A3I_SEQLEN * ld + e];
  A3Walk s{0, a.ints[A3I_FRAMES * ld + e], a.ints[A3I_REACHED * ld + e]};
  uint4* cd = reinterpret_cast<uint4*>(w.step + e * w.tp);
  const uint4* nb = cd;
  for (int t0 = 0; t0 < a.T; t0 += 64) {
    uint32_t wi[16];
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const uint4 in = t0 + 16 * v < a.T ? nb[(t0 >> 4) + v] : make_uint4(0, 0, 0, 0);
      wi[4 * v] = in.x; wi[4 * v + 1] = in.y; wi[4 * v + 2] = in.z; wi[4 * v + 3] = in.w;
    }
    uint32_t any = 0;
#pragma unroll
    for (int q = 0; q < 16; ++q) any |= wi[q];
    if (any & 0x40404040u) {                                         // rare: a flagged env-step among these 64
      // One bit per flagged byte, then one float64 re-decision per loop trip: every lane of the warp that holds a flagged
      // byte makes its FIRST trip together with the others (same code, no divergence), so a warp pays for the largest
      // count in one lane -- almost always one -- not for the sum over its lanes.
      uint64_t pend = 0;
#pragma unroll
      for (int q = 0; q < 16; ++q)                                   // bits 6, 14, 22, 30 of word q -> bits 4q .. 4q + 3
        pend |= (uint64_t)((((wi[q] & 0x40404040u) << 1) * 0x00204081u) >> 28) << (4 * q);
#pragma unroll 1
      while (pend) {
        const int k = __ffsll((long long)pend) - 1;
        pend &= pend - 1;
        if (t0 + k < a.T) {
          const uint32_t exact = a3_refix(a, ncand, t0 + k, e);
          const uint32_t keep = ~(0xffu << (8 * (k & 3))), put = exact << (8 * (k & 3));
#pragma unroll
          for (int q = 0; q < 16; ++q)                               // static indices: wi stays in registers
            if (q == (k >> 2)) wi[q] = (wi[q] & keep) | put;
        }
      }
    }
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      if (t0 + 16 * v < a.T) {
        uint32_t wo[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint32_t o = 0;
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            if (t0 + 16 * v + 4 * q + b < a.T) {                     // bytes past T are padding
              a3_walk_step(a.C, (wi[4 * v + q] >> (8 * b)) & 0xffu, s);
              o |= (uint32_t)(s.j | (s.reached << 3) | 0x80) << (8 * b);
            }
          }
          wo[q] = o;
        }
        cd[(t0 >> 4) + v] = make_uint4(wo[0], wo[1], wo[2], wo[3]);
      }
    }
  }
  a.ints[A3I_PHASE * ld + e] = (a.ints[A3I_PHASE * ld + e] + a.T) % a.C.period;
  a.ints[A3I_T1 * ld + e] = a3_cand(s.j, t1_0, t2_0, seq_len);
  a.ints[A3I_T2 * ld + e] = a3_cand(s.j + 1, t1_0, t2_0, seq_len);
  a.ints[A3I_FRAMES * ld + e] = s.frames; a.ints[A3I_REACHED * ld + e] = s.reached;
}

template <int BLOCK, int MINB>
__global__ void __launch_bounds__(BLOCK, MINB) a3_feat_kernel(A3Args a, A3Scratch w, int ncand) {
  const int env = blockIdx.x * BLOCK + threadIdx.x;
  if (env < a.n) a3_feat_item(a, w, ncand, blockIdx.y, env);
}

// The sequential pass and the second (env, t)-parallel pass OVERLAP.  The walk kernel (one thread per env) waits for the
// feat kernel, lets its dependent launch, and walks; the post kernel's CTAs are therefore scheduled while the walk runs
// (every walk CTA has started by then, so nothing a post thread waits for can be starved), load their records, and each
// thread waits for bit 7 of ITS state code -- the one thing it reads from the walk, so the byte is its own flag and no
// fence is involved.  An env whose walk has to re-take decisions in float64 (a3_refix, ~5 us) holds back only the
// warps it sits in, and the launch boundary between the two passes is gone.  The post kernel does not call
// griddepcontrol.wait: it is launched only once every walk CTA is past its own wait, i.e. after the feat kernel has
// completed and flushed.
__global__ void __launch_bounds__(64) a3_walk_kernel(A3Args a, A3Scratch w, int ncand) {
  pdl_wait();
  pdl_trigger();
  const int env = blockIdx.x * 64 + threadIdx.x;
  if (env < a.n) a3_walk(a, w, ncand, env);
}

template <int BLOCK>
__global__ void __launch_bounds__(BLOCK) a3_post_kernel(A3Args a, A3Scratch w) {
  const int t = blockIdx.y;
  const int env = blockIdx.x * BLOCK + threadIdx.x;
  if (env >= a.n) return;
  const size_t ld = a.ld, e = env;
  const unsigned lu = (unsigned)a.ld;
  const int mode = a.ints[A3I_MODE * ld + e], seq_len = a.ints[A3I_SEQLEN * ld + e];
  const int t1_0 = w.start[e], t2_0 = w.start[ld + e];
  // the two targets' rows depend on the state code (a second level of dependent loads): in most env-steps no target has
  // been reached yet in this call, so ask for the rows of candidates 0 and 1 while the record is being loaded
  {
    const float* p0 = a.sequence + e + (unsigned)(t1_0 * 4) * lu;
    const float* p1 = a.sequence + e + (unsigned)(a3_cand(1, t1_0, t2_0, seq_len) * 4) * lu;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      asm volatile("prefetch.global.L1 [%0];" ::"l"(row(p0, c, lu)));
      asm volatile("prefetch.global.L1 [%0];" ::"l"(row(p1, c, lu)));
    }
  }
  const A3Rec rec = a3_rec_load(w.feat + (size_t)t * A3_NREC * ld + e, lu);
  int code;
  {
    const volatile uint8_t* cp = w.step + e * w.tp + t;                // volatile: from L2, where the walk's store lands
    while (!((code = *cp) & 0x80)) __nanosleep(100);
  }
  const int j = code & 7;
  const float* tr = w.trig + e + (unsigned)(j * 4) * lu;               // candidate j, then candidate j + 1
  const A3TargetTrig tg{tr[0], *row(tr, 1, lu), *row(tr, 4, lu), *row(tr, 5, lu), *row(tr, 2, lu), *row(tr, 3, lu)};
  float goal[8], tm2, tm4, total;
  a3_task_post(a.C, rec, mode, a3_cand(j, t1_0, t2_0, seq_len), a3_cand(j + 1, t1_0, t2_0, seq_len), (code & 8) != 0,
               SeqGlobal{a.sequence + e, ld}, &tg, goal, tm2, tm4, total);
  if (a.o.obs) {
    float* ob = a.o.obs + ((size_t)t * A3_NOBS + 33) * ld + e;
#pragma unroll
    for (int k = 0; k < 8; ++k) __stcs(row(ob, k, lu), goal[k]);
  }
  if (a.o.terms) {
    float* tp = a.o.terms + (size_t)t * 6 * ld + e;
    __stcs(row(tp, 2, lu), tm2);
    __stcs(row(tp, 4, lu), tm4);
  }
  if (a.o.reward) a.o.reward[(size_t)t * ld + e] = total;
}

// (Measured and rejected: finishing the discounted returns inside the post pass -- a CTA owning 32 envs x all steps, each
// thread walking 8 consecutive steps and composing the affine recurrence from the rewards it has just computed.  Bit-equal
// to post + affine_scan, but 52 us unrolled (instruction cache) / 59 us rolled against 28 + 10 us for the two kernels: one
// thread per (env, t) hides the record / table latencies far better than eight sequential steps per thread.)
struct A3ResetArgs {
  A3TaskConst C;
  const float* init_qpos;   // device [25]
  uint64_t seed;
  uint32_t env_id0;
  const uint8_t* mask;
  uint32_t* reset_count;
  float step_h;
  float* qpos; float* qvel; int32_t* ints; float* sequence; float* obs;
  int n, ld;
};

// The reset of one env: the draws of counter reset_count[env] (then incremented), pose, FK for the foot positions
// transform_sequence reads, WalkingTask.reset; writes qpos, qvel, the task ints, the footstep plan and -- a.obs not NULL --
// the first observation.  Shared by the masked reset and the auto-reset after a step (Args: A3ResetArgs, A3AutoResetArgs).
template <class Args>
__device__ __forceinline__ void a3_reset_env(const Args& a, int env) {
  const size_t ld = a.ld, e = env;
  const uint32_t rc = a.reset_count[e];
  a.reset_count[e] = rc + 1;
  float u[A3_NU], q[A3_NQ], qd[A3_NV];
  a3_reset_uniforms(a.seed, a.env_id0 + env, rc, u);
  a3_reset_qpos_qvel(a.init_qpos, u, q, qd);
  A3Sink<NullFkSink> S{};
  om_fk_pos_stick_figure_a3(q, qd, S);                                 // set_state -> mj_forward
  A3TaskRegs s;
  a3_task_reset(a.C, S.f, u, a.step_h, s, SeqStore{a.sequence + e, ld});
#pragma unroll
  for (int k = 0; k < A3_NQ; ++k) a.qpos[k * ld + e] = q[k];
#pragma unroll
  for (int k = 0; k < A3_NV; ++k) a.qvel[k * ld + e] = qd[k];
  a.ints[A3I_PHASE * ld + e] = s.phase; a.ints[A3I_T1 * ld + e] = s.t1; a.ints[A3I_T2 * ld + e] = s.t2;
  a.ints[A3I_FRAMES * ld + e] = s.frames; a.ints[A3I_MODE * ld + e] = s.mode; a.ints[A3I_SEQLEN * ld + e] = s.seq_len;
  a.ints[A3I_REACHED * ld + e] = s.reached;
  if (a.obs) {                                                         // get_obs: goal steps are zero after task.reset
    float obs[A3_NOBS];
    a3_obs_robot(q, qd, obs);
    const float* lrow = a.C.lut + (size_t)s.phase * A3_LUT_COLS;
    obs[31] = lrow[4];
    obs[32] = lrow[5];
#pragma unroll
    for (int k = 33; k < A3_NOBS; ++k) obs[k] = 0.f;
#pragma unroll
    for (int k = 0; k < A3_NOBS; ++k) a.obs[k * ld + e] = obs[k];
  }
}

__global__ void __launch_bounds__(128) a3_reset_kernel(A3ResetArgs a) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= a.n) return;
  if (a.mask && !a.mask[env]) return;
  a3_reset_env(a, env);
}

// The PPO sampler's path bookkeeping after one step (rl/algos/ppo.py:150-198): traj_len += 1; the path ends on done or at
// max_traj_len (0 = never); path_end = 1 (done: bootstrap 0, wins over a truncation on the same step), 2 (truncated:
// bootstrap V(final obs)) or 0; an env whose path ended is reset exactly as a3_reset_kernel resets it.  obs = the step's
// observation (obs_in) where no reset happened, the new first observation where one did.
struct A3AutoResetArgs {
  A3TaskConst C;
  const float* init_qpos;
  uint64_t seed;
  uint32_t env_id0;
  float step_h;
  int max_traj_len;
  const uint8_t* done;
  uint32_t* reset_count; int32_t* traj_len;
  float* qpos; float* qvel; int32_t* ints; float* sequence;
  const float* obs_in; float* obs;
  uint8_t* last; uint8_t* path_end;
  int n, ld;
};

__global__ void __launch_bounds__(128) a3_autoreset_kernel(A3AutoResetArgs a) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= a.n) return;
  const size_t ld = a.ld, e = env;
  const bool done = a.done[e] != 0;
  const int tl = a.traj_len[e] + 1;
  const bool trunc = a.max_traj_len > 0 && tl >= a.max_traj_len;
  const bool end = done || trunc;
  a.last[e] = end ? 1 : 0;
  a.path_end[e] = done ? 1 : (trunc ? 2 : 0);
  a.traj_len[e] = end ? 0 : tl;
  if (end) {
    a3_reset_env(a, env);
  } else if (a.obs != a.obs_in) {                                      // the step's observation stays the env's observation
    float v[A3_NOBS];
#pragma unroll
    for (int k = 0; k < A3_NOBS; ++k) v[k] = a.obs_in[k * ld + e];
#pragma unroll
    for (int k = 0; k < A3_NOBS; ++k) a.obs[k * ld + e] = v[k];
  }
}

}  // namespace om

using namespace om;

struct OmA3Task {
  A3TaskConst C;
  float* lut = nullptr;        // device [period][6]
  float* init_qpos = nullptr;  // device [25]
  // scratch of the time-parallel replay (records, state codes, env-block counters), grown on demand and kept; one
  // replay call per handle may be in flight at a time
  mutable void* scratch = nullptr;
  mutable size_t scratch_bytes = 0;
};

extern "C" int om_a3_task_create(const OmA3TaskDesc* d, OmA3Task** out) {
  OM_REQUIRE(d && out, "om_a3_task_create: null argument");
  OM_REQUIRE(d->period >= 2 && d->period <= 4096 && d->period % 2 == 0, "om_a3_task_create: period %d must be even and in [2,4096]", d->period);
  OM_REQUIRE(d->delay_frames >= 0 && d->total_mass > 0 && d->clock_lut_host && d->init_qpos_host, "om_a3_task_create: bad description");
  std::vector<float> lut((size_t)d->period * A3_LUT_COLS);
  for (int p = 0; p < d->period; ++p) {
    for (int c = 0; c < 4; ++c) lut[(size_t)p * A3_LUT_COLS + c] = (float)d->clock_lut_host[p * 4 + c];
    lut[(size_t)p * A3_LUT_COLS + 4] = (float)std::sin(2.0 * M_PI * p / d->period);     // StickFigureA3.py:147-148
    lut[(size_t)p * A3_LUT_COLS + 5] = (float)std::cos(2.0 * M_PI * p / d->period);
  }
  float iq[A3_NQ];
  for (int k = 0; k < A3_NQ; ++k) iq[k] = (float)d->init_qpos_host[k];
  OmA3Task* t = new OmA3Task();
  cudaError_t e = cudaMalloc(&t->lut, lut.size() * sizeof(float));
  if (e == cudaSuccess) e = cudaMalloc(&t->init_qpos, sizeof iq);
  if (e == cudaSuccess) e = cudaMemcpy(t->lut, lut.data(), lut.size() * sizeof(float), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(t->init_qpos, iq, sizeof iq, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    if (t->lut) cudaFree(t->lut);
    if (t->init_qpos) cudaFree(t->init_qpos);
    delete t;
    return fail("om_a3_task_create: device upload failed: %s (no CPU path)", cudaGetErrorString(e));
  }
  t->C.period = d->period;
  t->C.delay_frames = d->delay_frames;
  t->C.fmax = (float)(d->total_mass * 9.8 * 0.5);
  t->C.vmax = 0.2f;
  t->C.inv_fmax = 1.0f / t->C.fmax;
  t->C.inv_vmax = 1.0f / t->C.vmax;
  t->C.target_radius = d->target_radius;
  t->C.near_d2 = a3_near_d2(d->target_radius);
  a3_near_band(d->target_radius, &t->C.near_lo2, &t->C.near_hi2);
  t->C.goal_height_ref = d->goal_height_ref;
  t->C.deadzone = 0.01 + 0.05 * d->goal_speed_ref;
  t->C.lut = t->lut;
  *out = t;
  return 0;
}

extern "C" void om_a3_task_destroy(OmA3Task* t) {
  if (!t) return;
  cudaFree(t->lut);
  cudaFree(t->init_qpos);
  if (t->scratch) cudaFree(t->scratch);
  delete t;
}

static int a3_step_impl(const OmModel* m, const OmA3Task* task, const float* qpos, const float* qvel, const float* contact,
                        int n_steps, const OmA3State* state, const OmA3Out* out, const OmA3Returns* rets, int n, int ld,
                        void* stream) {
  OM_REQUIRE(m && task && state && out, "om_a3_task_step: null argument");
  OM_REQUIRE(m->specialised == SPEC_A3, "om_a3_task_step: model is not the StickFigureA3 model");
  OM_REQUIRE(n >= 0 && ld >= n && n_steps >= 0, "om_a3_task_step: bad sizes (n=%d ld=%d n_steps=%d)", n, ld, n_steps);
  OM_REQUIRE((unsigned long long)ld * 128ull < 0xffffffffull, "om_a3_task_step: ld too large for 32-bit row offsets");
  if (n == 0 || n_steps == 0) return 0;
  OM_REQUIRE(qpos && qvel && contact && state->ints && state->sequence, "om_a3_task_step: null input / state");
  A3Args a{task->C, qpos, qvel, contact, state->ints, state->sequence, *out, n_steps, n, ld};
  const bool want_fk = out->xpos || out->xquat || out->site_xpos || out->site_xmat || out->cvel;
  constexpr int BLOCK = 64;
  const int grid = ceil_div(n, BLOCK);
  cudaStream_t st = (cudaStream_t)stream;
  // Several steps: time-parallel replay (measured faster than the fused kernel at 16384 and at 262144 envs x 64 steps:
  // 0.37 vs 0.21 and 0.72 vs 0.65 of the HBM roofline); one step: the fused kernel, one launch.
  int split = !want_fk && n_steps >= 2;
  if (g_knobs.a3_split >= 0) split = g_knobs.a3_split != 0 && !want_fk;             // tuning / test hook (om_debug_set)
  if (split) {
    constexpr int FB = 128;
    const int env_blocks = ceil_div(n, FB);
    // layout: [records][start ints + heading table][per-step bytes]
    const size_t feat_b = (size_t)n_steps * A3_NREC * (size_t)ld * sizeof(float);
    const size_t int_b = ((size_t)(2 + (A3_MAX_CAND + 1) * 4) * ld * sizeof(int32_t) + 15) / 16 * 16;   // byte arrays 16-B aligned
    const int tp_max = (n_steps + 15) / 16 * 16;
    const size_t byte_b = (size_t)tp_max * (size_t)ld;
    const size_t need = feat_b + int_b + byte_b;
    OM_REQUIRE(env_blocks <= 65535, "om_a3_task_step: at most %d envs per multi-step call", 65535 * FB);
    if (task->scratch_bytes < need) {
      if (task->scratch) OM_CUDA_OK(cudaFree(task->scratch));  // synchronises: no earlier call still reads it
      task->scratch = nullptr;
      task->scratch_bytes = 0;
      OM_CUDA_OK(cudaMalloc(&task->scratch, need));
      task->scratch_bytes = need;
    }
    char* base = (char*)task->scratch;
    A3Scratch w{(float*)base, (uint8_t*)(base + feat_b + int_b), 0,
                (int32_t*)(base + feat_b), (float*)(base + feat_b) + 2 * (size_t)ld};
    // sub-calls no longer than the candidate bits cover (150 steps with the reference's 30 delay frames)
    const int max_call = a3_max_steps_per_call(task->C.delay_frames);
    for (int c0 = 0; c0 < n_steps; c0 += max_call) {
      const int len = n_steps - c0 < max_call ? n_steps - c0 : max_call;
      A3Args sub = a;
      sub.qpos += (size_t)c0 * A3_NQ * ld; sub.qvel += (size_t)c0 * A3_NV * ld; sub.contact += (size_t)c0 * 4 * ld;
      if (sub.o.obs) sub.o.obs += (size_t)c0 * A3_NOBS * ld;
      if (sub.o.terms) sub.o.terms += (size_t)c0 * 6 * ld;
      if (sub.o.reward) sub.o.reward += (size_t)c0 * ld;
      if (sub.o.done) sub.o.done += (size_t)c0 * ld;
      sub.T = len;
      w.tp = (len + 15) / 16 * 16;
      OM_REQUIRE(len <= 65535, "om_a3_task_step: at most 65535 steps per call");
      const int ncand = a3_num_cand_host(len, task->C.delay_frames);
      // 64-thread CTAs, ten per SM (the same 20 warps as 128 x 5, finer-grained: 0.5 % / 1.5 % faster at 16384 / 262144
      // envs); knob values 4 / 5 / 6: 128-thread CTAs compiled for that many per SM (tuning)
      if (g_knobs.a3_feat_minb == 6) a3_feat_kernel<FB, 6><<<dim3(env_blocks, len), FB, 0, st>>>(sub, w, ncand);
      else if (g_knobs.a3_feat_minb == 5) a3_feat_kernel<FB, 5><<<dim3(env_blocks, len), FB, 0, st>>>(sub, w, ncand);
      else if (g_knobs.a3_feat_minb == 4) a3_feat_kernel<FB, 4><<<dim3(env_blocks, len), FB, 0, st>>>(sub, w, ncand);
      else a3_feat_kernel<64, 10><<<dim3(ceil_div(n, 64), len), 64, 0, st>>>(sub, w, ncand);
      OM_LAUNCHED();
      OM_CUDA_OK(launch_pdl(a3_walk_kernel, dim3(ceil_div(n, 64)), dim3(64), 0, st, sub, w, ncand));
      OM_LAUNCHED();
      OM_CUDA_OK(launch_pdl(a3_post_kernel<FB>, dim3(env_blocks, len), dim3(FB), 0, st, sub, w));
      OM_LAUNCHED();
    }
    if (rets)                                     // the returns scan over the rewards just written (same stream, same call)
      return om_ppo_returns(out->reward, rets->values, rets->path_end ? rets->path_end : out->done, rets->v_next, rets->v_last,
                            rets->gamma, n_steps, n, ld, rets->ret, rets->adv, stream);
    return 0;
  }
  if (want_fk) a3_task_kernel<BLOCK, true><<<grid, BLOCK, 0, st>>>(a);
  else a3_task_kernel<BLOCK, false><<<grid, BLOCK, 0, st>>>(a);
  OM_LAUNCHED();
  if (rets)
    return om_ppo_returns(out->reward, rets->values, rets->path_end ? rets->path_end : out->done, rets->v_next, rets->v_last,
                          rets->gamma, n_steps, n, ld, rets->ret, rets->adv, stream);
  return 0;
}

extern "C" int om_a3_task_step(const OmModel* m, const OmA3Task* task, const float* qpos, const float* qvel,
                               const float* contact, int n_steps, const OmA3State* state, const OmA3Out* out, int n, int ld,
                               void* stream) {
  return a3_step_impl(m, task, qpos, qvel, contact, n_steps, state, out, nullptr, n, ld, stream);
}

extern "C" int om_a3_task_rollout(const OmModel* m, const OmA3Task* task, const float* qpos, const float* qvel,
                                  const float* contact, int n_steps, const OmA3State* state, const OmA3Out* out,
                                  const OmA3Returns* returns, int n, int ld, void* stream) {
  OM_REQUIRE(returns && out, "om_a3_task_rollout: null argument");
  OM_REQUIRE(out->reward && returns->ret, "om_a3_task_rollout: the reward and ret buffers are required");
  OM_REQUIRE(returns->path_end || out->done, "om_a3_task_rollout: the returns need the done flags (out->done) or path_end");
  OM_REQUIRE(!returns->adv || returns->values, "om_a3_task_rollout: advantages need values");
  return a3_step_impl(m, task, qpos, qvel, contact, n_steps, state, out, returns, n, ld, stream);
}

// WalkingTask.reset's step height for the curriculum position iteration_count (walking_task.py:378)
static float a3_step_height(double iteration_count) {
  double h = (iteration_count - 3000.0) / 8000.0;
  h = (h < 0.0 ? 0.0 : (h > 1.0 ? 1.0 : h)) * 0.1;
  return (float)h;
}

extern "C" int om_a3_reset(const OmModel* m, const OmA3Task* task, uint64_t seed, uint32_t env_id0, const uint8_t* mask,
                           uint32_t* reset_count, double iteration_count, float* qpos, float* qvel, const OmA3State* state,
                           float* obs, int n, int ld, void* stream) {
  OM_REQUIRE(m && task && state, "om_a3_reset: null argument");
  OM_REQUIRE(m->specialised == SPEC_A3, "om_a3_reset: model is not the StickFigureA3 model");
  OM_REQUIRE(n >= 0 && ld >= n, "om_a3_reset: need 0 <= n <= ld");
  if (n == 0) return 0;
  OM_REQUIRE(reset_count && qpos && qvel && state->ints && state->sequence, "om_a3_reset: null state");
  A3ResetArgs a{task->C, task->init_qpos, seed, env_id0, mask, reset_count, a3_step_height(iteration_count), qpos, qvel,
                state->ints, state->sequence, obs, n, ld};
  a3_reset_kernel<<<ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(a);
  OM_LAUNCHED();
  return 0;
}

extern "C" int om_a3_autoreset(const OmModel* m, const OmA3Task* task, uint64_t seed, uint32_t env_id0,
                               const OmA3AutoResetArgs* args, int n, int ld, void* stream) {
  OM_REQUIRE(m && task && args, "om_a3_autoreset: null argument");
  OM_REQUIRE(m->specialised == SPEC_A3, "om_a3_autoreset: model is not the StickFigureA3 model");
  OM_REQUIRE(n >= 0 && ld >= n, "om_a3_autoreset: need 0 <= n <= ld (n=%d ld=%d)", n, ld);
  const OmA3AutoResetArgs& r = *args;
  OM_REQUIRE(r.max_traj_len >= 0, "om_a3_autoreset: max_traj_len %d < 0 (0 = no limit)", r.max_traj_len);
  if (n == 0) return 0;
  OM_REQUIRE(r.done && r.reset_count && r.traj_len && r.qpos && r.qvel && r.state.ints && r.state.sequence && r.obs_in &&
             r.obs && r.last && r.path_end,
             "om_a3_autoreset: null input / state (done, reset_count, traj_len, qpos, qvel, state, obs_in, obs, last and "
             "path_end are required)");
  A3AutoResetArgs a{task->C, task->init_qpos, seed, env_id0, a3_step_height(r.iteration_count), r.max_traj_len, r.done,
                    r.reset_count, r.traj_len, r.qpos, r.qvel, r.state.ints, r.state.sequence, r.obs_in, r.obs, r.last,
                    r.path_end, n, ld};
  a3_autoreset_kernel<<<ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(a);
  OM_LAUNCHED();
  return 0;
}
