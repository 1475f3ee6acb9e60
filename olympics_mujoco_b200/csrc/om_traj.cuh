// Device view of a reference-trajectory table (K3) and the gather / reset helpers shared by kernels.
#pragma once
#include "om_common.cuh"

namespace om {

struct TrajDev {
  const float* rows;   // [n_traj][T][kpad] sample-major rows (one 16-byte aligned row per sample)
  const double* xy;    // [n_traj][T][2]   channels 0,1 (root x, y) in float64
  const double* cdq;   // [n_traj][T+1][K/2] exclusive prefix sums of the velocity channels (float64):
                       //   cdq[tr][i][k] = sum_{j<i} rows[tr][j][K/2+k]  (time-parallel playback)
  const double* psum;  // [n_traj][T+1][2 (K-2)] exclusive prefix sums of the observation rows (channels 2..K-1) and of
                       //   their squares, float64 (S1 of a playback call as prefix differences); null unless K is the
                       //   key count of a UnitreeH1 model with fused kernels (32, 34, 48 or 50)
  int K, kpad, n_traj, T;
};

// reset_trajectory draws (trajectory.py:304,311) under the Philox contract
OM_HD void traj_draw(const TrajDev& t, uint64_t seed, uint32_t env_id, uint32_t reset_count, int& traj_no, int& step_no) {
  const U4 w = om_draw(seed, env_id, reset_count, 0u);
  traj_no = to_int(w.x, t.n_traj);
  step_no = to_int(w.y, t.T);
}

// one sample row into registers (KPAD == t.kpad, checked on the host); vectorised 16-byte gathers
template <int KPAD>
OM_HD void traj_load_row(const TrajDev& t, int traj_no, int step_no, float (&samp)[KPAD]) {
  static_assert(KPAD % 4 == 0, "rows are padded to whole float4s");
  const float4* r = reinterpret_cast<const float4*>(t.rows + ((size_t)traj_no * t.T + step_no) * t.kpad);
#pragma unroll
  for (int v = 0; v < KPAD / 4; ++v) {
    const float4 x = __ldg(r + v);
    samp[4 * v] = x.x; samp[4 * v + 1] = x.y; samp[4 * v + 2] = x.z; samp[4 * v + 3] = x.w;
  }
}

// the sample a reset starts from: row (traj_no, step_no) with root x, y re-centred on that row (reset_trajectory,
// trajectory.py:316-320) -- x - x_off and y - y_off are exactly zero there
template <int KPAD>
OM_HD void traj_reset_row(const TrajDev& t, int traj_no, int step_no, float (&samp)[KPAD]) {
  traj_load_row(t, traj_no, step_no, samp);
  samp[0] = 0.f; samp[1] = 0.f;
}

// get_current_sample (trajectory.py:381-387) for one env into a [K][ld] SoA array
OM_HD void traj_write_sample(const TrajDev& t, int traj_no, int step_no, double ox, double oy, float* sample, int ld, int env) {
  const size_t row = (size_t)traj_no * t.T + step_no;
  sample[env] = (float)(t.xy[row * 2] - ox);
  sample[(size_t)ld + env] = (float)(t.xy[row * 2 + 1] - oy);
  const float* r = t.rows + row * t.kpad;
  for (int k = 2; k < t.K; ++k) sample[(size_t)k * ld + env] = __ldg(r + k);
}

}  // namespace om

// the OmTraj handle of the C ABI (om_traj.cu creates it; om_reset.cu reads its table)
struct OmTraj {
  om::TrajDev d;
  // Scratch of the time-parallel playback kernel (episode-start snapshot of the carried state), grown on demand
  // and kept: a stream-ordered allocation per call cost more than the kernel whenever the pool had been trimmed.
  // One playback call per handle may be in flight at a time.
  mutable char* scratch = nullptr;
  mutable size_t scratch_bytes = 0;
  // fork / join of the observation-moments kernel beside the time-parallel playback kernel (both only READ the snapshot)
  mutable cudaStream_t side = nullptr;
  mutable cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
};
