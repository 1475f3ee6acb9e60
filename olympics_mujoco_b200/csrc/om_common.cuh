// Shared host/device helpers for libom_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <string>

#include "../../include/om_b200.h"

#ifndef OM_HD
#define OM_HD __device__ __forceinline__
#endif

namespace om {

// ---------------------------------------------------------------- errors / bookkeeping (host)
std::string& last_error();
int fail(const char* fmt, ...);
extern std::atomic<long long> g_launches;

// Tuning / test knobs (om_debug_set; initialised ONCE from the OM_* environment variables when the library is loaded --
// no getenv on any launch path).  -1 / 0 = automatic.
struct Knobs {
  int play_chunk = 0;     // OM_PLAY_CHUNK   time-chunk length of the time-parallel playback kernel
  int h1_split = -1;      // OM_H1_SPLIT     1 / 0: force / forbid the three-threads-per-env H1 step kernel
  int a3_split = -1;      // OM_A3_SPLIT     1 / 0: force / forbid the time-parallel A3 replay
  int serial_scan = 0;    // OM_SERIAL_SCAN  1: one-thread-per-env returns / GAE kernels
  int disc_vail2 = -1;    // OM_DISC_VAIL2   VAIL kernel: -1 / 4 one CTA per SM with the A operand in TMEM (default), 1 two CTAs per SM
                          //                 (shared-memory operands), 3 two CTAs per SM with A in TMEM, 0 the kernels that also serve GAIL
  int disc_pg2 = -1;      // OM_DISC_PG2     1 / 0: two producer warpgroups
  int a3_feat_minb = 0;   // OM_A3_FEAT_MINB 0: 64-thread CTAs, ten per SM (default); 4 / 5 / 6: 128-thread CTAs, that many per SM (tuning)
};
extern Knobs g_knobs;

#define OM_CUDA_OK(expr)                                                                     \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) return om::fail("%s failed: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

#define OM_LAUNCHED()                                                                      \
  do {                                                                                     \
    om::g_launches.fetch_add(1, std::memory_order_relaxed);                                \
    cudaError_t _e = cudaGetLastError();                                                   \
    if (_e != cudaSuccess) return om::fail("kernel launch failed: %s", cudaGetErrorString(_e)); \
  } while (0)

#define OM_REQUIRE(cond, ...) \
  do {                        \
    if (!(cond)) return om::fail(__VA_ARGS__); \
  } while (0)

inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// Programmatic dependent launch: a chain of small kernels on one stream (snapshot -> playback -> scan -> moments -> stats ->
// normalise; feat -> walk -> post -> scan) pays a launch-and-drain gap at every boundary.  Launched with this attribute a
// kernel's CTAs are scheduled while its predecessor drains; the kernel itself calls pdl_wait() (griddepcontrol.wait) before it
// touches anything the predecessor wrote, which blocks until the predecessor has completed and flushed -- whatever kernel
// that was (ours or the caller's).  No early trigger is used, so nothing else about the ordering changes.
template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// Called at the START of a TINY kernel: its dependent's CTAs may become resident right away (the machine is otherwise idle)
// and park in pdl_wait() until this kernel has completed -- the dependent's launch and ramp-up hide under this kernel.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif

// ---------------------------------------------------------------- device tables of a model
constexpr int MAXB = OM_MAX_BODY;
constexpr int MAXJ = OM_MAX_JNT;
constexpr int MAXS = OM_MAX_SITE;
constexpr int MAXQ = 64;

struct ModelTab {
  int nbody, njnt, nsite, nq, nv;
  int body_parent[MAXB], body_root[MAXB], body_jntadr[MAXB], body_jntnum[MAXB];
  int jnt_type[MAXJ], jnt_qposadr[MAXJ], jnt_dofadr[MAXJ];
  int site_body[MAXS];
  float body_pos[MAXB * 3], body_quat[MAXB * 4], body_ipos[MAXB * 3], body_mass[MAXB];
  float tree_inv_mass[MAXB];  // 1 / subtree mass, indexed by root body id
  float jnt_axis[MAXJ * 3], jnt_pos[MAXJ * 3], qpos0[MAXQ];
  float site_pos[MAXS * 3], site_quat[MAXS * 4];
};

enum Specialised { SPEC_NONE = 0, SPEC_H1 = 1, SPEC_A3 = 2 };

}  // namespace om

struct OmModel {
  om::ModelTab host;
  om::ModelTab* dev = nullptr;
  int specialised = om::SPEC_NONE;
  int h1_variant = 0;   // UnitreeH1 model with fused playback / live-step kernels: 1 default, 2.. gen/h1v/list.h; else 0
  int device = 0;
  // om_model_bind_env_body_mass: body env_mass_body's mass is env_mass[env] (device, [env_mass_ld]) in every FK of this
  // model; env_mass_m0 = the other bodies' mass in its tree.  Null: the tables' mass.
  const float* env_mass = nullptr;
  int env_mass_body = -1, env_mass_ld = 0;
  float env_mass_m0 = 0.f;
};

#include "om_math.cuh"
