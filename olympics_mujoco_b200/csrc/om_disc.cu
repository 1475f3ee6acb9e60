// K4: GAIL / VAIL discriminator reward  r = -log(1 - sigmoid(D(s)) + 1e-8)
//   make_discrim_reward   imitation_lib/imitation/gail_TRPO.py:320-327   (discrim_output :315-318, VAIL vail_TRPO.py:18-21)
//   VariationalNet.forward imitation_lib/utils/networks.py:258-284 (reparameterize :21-24), DiscriminatorNetwork.forward
//   :208-234, FullyConnectedNetwork :94-158, Standardizer.forward :68-74; shapes examples/imitation_learning/utils.py:151-179
//   + confs.yaml:113-130:  VAIL 32 -relu-> 256 -relu-> 128 -> (mu, logvar)[128+128] -> z -> 1 ;  GAIL 32 -tanh-> 512 -tanh-> 256 -> 1.
//
// The only dense contraction on the hot path, so the only tcgen05 kernel.  One persistent CTA per SM owns 128-sample
// tiles: TMEM lane = sample, TMEM column = layer output, so producer thread t owns sample t in every epilogue and the
// final 128->1 / 256->1 head is a per-thread dot product.  Each layer is D[128 x N] += A[128 x K] B[N x K]^T on
// tcgen05.mma kind::tf32 (M=128, N<=256, K=8), streamed in K-chunks:
//   * A chunk (32 K-elements of the previous layer's activations): tcgen05.ld from TMEM -> bias + activation -> hi/lo
//     split -> st.shared in the canonical K-major no-swizzle UMMA layout [k/4][row][4] (16-byte rows contiguous:
//     conflict-free stores); 2-stage ring;
//   * B sub-chunk (16 K-elements of the weights): a pre-split image in exactly that layout, fetched by cp.async.bulk
//     (TMA, 1-D, several 8 KB pieces in flight) onto an mbarrier; 4-stage ring;
//   * warp-specialised: 4 producer/epilogue warps, one MMA-issuing thread, one copy-issuing thread, mbarriers only;
//   * fp32 fidelity: every product is evaluated as 3xTF32 (a_hi b_hi + a_lo b_hi + a_hi b_lo, hi = cvt.rna.tf32), fp32
//     accumulation in TMEM -- the north star's 1e-5 tolerance on rewards rules out plain TF32 (~1e-3).
#include <cstdlib>
#include <cstring>
#include <vector>

#include "om_common.cuh"

namespace om {

constexpr int DISC_IN = 32;        // observation size of the H1 discriminators
constexpr int KC = 32;             // K-chunk (elements) = 4 MMA k-steps of 8
constexpr int TILE = 128;          // samples per CTA tile = UMMA_M
constexpr int STAGE_A_BYTES = TILE * KC * 4 * 2;      // hi + lo
constexpr int DISC_MAX_PAR = 512 + 256 + 256 + 256 + 64;   // biases + head weights + standardiser, staged in shared memory

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
// Bounded spin: a mis-programmed descriptor or copy must surface as a launch failure, not as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  for (uint32_t spins = 0; !mbar_try_wait(bar, parity); ++spins)
    if (spins > (1u << 24)) __trap();
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// One lane of a CONVERGED warp.  The MMA-issuing code is entered through this rather than through `tid == ...`: ptxas then
// knows that a single thread executes it and emits the tcgen05.mma instructions back to back; behind a thread-index test it
// wraps every one of them in a five-instruction elect / vote loop, and at ~70 cycles of issue per 64-cycle MMA the issuing
// thread, not the tensor pipe, paced the N = 128 kernels.
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
               ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc), "r"(0u) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 consecutive TMEM columns of this thread's lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
               "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                 "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
                 "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
                 "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
               : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
// 16 consecutive TMEM columns of this thread's lane
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                 "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
               : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// cvt.rna.tf32.f32 (round to nearest, ties away from zero) as two integer-pipe instructions: the conversion instruction
// issues on the XU pipe (16 lanes / clk / SM), which ncu showed 62 % busy -- busier than the tensor pipe -- in
// disc_vail2_kernel (36 chunks x 16 conversions per sample).  Same bits as the host-side split_tf32.
__device__ __forceinline__ float tf32_rna(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u); }
// h[i] = relu(h[i] + bias[i]) for 16 consecutive parameters read from shared memory as four 128-bit loads (64-byte
// aligned; scalar loads made the bias reads a third of the kernel's shared-memory wavefronts)
__device__ __forceinline__ void bias_relu16(float (&h)[16], const float* bias) {
  const float4* q = reinterpret_cast<const float4*>(bias);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 t = q[i];
    h[4 * i] = fmaxf(h[4 * i] + t.x, 0.f); h[4 * i + 1] = fmaxf(h[4 * i + 1] + t.y, 0.f);
    h[4 * i + 2] = fmaxf(h[4 * i + 2] + t.z, 0.f); h[4 * i + 3] = fmaxf(h[4 * i + 3] + t.w, 0.f);
  }
}

// K-major, no-swizzle shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): 8-row x 16-byte core matrices,
// `lbo` = byte stride between the two 16-byte K slices of one MMA, `sbo` = byte stride between 8-row groups.
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) |
         (1ull << 46);      // version 1 (sm_100), base offset 0, layout type 0 = SWIZZLE_NONE
}
// cute::UMMA::InstrDescriptor: c F32 (1<<4), a/b TF32 (2<<7, 2<<10), both K-major, N>>3 at bit 17, M>>4 at bit 24
__host__ __device__ constexpr uint32_t idesc_tf32(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// ---------------------------------------------------------------- weight image (built on the host at create time)
// Chunk order = issue order of the kernel: for each 256-wide block nb of layer 1: [L1(nb)] then N1blk/32 chunks of layer 2;
// then (VAIL) N2/32 chunks of the [mu; logvar] layer.  Each chunk: hi image [8][rows][4] floats, then lo image.
struct DiscShape {
  int kind, n1, n2, z;          // kind 0 VAIL, 1 GAIL
  __host__ __device__ int n1_blocks() const { return n1 / 256; }
  __host__ __device__ int chunks_per_tile() const { return n1_blocks() * (1 + 8) + (kind == 0 ? n2 / KC : 0); }
};

struct DiscArgs {
  DiscShape sh;
  const float* image;           // pre-split weight chunks
  const float* params;          // b1[n1], b2[n2], (VAIL: bmu|blv [2z]), head weights wd[z or n2], bd
  const float* s; const float* mean; const float* stdv; const float* eps;
  float* reward; float* d_out; float* kl_out;
  int n, ld;
};

// Input width of the default kernels (disc_vail4_kernel, disc_reward_pg2_kernel).  IN = 0 is the build for the default
// H1 observation: 32 inputs, one 32-column input chunk, DiscArgs.  IN = 1 / 2 serve any other width n_in <= 32 IN: one /
// two input chunks, n_in given at run time in a derived argument type (so that the 32-input kernels keep their
// parameters), input rows at or beyond n_in never read and their standardised value 0 (the host image gives the padding
// columns of W1 zero weights).
constexpr int DISC_MAX_IN = 64;
struct DiscArgsIn : DiscArgs { int n_in; };
template <int IN> struct DiscInput {
  using Args = DiscArgsIn;
  static constexpr int NCH = IN;                // 32-column input chunks
  __device__ static int n_in(const Args& a) { return a.n_in; }
};
template <> struct DiscInput<0> {
  using Args = DiscArgs;
  static constexpr int NCH = 1;
  __device__ static int n_in(const Args&) { return DISC_IN; }
};

enum { ACT_RELU = 0, ACT_TANH = 1 };
template <int ACT> __device__ __forceinline__ float act(float x) { return ACT == ACT_RELU ? fmaxf(x, 0.f) : tanhf(x); }

// split 32 activations of this thread's sample into the hi / lo A-stage images
__device__ __forceinline__ void store_a_chunk(uint8_t* stage, int row, const float (&a)[32]) {
  float4* hi = reinterpret_cast<float4*>(stage) + row;                       // [kc][128 rows] float4
  float4* lo = reinterpret_cast<float4*>(stage + TILE * KC * 4) + row;
#pragma unroll
  for (int kc = 0; kc < 8; ++kc) {
    float4 h, l;
    h.x = tf32_rna(a[4 * kc]); h.y = tf32_rna(a[4 * kc + 1]); h.z = tf32_rna(a[4 * kc + 2]); h.w = tf32_rna(a[4 * kc + 3]);
    l.x = a[4 * kc] - h.x; l.y = a[4 * kc + 1] - h.y; l.z = a[4 * kc + 2] - h.z; l.w = a[4 * kc + 3] - h.w;
    hi[kc * TILE] = h;
    lo[kc * TILE] = l;
  }
}

// Warp roles (192 threads): warps 0-3 = producers / epilogue (thread t owns sample t = TMEM lane t), warp 4 lane 0 =
// MMA issuer, warp 5 lane 0 = weight-copy (TMA) issuer.  Rings: A 2 stages x 32 K-elements, B 4 stages x 16 K-elements.
//   a_full[2]  producers -> issuer   (128 arrivals)        a_free[2]  tcgen05.commit -> producers (stage reuse AND
//   b_full[4]  bulk copy -> issuer   (transaction bytes)              "all MMAs up to this chunk are complete")
//   b_free[4]  tcgen05.commit -> copy issuer
// All three roles walk the same static chunk schedule; ga / qb count A chunks / B sub-chunks since kernel start, so
// stage = counter mod ring and the mbarrier parity = (counter / ring) & 1.
constexpr int KB = 16;                                 // K elements per B sub-chunk (2 MMA k-steps)
constexpr int NSB = 4;
constexpr int STAGE_B2_BYTES = 256 * KB * 4 * 2;       // 32 KB
constexpr int COPY_PIECE = 8192;                       // several bulk copies in flight per sub-chunk

template <int N1, int N2, bool VAIL, bool KL>
__global__ void __launch_bounds__(192, 1) disc_reward_kernel(DiscArgs a) {
  constexpr int ACT = VAIL ? ACT_RELU : ACT_TANH;
  constexpr int NB1 = N1 / 256;                 // 256-wide column blocks of layer 1
  constexpr int Z = 128;
  constexpr int N3 = 2 * Z;
  constexpr int D1_COL = 0, D2_COL = 256, D3_COL = 0;
  constexpr int HEAD_K = VAIL ? Z : N2;
  static_assert(N1 % 256 == 0 && N2 % 32 == 0 && N2 <= 256, "unsupported discriminator shape");
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* stA = smem;                                            // 2 x STAGE_A_BYTES
  uint8_t* stB = smem + 2 * STAGE_A_BYTES;                        // NSB x STAGE_B2_BYTES
  float* par = reinterpret_cast<float*>(stB + NSB * STAGE_B2_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(par + DISC_MAX_PAR + 4);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);
  const float* b1 = par;
  const float* b2 = par + N1;
  const float* b3 = par + N1 + N2;                          // VAIL: bmu | blv
  const float* wd = par + N1 + N2 + (VAIL ? N3 : 0);
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t bar0 = smem_u32(bars);
  auto a_full = [&](int s_) { return bar0 + 8u * s_; };
  auto a_free = [&](int s_) { return bar0 + 8u * (2 + s_); };
  auto b_full = [&](int s_) { return bar0 + 8u * (4 + s_); };
  auto b_free = [&](int s_) { return bar0 + 8u * (8 + s_); };

  constexpr int NPAR = N1 + N2 + (VAIL ? N3 : 0) + HEAD_K + 1;
  for (int i = tid; i < NPAR; i += 192) par[i] = a.params[i];
  float* s_mean = par + DISC_MAX_PAR - 2 * DISC_IN;          // Standardizer snapshot: mean, 1 / std
  float* s_inv = s_mean + DISC_IN;
  if (tid < DISC_IN) { s_mean[tid] = a.mean[tid]; s_inv[tid] = 1.0f / a.stdv[tid]; }
  if (tid == 0) {
    for (int s_ = 0; s_ < 2; ++s_) { mbar_init(a_full(s_), 128); mbar_init(a_free(s_), 1); }
    for (int s_ = 0; s_ < NSB; ++s_) { mbar_init(b_full(s_), 1); mbar_init(b_free(s_), 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int ntiles = (a.n + TILE - 1) / TILE;

  if (warp == 5) {
    // ===================================================== weight-copy issuer
    if (tid == 160) {
      int qb = 0;
      auto copy_chunk = [&](const float*& img, int rows) {                 // one A chunk = two B sub-chunks
        for (int hb = 0; hb < 2; ++hb, ++qb) {
          const int sb = qb & (NSB - 1);
          if (qb >= NSB) mbar_wait(b_free(sb), (uint32_t)((qb / NSB) - 1) & 1u);
          const uint32_t bytes = (uint32_t)rows * KB * 4 * 2;
          mbar_expect_tx(b_full(sb), bytes);
          const uint32_t dst = smem_u32(stB + sb * STAGE_B2_BYTES);
          for (uint32_t off = 0; off < bytes; off += COPY_PIECE)
            bulk_g2s(dst + off, reinterpret_cast<const uint8_t*>(img) + off, COPY_PIECE, b_full(sb));
          img += bytes / 4;
        }
      };
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const float* img = a.image;
        for (int nb = 0; nb < NB1; ++nb) {
          copy_chunk(img, 256);
          for (int c = 0; c < 8; ++c) copy_chunk(img, N2);
        }
        if (VAIL)
          for (int c = 0; c < N2 / KC; ++c) copy_chunk(img, N3);
      }
    }
  } else if (warp == 4) {
    // ===================================================== MMA issuer
    if (elect_one_sync()) {
      int ga = 0, qb = 0;
      auto mma_chunk = [&](int rows, uint32_t d_col, bool first) {
        const int sa = ga & 1;
        mbar_wait(a_full(sa), (uint32_t)(ga >> 1) & 1u);
        tc_fence_after();
        const uint32_t a_hi = smem_u32(stA + sa * STAGE_A_BYTES), a_lo = a_hi + TILE * KC * 4;
        const uint32_t a_lbo = TILE * 16, b_lbo = (uint32_t)rows * 16, sbo = 128;
        const uint32_t idesc = idesc_tf32(TILE, rows);
        for (int hb = 0; hb < 2; ++hb, ++qb) {
          const int sb = qb & (NSB - 1);
          mbar_wait(b_full(sb), (uint32_t)(qb / NSB) & 1u);
          const uint32_t b_hi = smem_u32(stB + sb * STAGE_B2_BYTES), b_lo = b_hi + (uint32_t)rows * KB * 4;
#pragma unroll
          for (int j = 0; j < KB / 8; ++j) {
            const uint32_t ao = (uint32_t)(hb * (KB / 8) + j) * 2 * a_lbo, bo = (uint32_t)j * 2 * b_lbo;
            const uint64_t dah = smem_desc(a_hi + ao, a_lbo, sbo), dal = smem_desc(a_lo + ao, a_lbo, sbo);
            const uint64_t dbh = smem_desc(b_hi + bo, b_lbo, sbo), dbl = smem_desc(b_lo + bo, b_lbo, sbo);
            umma_tf32(tmem + d_col, dal, dbh, idesc, (first && hb == 0 && j == 0) ? 0u : 1u);     // small terms first
            umma_tf32(tmem + d_col, dah, dbl, idesc, 1u);
            umma_tf32(tmem + d_col, dah, dbh, idesc, 1u);
          }
          umma_commit(b_free(sb));
        }
        umma_commit(a_free(sa));
        ++ga;
      };
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        for (int nb = 0; nb < NB1; ++nb) {
          mma_chunk(256, D1_COL, true);
          for (int c = 0; c < 8; ++c) mma_chunk(N2, D2_COL, nb == 0 && c == 0);
        }
        if (VAIL)
          for (int c = 0; c < N2 / KC; ++c) mma_chunk(N3, D3_COL, c == 0);
      }
    }
  } else {
    // ===================================================== producers / epilogue (128 threads)
    const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);     // this warp's 32 TMEM lanes
    const float bd = par[NPAR - 1];
    int ga = 0;
    // commit of A chunk h has completed  <=>  phase (h >> 1) of a_free[h & 1] has completed
    auto wait_chunk = [&](int h) {
      if (h >= 0) {
        mbar_wait(a_free(h & 1), (uint32_t)(h >> 1) & 1u);
        tc_fence_after();
      }
    };
    auto put_chunk = [&](const float (&act_in)[32]) {
      wait_chunk(ga - 2);                                                // the stage is free
      store_a_chunk(stA + (ga & 1) * STAGE_A_BYTES, tid, act_in);
      fence_proxy_async();                                               // generic-proxy stores -> async proxy (UMMA)
      tc_fence_before();                                                 // earlier tcgen05.ld before later MMAs
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a_full(ga & 1)) : "memory");
      ++ga;
    };
    // raw observation row of this thread's sample; the NEXT tile's row is requested while the current tile computes
    auto load_row = [&](int tile_, float (&raw)[DISC_IN]) {
      const int env_ = tile_ * TILE + tid;
#pragma unroll
      for (int k = 0; k < DISC_IN; ++k) raw[k] = (tile_ < ntiles && env_ < a.n) ? a.s[(size_t)k * a.ld + env_] : 0.f;
    };
    float xn[DISC_IN];
    load_row(blockIdx.x, xn);
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      const int env = tile * TILE + tid;
      const bool live = env < a.n;
      // ---- standardised input row (Standardizer.forward networks.py:73-74 with a frozen snapshot)
      float x[DISC_IN];
#pragma unroll
      for (int k = 0; k < DISC_IN; ++k) x[k] = live ? (xn[k] - s_mean[k]) * s_inv[k] : 0.f;
      load_row(tile + gridDim.x, xn);
#pragma unroll 1
      for (int nb = 0; nb < NB1; ++nb) {
        put_chunk(x);                                                    // layer 1, column block nb
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {                                    // layer 2, K-chunks fed by this block
          if (c == 0) wait_chunk(ga - 1);                                // D1 block complete
          float h[32];
          tmem_ld32(lane_addr + D1_COL + c * KC, h);
#pragma unroll
          for (int i = 0; i < 32; ++i) h[i] = act<ACT>(h[i] + b1[nb * 256 + c * KC + i]);
          put_chunk(h);
        }
      }
      float dval = 0.f, klv = 0.f;
      if (VAIL) {
#pragma unroll 1
        for (int c = 0; c < N2 / KC; ++c) {                              // [mu; logvar] layer
          if (c == 0) wait_chunk(ga - 1);                                // D2 complete
          float h[32];
          tmem_ld32(lane_addr + D2_COL + c * KC, h);
#pragma unroll
          for (int i = 0; i < 32; ++i) h[i] = act<ACT>(h[i] + b2[c * KC + i]);
          put_chunk(h);
        }
        // z = mu + exp(logvar / 2) * eps (networks.py:21-24), d = wd . z + bd.  The noise rows are requested one block
        // ahead so that their latency hides behind the last MMAs / the TMEM loads.
        auto load_eps = [&](int c, float (&e)[32]) {
#pragma unroll
          for (int i = 0; i < 32; ++i) e[i] = (a.eps && live) ? a.eps[(size_t)(c * 32 + i) * a.ld + env] : 0.f;
        };
        auto head_block = [&](int c, const float (&e)[32]) {
          float mu[32], lv[32];
          tmem_ld32(lane_addr + D3_COL + c * 32, mu);
          tmem_ld32(lane_addr + D3_COL + Z + c * 32, lv);
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int j = c * 32 + i;
            const float m = mu[i] + b3[j], l = lv[i] + b3[Z + j], sd = expf(0.5f * l);
            dval = fmaf(wd[j], fmaf(sd, e[i], m), dval);
            if (KL) klv += fmaf(m, m, fmaf(sd, sd, -l)) - 1.f;       // VDBLoss.kl_divergence, math.py:83-86
          }
        };
        float e0[32], e1[32];
        load_eps(0, e0);
        wait_chunk(ga - 1);
        static_assert(Z == 128, "head unrolled for z = 128");
        load_eps(1, e1); head_block(0, e0);
        load_eps(2, e0); head_block(1, e1);
        load_eps(3, e1); head_block(2, e0);
        head_block(3, e1);
      } else {
        wait_chunk(ga - 1);
#pragma unroll 1
        for (int c = 0; c < N2 / 32; ++c) {
          float h[32];
          tmem_ld32(lane_addr + D2_COL + c * 32, h);
#pragma unroll
          for (int i = 0; i < 32; ++i) dval = fmaf(wd[c * 32 + i], act<ACT>(h[i] + b2[c * 32 + i]), dval);
        }
      }
      dval += bd;
      if (live) {
        // 1 - sigmoid(d) evaluated as sigmoid(-d): no cancellation for large d (gail_TRPO.py:326-327)
        const float one_minus_p = 1.f / (1.f + expf(dval));
        if (a.reward) a.reward[env] = -logf(one_minus_p + 1e-8f);
        if (a.d_out) a.d_out[env] = dval;
        if (VAIL && KL) a.kl_out[env] = 0.5f * klv;
      }
      // the next tile's layer-1 MMA overwrites the columns read above: put_chunk orders these loads before its arrive
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

// ---------------------------------------------------------------- two producer warpgroups per CTA
// Stall sampling of the kernel above puts the tensor pipe behind the PRODUCERS: one thread per sample turns 32 TMEM
// columns into a hi / lo shared-memory chunk in ~250 instructions while the three MMAs of that chunk take less.  Here
// eight producer warps share a tile: thread t and thread t + 128 own the same sample (TMEM lane t mod 128 -- a warp may
// touch the 32 lanes given by its index mod 4) and each handles 16 of the 32 columns of every chunk, half of the input
// row, half of the latent dimensions / head weights; the two partial head sums meet in shared memory behind one named
// barrier.  Same rings, same schedule, same issuer code as above; 320 threads (warp 8 = MMA issuer, warp 9 = copies).
__device__ __forceinline__ void store_a_half(uint8_t* stage, int row, int half, const float (&a)[16]) {
  float4* hi = reinterpret_cast<float4*>(stage) + row;                       // [kc][128 rows] float4
  float4* lo = reinterpret_cast<float4*>(stage + TILE * KC * 4) + row;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int kc = 4 * half + j;
    float4 h, l;
    h.x = tf32_rna(a[4 * j]); h.y = tf32_rna(a[4 * j + 1]); h.z = tf32_rna(a[4 * j + 2]); h.w = tf32_rna(a[4 * j + 3]);
    l.x = a[4 * j] - h.x; l.y = a[4 * j + 1] - h.y; l.z = a[4 * j + 2] - h.z; l.w = a[4 * j + 3] - h.w;
    hi[kc * TILE] = h;
    lo[kc * TILE] = l;
  }
}

template <int N1, int N2, bool VAIL, bool KL, int IN = 0>
__global__ void __launch_bounds__(320, 1) disc_reward_pg2_kernel(typename DiscInput<IN>::Args a) {
  constexpr int ACT = VAIL ? ACT_RELU : ACT_TANH;
  constexpr int NB1 = N1 / 256;
  constexpr int Z = 128;
  constexpr int N3 = 2 * Z;
  constexpr int D1_COL = 0, D2_COL = 256, D3_COL = 0;
  constexpr int HEAD_K = VAIL ? Z : N2;
  constexpr int NPROD = 256;
  constexpr int NCH = DiscInput<IN>::NCH, KIN = KC * NCH;            // input chunks, padded input width
  static_assert(N1 % 256 == 0 && N2 % 32 == 0 && N2 <= 256, "unsupported discriminator shape");
  static_assert(DISC_MAX_PAR - 2 * KIN >= N1 + N2 + (VAIL ? N3 : 0) + HEAD_K + 1, "standardiser slots overlap the parameters");
  const int nin = DiscInput<IN>::n_in(a);
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* stA = smem;
  uint8_t* stB = smem + 2 * STAGE_A_BYTES;
  float* par = reinterpret_cast<float*>(stB + NSB * STAGE_B2_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(par + DISC_MAX_PAR + 4);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 12);
  float* red = reinterpret_cast<float*>(tmem_slot + 4);                      // [2][128]: partial logit, partial KL of half 1
  const float* b1 = par;
  const float* b2 = par + N1;
  const float* b3 = par + N1 + N2;
  const float* wd = par + N1 + N2 + (VAIL ? N3 : 0);
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t bar0 = smem_u32(bars);
  auto a_full = [&](int s_) { return bar0 + 8u * s_; };
  auto a_free = [&](int s_) { return bar0 + 8u * (2 + s_); };
  auto b_full = [&](int s_) { return bar0 + 8u * (4 + s_); };
  auto b_free = [&](int s_) { return bar0 + 8u * (8 + s_); };

  constexpr int NPAR = N1 + N2 + (VAIL ? N3 : 0) + HEAD_K + 1;
  for (int i = tid; i < NPAR; i += 320) par[i] = a.params[i];
  float* s_mean = par + DISC_MAX_PAR - 2 * KIN;
  float* s_inv = s_mean + KIN;
  if (tid < KIN) {
    const bool in_ = IN == 0 || tid < nin;                            // padding columns: mean 0, 1 / std 0
    s_mean[tid] = in_ ? a.mean[tid] : 0.f;
    s_inv[tid] = in_ ? 1.0f / a.stdv[tid] : 0.f;
  }
  if (tid == 0) {
    for (int s_ = 0; s_ < 2; ++s_) { mbar_init(a_full(s_), NPROD); mbar_init(a_free(s_), 1); }
    for (int s_ = 0; s_ < NSB; ++s_) { mbar_init(b_full(s_), 1); mbar_init(b_free(s_), 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int ntiles = (a.n + TILE - 1) / TILE;

  if (warp == 9) {
    // ===================================================== weight-copy issuer (as in disc_reward_kernel)
    if (tid == 288) {
      int qb = 0;
      auto copy_chunk = [&](const float*& img, int rows) {
        for (int hb = 0; hb < 2; ++hb, ++qb) {
          const int sb = qb & (NSB - 1);
          if (qb >= NSB) mbar_wait(b_free(sb), (uint32_t)((qb / NSB) - 1) & 1u);
          const uint32_t bytes = (uint32_t)rows * KB * 4 * 2;
          mbar_expect_tx(b_full(sb), bytes);
          const uint32_t dst = smem_u32(stB + sb * STAGE_B2_BYTES);
          for (uint32_t off = 0; off < bytes; off += COPY_PIECE)
            bulk_g2s(dst + off, reinterpret_cast<const uint8_t*>(img) + off, COPY_PIECE, b_full(sb));
          img += bytes / 4;
        }
      };
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const float* img = a.image;
        for (int nb = 0; nb < NB1; ++nb) {
#pragma unroll
          for (int ch = 0; ch < NCH; ++ch) copy_chunk(img, 256);
          for (int c = 0; c < 8; ++c) copy_chunk(img, N2);
        }
        if (VAIL)
          for (int c = 0; c < N2 / KC; ++c) copy_chunk(img, N3);
      }
    }
  } else if (warp == 8) {
    // ===================================================== MMA issuer (as in disc_reward_kernel)
    if (elect_one_sync()) {
      int ga = 0, qb = 0;
      auto mma_chunk = [&](int rows, uint32_t d_col, bool first) {
        const int sa = ga & 1;
        mbar_wait(a_full(sa), (uint32_t)(ga >> 1) & 1u);
        tc_fence_after();
        const uint32_t a_hi = smem_u32(stA + sa * STAGE_A_BYTES), a_lo = a_hi + TILE * KC * 4;
        const uint32_t a_lbo = TILE * 16, b_lbo = (uint32_t)rows * 16, sbo = 128;
        const uint32_t idesc = idesc_tf32(TILE, rows);
        for (int hb = 0; hb < 2; ++hb, ++qb) {
          const int sb = qb & (NSB - 1);
          mbar_wait(b_full(sb), (uint32_t)(qb / NSB) & 1u);
          const uint32_t b_hi = smem_u32(stB + sb * STAGE_B2_BYTES), b_lo = b_hi + (uint32_t)rows * KB * 4;
#pragma unroll
          for (int j = 0; j < KB / 8; ++j) {
            const uint32_t ao = (uint32_t)(hb * (KB / 8) + j) * 2 * a_lbo, bo = (uint32_t)j * 2 * b_lbo;
            const uint64_t dah = smem_desc(a_hi + ao, a_lbo, sbo), dal = smem_desc(a_lo + ao, a_lbo, sbo);
            const uint64_t dbh = smem_desc(b_hi + bo, b_lbo, sbo), dbl = smem_desc(b_lo + bo, b_lbo, sbo);
            umma_tf32(tmem + d_col, dal, dbh, idesc, (first && hb == 0 && j == 0) ? 0u : 1u);
            umma_tf32(tmem + d_col, dah, dbl, idesc, 1u);
            umma_tf32(tmem + d_col, dah, dbh, idesc, 1u);
          }
          umma_commit(b_free(sb));
        }
        umma_commit(a_free(sa));
        ++ga;
      };
      for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        for (int nb = 0; nb < NB1; ++nb) {
#pragma unroll
          for (int ch = 0; ch < NCH; ++ch) mma_chunk(256, D1_COL, ch == 0);
          for (int c = 0; c < 8; ++c) mma_chunk(N2, D2_COL, nb == 0 && c == 0);
        }
        if (VAIL)
          for (int c = 0; c < N2 / KC; ++c) mma_chunk(N3, D3_COL, c == 0);
      }
    }
  } else {
    // ===================================================== producers / epilogue (256 threads, two per sample)
    const int row = tid & 127, half = tid >> 7;
    const uint32_t lane_addr = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const float bd = par[NPAR - 1];
    int ga = 0;
    auto wait_chunk = [&](int h) {
      if (h >= 0) {
        mbar_wait(a_free(h & 1), (uint32_t)(h >> 1) & 1u);
        tc_fence_after();
      }
    };
    auto put_half = [&](const float (&act_in)[16]) {
      wait_chunk(ga - 2);
      store_a_half(stA + (ga & 1) * STAGE_A_BYTES, row, half, act_in);
      fence_proxy_async();
      tc_fence_before();
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a_full(ga & 1)) : "memory");
      ++ga;
    };
    // this thread's 16 columns of every input chunk: input 32 ch + 16 half + k at [ch][k]
    auto load_row = [&](int tile_, float (&raw)[NCH][16]) {
      const int env_ = tile_ * TILE + row;
#pragma unroll
      for (int j = 0; j < 16 * NCH; ++j) {
        const int r = KC * (j / 16) + 16 * half + j % 16;
        raw[j / 16][j % 16] = (tile_ < ntiles && env_ < a.n && (IN == 0 || r < nin)) ? a.s[(size_t)r * a.ld + env_] : 0.f;
      }
    };
    float xn[NCH][16];
    load_row(blockIdx.x, xn);
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      const int env = tile * TILE + row;
      const bool live = env < a.n;
      float x[NCH][16];
#pragma unroll
      for (int j = 0; j < 16 * NCH; ++j) {
        const int r = KC * (j / 16) + 16 * half + j % 16;
        x[j / 16][j % 16] = live ? (xn[j / 16][j % 16] - s_mean[r]) * s_inv[r] : 0.f;
      }
      load_row(tile + gridDim.x, xn);
#pragma unroll 1
      for (int nb = 0; nb < NB1; ++nb) {
        put_half(x[0]);                                                  // layer 1, column block nb
        if constexpr (NCH == 2) put_half(x[1]);
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {                                    // layer 2, K-chunks fed by this block
          if (c == 0) wait_chunk(ga - 1);
          float h[16];
          tmem_ld16(lane_addr + D1_COL + c * KC + 16 * half, h);
#pragma unroll
          for (int i = 0; i < 16; ++i) h[i] = act<ACT>(h[i] + b1[nb * 256 + c * KC + 16 * half + i]);
          put_half(h);
        }
      }
      float dval = 0.f, klv = 0.f;
      if (VAIL) {
#pragma unroll 1
        for (int c = 0; c < N2 / KC; ++c) {                              // [mu; logvar] layer
          if (c == 0) wait_chunk(ga - 1);
          float h[16];
          tmem_ld16(lane_addr + D2_COL + c * KC + 16 * half, h);
#pragma unroll
          for (int i = 0; i < 16; ++i) h[i] = act<ACT>(h[i] + b2[c * KC + 16 * half + i]);
          put_half(h);
        }
        // this half's 64 latent dimensions: z = mu + exp(logvar / 2) * eps, d += wd . z
        static_assert(Z == 128, "head unrolled for z = 128");
        float e0[32], e1[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          e0[i] = (a.eps && live) ? a.eps[(size_t)(64 * half + i) * a.ld + env] : 0.f;
          e1[i] = (a.eps && live) ? a.eps[(size_t)(64 * half + 32 + i) * a.ld + env] : 0.f;
        }
        wait_chunk(ga - 1);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          float mu[32], lv[32];
          tmem_ld32(lane_addr + D3_COL + 64 * half + 32 * q, mu);
          tmem_ld32(lane_addr + D3_COL + Z + 64 * half + 32 * q, lv);
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int j = 64 * half + 32 * q + i;
            const float m = mu[i] + b3[j], l = lv[i] + b3[Z + j], sd = expf(0.5f * l);
            dval = fmaf(wd[j], fmaf(sd, q == 0 ? e0[i] : e1[i], m), dval);
            if (KL) klv += fmaf(m, m, fmaf(sd, sd, -l)) - 1.f;
          }
        }
      } else {
        wait_chunk(ga - 1);
#pragma unroll 1
        for (int c = 0; c < N2 / 64; ++c) {
          float h[32];
          tmem_ld32(lane_addr + D2_COL + (N2 / 2) * half + c * 32, h);
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int j = (N2 / 2) * half + c * 32 + i;
            dval = fmaf(wd[j], act<ACT>(h[i] + b2[j]), dval);
          }
        }
      }
      // the two halves of a sample meet: half 1 hands its partial sums to half 0
      if (half == 1) { red[row] = dval; red[128 + row] = klv; }
      tc_fence_before();
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (half == 0 && live) {
        dval += red[row] + bd;
        const float one_minus_p = 1.f / (1.f + expf(dval));
        if (a.reward) a.reward[env] = -logf(one_minus_p + 1e-8f);
        if (a.d_out) a.d_out[env] = dval;
        if (VAIL && KL) a.kl_out[env] = 0.5f * (klv + red[128 + row]);
      }
      asm volatile("bar.sync 2, 256;" ::: "memory");                     // red[] may be rewritten by the next tile
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

// ---------------------------------------------------------------- VAIL, two CTAs per SM
// The single-CTA kernel above leaves the tensor pipe idle at every layer boundary (layer l+1's first A chunk needs
// layer l's complete accumulator) and during the head.  This variant halves every per-CTA resource -- 256 TMEM
// columns, 100 KB of shared memory, <= 168 registers -- so that TWO CTAs share an SM and one CTA's boundaries and heads
// hide under the other's MMAs.  To fit 256 TMEM columns every MMA is N = 128:
//   layer 1 in two 128-column blocks (DA = cols 0-127), each feeding 8 K-chunks of layer 2 (DB = cols 128-255);
//   the [mu; logvar] layer in two 128-row blocks whose rows are INTERLEAVED on the host (block h = mu[64h..64h+63] then
//   logvar[64h..64h+63]) into DA again, so that the head consumes 64 latent dimensions per block.
// One ring of 3 stages; a stage = 16 K-elements of A (hi, lo) and of B (hi, lo), 32 KB.
constexpr int V2_KC = 16, V2_NS = 3, V2_ROWS = 128;
constexpr int V2_A_BYTES = TILE * V2_KC * 4;           // one of hi / lo: 8 KB
constexpr int V2_B_BYTES = V2_ROWS * V2_KC * 4;        // 8 KB
constexpr int V2_STAGE_BYTES = 2 * V2_A_BYTES + 2 * V2_B_BYTES;
constexpr int V2_NPAR = 256 + 128 + 256 + 128 + 1;     // b1, b2, b3 (interleaved like the rows), wd, bd
constexpr int V2_CHUNKS_PER_TILE = 2 * (2 + 8) + 2 * 8;

__device__ __forceinline__ void store_a16(uint8_t* stage, int row, const float (&a)[16]) {
  float4* hi = reinterpret_cast<float4*>(stage) + row;                       // [kc][128 rows] float4
  float4* lo = reinterpret_cast<float4*>(stage + V2_A_BYTES) + row;
#pragma unroll
  for (int kc = 0; kc < 4; ++kc) {
    float4 h, l;
    h.x = tf32_rna(a[4 * kc]); h.y = tf32_rna(a[4 * kc + 1]); h.z = tf32_rna(a[4 * kc + 2]); h.w = tf32_rna(a[4 * kc + 3]);
    l.x = a[4 * kc] - h.x; l.y = a[4 * kc + 1] - h.y; l.z = a[4 * kc + 2] - h.z; l.w = a[4 * kc + 3] - h.w;
    hi[kc * TILE] = h;
    lo[kc * TILE] = l;
  }
}

template <bool KL>
__global__ void __launch_bounds__(192, 2) disc_vail2_kernel(DiscArgs a) {
  constexpr int Z = 128, DA = 0, DB = 128;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* ring = smem;
  float* par = reinterpret_cast<float*>(smem + V2_NS * V2_STAGE_BYTES);
  float* s_mean = par + V2_NPAR + 3;
  float* s_inv = s_mean + DISC_IN;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_inv + DISC_IN);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * V2_NS);
  const float* b1 = par;
  const float* b2 = par + 256;
  const float* b3 = par + 384;            // per 128-row block h: [bmu[64h..], blv[64h..]]
  const float* wd = par + 640;
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t bar0 = smem_u32(bars);
  auto a_full = [&](int s_) { return bar0 + 8u * s_; };
  auto b_full = [&](int s_) { return bar0 + 8u * (V2_NS + s_); };
  auto s_free = [&](int s_) { return bar0 + 8u * (2 * V2_NS + s_); };

  for (int i = tid; i < V2_NPAR; i += 192) par[i] = a.params[i];
  if (tid < DISC_IN) { s_mean[tid] = a.mean[tid]; s_inv[tid] = 1.0f / a.stdv[tid]; }
  if (tid == 0) {
    for (int s_ = 0; s_ < V2_NS; ++s_) { mbar_init(a_full(s_), 128); mbar_init(b_full(s_), 1); mbar_init(s_free(s_), 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int ntiles = (a.n + TILE - 1) / TILE;
  int my_tiles = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) ++my_tiles;
  const int total_chunks = my_tiles * V2_CHUNKS_PER_TILE;

  if (warp == 5) {
    // ===================================================== weight-copy issuer: the image repeats every tile
    if (tid == 160) {
      for (int g = 0; g < total_chunks; ++g) {
        const int st = g % V2_NS, use = g / V2_NS;
        if (use > 0) mbar_wait(s_free(st), (uint32_t)(use - 1) & 1u);
        mbar_expect_tx(b_full(st), 2 * V2_B_BYTES);
        const uint8_t* src = reinterpret_cast<const uint8_t*>(a.image) + (size_t)(g % V2_CHUNKS_PER_TILE) * 2 * V2_B_BYTES;
        const uint32_t dst = smem_u32(ring + st * V2_STAGE_BYTES + 2 * V2_A_BYTES);
        bulk_g2s(dst, src, V2_B_BYTES, b_full(st));
        bulk_g2s(dst + V2_B_BYTES, src + V2_B_BYTES, V2_B_BYTES, b_full(st));
      }
    }
  } else if (warp == 4) {
    // ===================================================== MMA issuer
    if (elect_one_sync()) {
      const uint32_t idesc = idesc_tf32(TILE, V2_ROWS);
      const uint32_t lbo = TILE * 16, sbo = 128;                  // A and B both have 128 rows
      for (int g = 0; g < total_chunks; ++g) {
        const int st = g % V2_NS, use = g / V2_NS, c = g % V2_CHUNKS_PER_TILE;
        // position in the tile schedule -> accumulator and "first" flag
        uint32_t d_col;
        bool first;
        if (c < 20) {
          const int r = c % 10;                                   // 0,1: layer 1 of this block; 2..9: layer 2
          d_col = r < 2 ? DA : DB;
          first = r < 2 ? (r == 0) : (c == 2);                    // layer 2 accumulates over both blocks
        } else {
          d_col = DA;
          first = ((c - 20) % 8) == 0;
        }
        mbar_wait(a_full(st), (uint32_t)use & 1u);
        mbar_wait(b_full(st), (uint32_t)use & 1u);
        tc_fence_after();
        const uint32_t a_hi = smem_u32(ring + st * V2_STAGE_BYTES), a_lo = a_hi + V2_A_BYTES;
        const uint32_t b_hi = a_hi + 2 * V2_A_BYTES, b_lo = b_hi + V2_B_BYTES;
#pragma unroll
        for (int j = 0; j < V2_KC / 8; ++j) {
          const uint32_t o = (uint32_t)j * 2 * lbo;
          const uint64_t dah = smem_desc(a_hi + o, lbo, sbo), dal = smem_desc(a_lo + o, lbo, sbo);
          const uint64_t dbh = smem_desc(b_hi + o, lbo, sbo), dbl = smem_desc(b_lo + o, lbo, sbo);
          umma_tf32(tmem + d_col, dal, dbh, idesc, (first && j == 0) ? 0u : 1u);
          umma_tf32(tmem + d_col, dah, dbl, idesc, 1u);
          umma_tf32(tmem + d_col, dah, dbh, idesc, 1u);
        }
        umma_commit(s_free(st));
      }
    }
  } else {
    // ===================================================== producers / epilogue (128 threads)
    const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
    const float bd = par[V2_NPAR - 1];
    int g = 0;
    auto wait_chunk = [&](int h) {                         // all MMAs up to and including chunk h are complete
      if (h >= 0) {
        mbar_wait(s_free(h % V2_NS), (uint32_t)(h / V2_NS) & 1u);
        tc_fence_after();
      }
    };
    auto put = [&](const float (&act_in)[16]) {
      wait_chunk(g - V2_NS);
      store_a16(ring + (g % V2_NS) * V2_STAGE_BYTES, tid, act_in);
      fence_proxy_async();
      tc_fence_before();
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a_full(g % V2_NS)) : "memory");
      ++g;
    };
    auto load_row = [&](int tile_, float (&raw)[DISC_IN]) {
      const int env_ = tile_ * TILE + tid;
#pragma unroll
      for (int k = 0; k < DISC_IN; ++k) raw[k] = (tile_ < ntiles && env_ < a.n) ? a.s[(size_t)k * a.ld + env_] : 0.f;
    };
    float xn[DISC_IN];
    load_row(blockIdx.x, xn);
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      const int env = tile * TILE + tid;
      const bool live = env < a.n;
      float x[DISC_IN];
#pragma unroll
      for (int k = 0; k < DISC_IN; ++k) x[k] = live ? (xn[k] - s_mean[k]) * s_inv[k] : 0.f;
      load_row(tile + gridDim.x, xn);
#pragma unroll 1
      for (int blk = 0; blk < 2; ++blk) {
        {
          float h0[16], h1[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) { h0[i] = x[i]; h1[i] = x[16 + i]; }
          put(h0);
          put(h1);
        }
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {
          if (c == 0) wait_chunk(g - 1);                                  // this layer-1 block is complete
          float h[16];
          tmem_ld16(lane_addr + DA + c * V2_KC, h);
          bias_relu16(h, b1 + blk * 128 + c * V2_KC);
          put(h);
        }
      }
      float dval = 0.f, klv = 0.f;
#pragma unroll 1
      for (int hb = 0; hb < 2; ++hb) {
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {
          if (c == 0 && hb == 0) wait_chunk(g - 1);                       // layer 2 complete
          float h[16];
          tmem_ld16(lane_addr + DB + c * V2_KC, h);
          bias_relu16(h, b2 + c * V2_KC);
          put(h);
        }
        // head over latent dimensions 64 hb .. 64 hb + 63: z = mu + exp(logvar / 2) eps, d += wd . z
        float e0[32], e1[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          e0[i] = (a.eps && live) ? a.eps[(size_t)(64 * hb + i) * a.ld + env] : 0.f;
          e1[i] = (a.eps && live) ? a.eps[(size_t)(64 * hb + 32 + i) * a.ld + env] : 0.f;
        }
        wait_chunk(g - 1);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          float mu[32], lv[32];
          tmem_ld32(lane_addr + DA + q * 32, mu);
          tmem_ld32(lane_addr + DA + 64 + q * 32, lv);
          const float4* bm4 = reinterpret_cast<const float4*>(b3 + 128 * hb + 32 * q);
          const float4* bl4 = reinterpret_cast<const float4*>(b3 + 128 * hb + 64 + 32 * q);
          const float4* wv4 = reinterpret_cast<const float4*>(wd + 64 * hb + 32 * q);
#pragma unroll
          for (int i4 = 0; i4 < 8; ++i4) {
            // biases / head weights: one 128-bit shared-memory load per four latent dimensions
            const float4 bm_ = bm4[i4], bl_ = bl4[i4], wv_ = wv4[i4];
            const float bmv[4] = {bm_.x, bm_.y, bm_.z, bm_.w}, blv[4] = {bl_.x, bl_.y, bl_.z, bl_.w};
            const float wvv[4] = {wv_.x, wv_.y, wv_.z, wv_.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int i = 4 * i4 + k;
              const float e = q == 0 ? e0[i] : e1[i];
              const float m = mu[i] + bmv[k], l = lv[i] + blv[k];
              const float sd = expf(0.5f * l);
              dval = fmaf(wvv[k], fmaf(sd, e, m), dval);
              if (KL) klv += fmaf(m, m, fmaf(sd, sd, -l)) - 1.f;       // VDBLoss.kl_divergence, math.py:83-86
            }
          }
        }
      }
      dval += bd;
      if (live) {
        const float one_minus_p = 1.f / (1.f + expf(dval));
        if (a.reward) a.reward[env] = -logf(one_minus_p + 1e-8f);
        if (a.d_out) a.d_out[env] = dval;
        if (KL) a.kl_out[env] = 0.5f * klv;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 256);
}


// ---------------------------------------------------------------- VAIL, two CTAs per SM, A operand in TENSOR MEMORY
// Why: with both operands in shared memory (the kernels above) a 3xTF32 k-step of 8 moves 12 KB of A reads + 12 KB of B
// reads through the SM's 128 B/clk shared-memory port in the 192 cycles its three M128 x N128 MMAs take, plus the 8 KB
// the producers store for the next A chunk and the 8 KB the bulk copy writes for the next B chunk: 213 B/clk wanted, 128
// available -- both SS kernels run at ~1.65x their tensor-pipe floor, whatever the producers do (measured: dropping the
// A stores buys 12 %, dropping the producers' loads and arithmetic 8 %).  Here the activations never touch shared memory:
// the epilogue of layer l writes the hi / lo A chunks of layer l + 1 straight into TMEM (tcgen05.st: thread t owns lane t
// = sample t, exactly the layout the MMA wants for an M = 128 A operand) and the MMA reads them from there
// (tcgen05.mma [d], [a_tmem], b_desc).  Shared memory then carries the weights only: 107 B/clk.
// TMEM budget of a CTA (256 columns, two CTAs per SM): ACC1 = 64 (a 64-wide block of layer 1, later of [mu; logvar]),
// ACC2 = 128 (layer 2), A ring = 2 stages x (16 hi + 16 lo) columns.  Hence 64-wide blocks: layer 1 in four blocks each
// feeding four K-chunks of layer 2; the [mu; logvar] layer in four blocks of 32 + 32 interleaved rows (host side), the head
// consuming 32 latent dimensions per block.  56 chunks of 16 K-elements per tile.
// MEASURED (B200, round 2): parity-green, but 82.0 us at 65536 samples and 975 us at 1 M against 74.2 / 815 us for
// disc_vail2_kernel.  The TMEM budget forces 16-element chunks, a two-stage A ring and nine accumulator drains per tile
// (vail2: five); each chunk costs a tcgen05.ld -> split -> tcgen05.st -> wait::st -> mbarrier -> MMA -> commit round
// trip of ~1200 cycles against 192-384 cycles of MMA, so the kernel is handshake-latency-bound although its
// shared-memory traffic is half.  Kept selectable (om_debug_set "disc_vail2" = 3) and under test; NOT the default.
// What would make it pay: one CTA per SM with all 512 columns (128-wide blocks, a four-stage ring of 32-element chunks).
constexpr int V3_KC = 16, V3_NSB = 4, V3_NSA = 2;
constexpr int V3_STAGE_B = 128 * V3_KC * 4 * 2;          // 16 KB: the largest B chunk (128 rows, hi + lo)
constexpr int V3_ACC1 = 0, V3_ACC2 = 64, V3_AR = 192;
constexpr int V3_NPAR = 256 + 128 + 256 + 128 + 1;       // b1, b2, b3 (interleaved like the rows), wd, bd
constexpr int V3_CHUNKS = 4 * (2 + 4) + 4 * 8;           // 56
__host__ __device__ constexpr int v3_rows(int c) { return c < 24 ? ((c % 6) < 2 ? 64 : 128) : 64; }
__host__ __device__ constexpr int v3_offset_bytes(int c) {          // start of chunk c in the image
  int o = 0;
  for (int i = 0; i < c; ++i) o += v3_rows(i) * V3_KC * 4 * 2;
  return o;
}
constexpr int V3_IMAGE_BYTES = v3_offset_bytes(V3_CHUNKS);

__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
               "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}"
               ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(acc), "r"(0u) : "memory");
}
// 16 consecutive TMEM columns of this thread's lane <- registers
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
               ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                 "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])),
                 "r"(__float_as_uint(v[7])), "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])),
                 "r"(__float_as_uint(v[11])), "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])),
                 "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
               : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// Load without the wait: several loads in flight, then tmem_ld_wait() on each register set (the "+r" operands keep the
// compiler from using the registers before the wait).
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                 "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
               : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :: "memory");
}

template <bool KL>
__global__ void __launch_bounds__(192, 2) disc_vail3_kernel(DiscArgs a) {
  constexpr int Z = 128;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* ring = smem;
  float* par = reinterpret_cast<float*>(smem + V3_NSB * V3_STAGE_B);
  float* s_mean = par + V3_NPAR + 3;
  float* s_inv = s_mean + DISC_IN;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_inv + DISC_IN);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * V3_NSA + 2 * V3_NSB);
  const float* b1 = par;
  const float* b2 = par + 256;
  const float* b3 = par + 384;            // per 64-row block h: [bmu[32h..32h+31], blv[32h..32h+31]]
  const float* wd = par + 640;
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t bar0 = smem_u32(bars);
  auto a_full = [&](int s_) { return bar0 + 8u * s_; };
  auto a_free = [&](int s_) { return bar0 + 8u * (V3_NSA + s_); };
  auto b_full = [&](int s_) { return bar0 + 8u * (2 * V3_NSA + s_); };
  auto b_free = [&](int s_) { return bar0 + 8u * (2 * V3_NSA + V3_NSB + s_); };

  for (int i = tid; i < V3_NPAR; i += 192) par[i] = a.params[i];
  if (tid < DISC_IN) { s_mean[tid] = a.mean[tid]; s_inv[tid] = 1.0f / a.stdv[tid]; }
  if (tid == 0) {
    for (int s_ = 0; s_ < V3_NSA; ++s_) { mbar_init(a_full(s_), 128); mbar_init(a_free(s_), 1); }
    for (int s_ = 0; s_ < V3_NSB; ++s_) { mbar_init(b_full(s_), 1); mbar_init(b_free(s_), 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const int ntiles = (a.n + TILE - 1) / TILE;
  int my_tiles = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) ++my_tiles;
  const int total_chunks = my_tiles * V3_CHUNKS;

  if (warp == 5) {
    // ===================================================== weight-copy issuer: the image repeats every tile
    if (tid == 160) {
      int c = 0, off = 0;
      for (int g = 0; g < total_chunks; ++g) {
        const int st = g % V3_NSB, use = g / V3_NSB;
        const int bytes = v3_rows(c) * V3_KC * 4 * 2;
        if (use > 0) mbar_wait(b_free(st), (uint32_t)(use - 1) & 1u);
        mbar_expect_tx(b_full(st), bytes);
        const uint8_t* src = reinterpret_cast<const uint8_t*>(a.image) + off;
        const uint32_t dst = smem_u32(ring + st * V3_STAGE_B);
        bulk_g2s(dst, src, bytes / 2, b_full(st));
        bulk_g2s(dst + bytes / 2, src + bytes / 2, bytes / 2, b_full(st));
        off += bytes;
        if (++c == V3_CHUNKS) { c = 0; off = 0; }
      }
    }
  } else if (warp == 4) {
    // ===================================================== MMA issuer
    if (elect_one_sync()) {
      int c = 0;
      for (int g = 0; g < total_chunks; ++g) {
        const int sa = g % V3_NSA, sb = g % V3_NSB;
        const int rows = v3_rows(c);
        uint32_t d_col;
        bool first;
        if (c < 24) {
          const int r = c % 6;                                   // 0,1: layer 1 of this block; 2..5: layer 2
          d_col = r < 2 ? V3_ACC1 : V3_ACC2;
          first = r < 2 ? (r == 0) : (c == 2);                   // layer 2 accumulates over the four blocks
        } else {
          d_col = V3_ACC1;
          first = ((c - 24) % 8) == 0;
        }
        const uint32_t idesc = idesc_tf32(TILE, rows);
        const uint32_t lbo = (uint32_t)rows * 16, sbo = 128;
        mbar_wait(a_full(sa), (uint32_t)(g / V3_NSA) & 1u);
        mbar_wait(b_full(sb), (uint32_t)(g / V3_NSB) & 1u);
        tc_fence_after();
        const uint32_t a_hi = tmem + V3_AR + sa * 32, a_lo = a_hi + 16;
        const uint32_t b_hi = smem_u32(ring + sb * V3_STAGE_B), b_lo = b_hi + rows * V3_KC * 4;
#pragma unroll
        for (int j = 0; j < V3_KC / 8; ++j) {
          const uint32_t o = (uint32_t)j * 2 * lbo;
          const uint64_t dbh = smem_desc(b_hi + o, lbo, sbo), dbl = smem_desc(b_lo + o, lbo, sbo);
          umma_tf32_ts(tmem + d_col, a_lo + 8 * j, dbh, idesc, (first && j == 0) ? 0u : 1u);
          umma_tf32_ts(tmem + d_col, a_hi + 8 * j, dbl, idesc, 1u);
          umma_tf32_ts(tmem + d_col, a_hi + 8 * j, dbh, idesc, 1u);
        }
        umma_commit(a_free(sa));
        umma_commit(b_free(sb));
        if (++c == V3_CHUNKS) c = 0;
      }
    }
  } else {
    // ===================================================== producers / epilogue (128 threads; thread t = TMEM lane t)
    const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
    const float bd = par[V3_NPAR - 1];
    int g = 0;
    auto wait_chunk = [&](int h) {                         // all MMAs up to and including chunk h are complete
      if (h >= 0) {
        mbar_wait(a_free(h % V3_NSA), (uint32_t)(h / V3_NSA) & 1u);
        tc_fence_after();
      }
    };
    auto put = [&](const float (&act_in)[16]) {
      float hi[16], lo[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) { hi[i] = tf32_rna(act_in[i]); lo[i] = act_in[i] - hi[i]; }
      wait_chunk(g - V3_NSA);                              // the MMAs that read this A stage last are complete
      const uint32_t at = lane_addr + V3_AR + (g % V3_NSA) * 32;
      tmem_st16(at, hi);
      tmem_st16(at + 16, lo);
      tmem_wait_st();
      tc_fence_before();
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a_full(g % V3_NSA)) : "memory");
      ++g;
    };
    auto load_row = [&](int tile_, float (&raw)[DISC_IN]) {
      const int env_ = tile_ * TILE + tid;
#pragma unroll
      for (int k = 0; k < DISC_IN; ++k) raw[k] = (tile_ < ntiles && env_ < a.n) ? a.s[(size_t)k * a.ld + env_] : 0.f;
    };
    float xn[DISC_IN];
    load_row(blockIdx.x, xn);
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      const int env = tile * TILE + tid;
      const bool live = env < a.n;
      float x[DISC_IN];
#pragma unroll
      for (int k = 0; k < DISC_IN; ++k) x[k] = live ? (xn[k] - s_mean[k]) * s_inv[k] : 0.f;
      load_row(tile + gridDim.x, xn);
#pragma unroll 1
      for (int blk = 0; blk < 4; ++blk) {
        {
          float h0[16], h1[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) { h0[i] = x[i]; h1[i] = x[16 + i]; }
          put(h0);
          put(h1);
        }
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          if (c == 0) wait_chunk(g - 1);                                  // this layer-1 block is complete
          float h[16];
          tmem_ld16(lane_addr + V3_ACC1 + c * V3_KC, h);
          bias_relu16(h, b1 + blk * 64 + c * V3_KC);
          put(h);
        }
      }
      float dval = 0.f, klv = 0.f;
#pragma unroll 1
      for (int hb = 0; hb < 4; ++hb) {
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {
          if (c == 0 && hb == 0) wait_chunk(g - 1);                       // layer 2 complete
          float h[16];
          tmem_ld16(lane_addr + V3_ACC2 + c * V3_KC, h);
          bias_relu16(h, b2 + c * V3_KC);
          put(h);
        }
        // head over latent dimensions 32 hb .. 32 hb + 31: z = mu + exp(logvar / 2) eps, d += wd . z
        float e[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) e[i] = (a.eps && live) ? a.eps[(size_t)(32 * hb + i) * a.ld + env] : 0.f;
        wait_chunk(g - 1);
        float mu[32], lv[32];
        tmem_ld32(lane_addr + V3_ACC1, mu);
        tmem_ld32(lane_addr + V3_ACC1 + 32, lv);
        const float4* bm4 = reinterpret_cast<const float4*>(b3 + 64 * hb);
        const float4* bl4 = reinterpret_cast<const float4*>(b3 + 64 * hb + 32);
        const float4* wv4 = reinterpret_cast<const float4*>(wd + 32 * hb);
#pragma unroll
        for (int i4 = 0; i4 < 8; ++i4) {
          const float4 bm_ = bm4[i4], bl_ = bl4[i4], wv_ = wv4[i4];
          const float bmv[4] = {bm_.x, bm_.y, bm_.z, bm_.w}, blv[4] = {bl_.x, bl_.y, bl_.z, bl_.w};
          const float wvv[4] = {wv_.x, wv_.y, wv_.z, wv_.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int i = 4 * i4 + k;
            const float m = mu[i] + bmv[k], l = lv[i] + blv[k];
            const float sd = expf(0.5f * l);
            dval = fmaf(wvv[k], fmaf(sd, e[i], m), dval);
            if (KL) klv += fmaf(m, m, fmaf(sd, sd, -l)) - 1.f;       // VDBLoss.kl_divergence, math.py:83-86
          }
        }
      }
      dval += bd;
      if (live) {
        const float one_minus_p = 1.f / (1.f + expf(dval));
        if (a.reward) a.reward[env] = -logf(one_minus_p + 1e-8f);
        if (a.d_out) a.d_out[env] = dval;
        if (KL) a.kl_out[env] = 0.5f * klv;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 256);
}


// ---------------------------------------------------------------- VAIL, ONE CTA per SM, A operand in tensor memory
// The answer to what held disc_vail3_kernel back: with all 512 TMEM columns a CTA affords 128-wide accumulator blocks
// (ACC1a, ACC1b, ACC2) and a two-stage A ring of 32-element chunks, so a tile is 13 A chunks and 18 B chunks instead of
// 56 + 56, every A chunk is produced ONCE (the input chunk feeds both layer-1 blocks, each layer-2 chunk both [mu; logvar]
// blocks), and the accumulators a layer reads are never the ones the MMA pipe is writing:
//   A0      = x                         -> B W1[0:128]   -> ACC1a      and  B W1[128:256] -> ACC1b
//   A1..A4  = relu(ACC1a + b1[0:128])   -> B W2[:, 0:128]   (4 chunks) -> ACC2
//   A5..A8  = relu(ACC1b + b1[128:256]) -> B W2[:, 128:256] (4 chunks) -> ACC2
//   A9..A12 = relu(ACC2 + b2)           -> B [mu; lv][0:64] -> ACC1a   and  B [mu; lv][64:128] -> ACC1b
//   head(h0) reads ACC1a, head(h1) reads ACC1b (z = mu + exp(lv / 2) eps, d += wd . z)
// Two producer warpgroups (threads t and t + 128 own sample t and split every chunk's 32 columns, the input row and the
// head, as in disc_reward_pg2_kernel), one MMA-issuing thread, one copy-issuing thread.  Besides the rings there is one
// mbarrier per "accumulator complete" event (r1a, r1b, r2, r3a, r3b: one phase per tile) and h_done (the heads have
// finished reading ACC1a / ACC1b: the next tile's layer 1 may overwrite them).  Shared memory carries weights only
// (six 32 KB stages).
constexpr int V4_KC = 32, V4_NSB = 6, V4_NSA = 2;
constexpr int V4_STAGE_B = 128 * V4_KC * 4 * 2;          // 32 KB: 128 rows x 32 K, hi + lo
constexpr int V4_ACC1A = 0, V4_ACC1B = 128, V4_ACC2 = 256, V4_AR = 384;
enum { V4_R1A = 0, V4_R1B, V4_R2, V4_R3A, V4_R3B, V4_NR };
// With NCH input chunks a tile is NCH + 12 A chunks and 2 NCH + 16 B chunks (both layer-1 blocks read every input chunk).
// The weight ring has as many stages as divide the B chunk count -- six for one input chunk (18 B chunks), five for two
// (20) -- so that the stage of every chunk of the unrolled tile body is a compile-time constant.
__host__ __device__ constexpr int v4_bchunks(int nch) { return 2 * nch + 16; }
__host__ __device__ constexpr int v4_nsb(int nch) { return v4_bchunks(nch) % V4_NSB == 0 ? V4_NSB : 5; }
__host__ __device__ constexpr size_t v4_smem(int nch) {
  return (size_t)v4_nsb(nch) * V4_STAGE_B + (V2_NPAR + 3 + 2 * KC * nch + 256) * sizeof(float) +
         (2 * V4_NSA + 2 * v4_nsb(nch) + V4_NR + 2) * 8 + 16;
}

//
// Where the time goes (clock counters in the MMA-issuing thread and in a producer thread; experiments that are not in the
// tree).  (a) The issuing thread itself paced the MMAs: a back-to-back M128 x N128 x K8 TF32 MMA takes 64 cycles
// (tools/micro/umma_rate.cu), but it went out every 92 cycles while the weight stage was a run-time index (four dependent
// uniform-datapath instructions per descriptor), every ~71 while the issuing code sat behind `tid == 256` (ptxas wraps
// each tcgen05.mma in a five-instruction elect / vote loop unless the branch is taken through elect.sync), plus ~100
// cycles per mbarrier wait even on a completed phase.  Unrolled tile body + elect_one_sync + weights waited for before the
// A chunk: 27.7 k -> 22.6 k cycles per tile at 1 M samples (802 -> 659 us), 69 -> 59 us at 65536.  (b) A tile's timeline
// now (65536 samples, 19.5 k cycles): input chunk + layer 1 + first hand-over 1.9 k, layer 2 eight chunks of ~830 (768 of
// MMA + what is left of the hand-over chain MMA-commit -> a_free -> tcgen05.st -> wait::st -> a_full -> issue of a two-stage
// ring), 1.7 k at the layer-2 -> layer-3 boundary, layer 3 four chunks of 1536 (MMA-bound), heads and output 3.5 k with
// 1.5 k of MMA under them.  216 MMAs are 13.8 k cycles: the pipe is busy 71 % of a tile.  (c) At 65536 samples a CTA has 3
// or 4 tiles (512 tiles over 148 SMs: 3.46 rounded up to 4 is 13.5 % lost to the tile count alone); a four-tile CTA
// lives 81 k cycles with its inputs in L2 (45.8 us at the 1.77 GHz the SM clock shows under this load, globaltimer against
// clock64), 90 k = 50.8 us after the L2 flush the benchmark does, 4 k of them prologue and drain; the benchmark's 59 us
// are that plus launch, block scheduling and completion.
// Measured against that, all parity-green, none faster: handing an A chunk over one put() late so that its TMEM-store
// latency sits under the next chunk's arithmetic, four TMEM loads in flight per block, the first weight chunks and input
// rows requested ahead of the prologue (neutral, kept); ROT = 1 / 2 below (next tile's layer 1 under this tile's heads:
// the next layer 2 does start 1.5 k cycles earlier, and this tile's layer 3 ends 1.5 k later); ROT = 3, the two producer
// warpgroups on alternate chunks, one ring stage each (identical time: the producers are not what layer 2 waits for); and
// a third warpgroup that does nothing but heads, with layer-1 block b issued after the first half of layer 2 (448 threads
// at 128 registers: 80 us / 832 us, not kept).
//
// ROT (opt-in through om_debug_set("disc_vail2", 6 / 5 / 7)): 3 = alternating producer warpgroups; 1 = the next tile's input chunk is handed over before the
// heads and the two layer-1 blocks are released one by one (h_done_a after head a's loads, h_done after head b's);
// 2 = the three accumulator blocks change roles from tile to tile instead, (L1a/L3a, L1b/L3b, L2)(i + 1) = (L2, L1a/L3a,
// L1b/L3b)(i): the next tile's first layer-1 block goes into the block this tile's layer 2 used (read out once A12
// exists), its second into the one head a has finished with, its layer 2 into the one head b has finished with.
template <bool KL, int ROT, int IN = 0>
__global__ void __launch_bounds__(320, 1) disc_vail4_kernel(typename DiscInput<IN>::Args a) {
  constexpr int NCH = DiscInput<IN>::NCH, KIN = KC * NCH;            // input chunks, padded input width
  constexpr int NSB = v4_nsb(NCH), BCH = v4_bchunks(NCH), ACH = NCH + 12;
  static_assert(IN == 0 || ROT == 0, "other input widths: the default schedule only");
  const int nin = DiscInput<IN>::n_in(a);
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* ring = smem;
  float* par = reinterpret_cast<float*>(smem + NSB * V4_STAGE_B);
  float* s_mean = par + V2_NPAR + 3;
  float* s_inv = s_mean + KIN;
  float* red = s_inv + KIN;                                     // [2][128] partial head sums of the second warpgroup
  uint64_t* bars = reinterpret_cast<uint64_t*>(red + 256);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * V4_NSA + 2 * NSB + V4_NR + 2);
  const float* b1 = par;
  const float* b2 = par + 256;
  const float* b3 = par + 384;            // per 128-row block h: [bmu[64h..64h+63], blv[64h..64h+63]]
  const float* wd = par + 640;
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t bar0 = smem_u32(bars);
  auto a_full = [&](int s_) { return bar0 + 8u * s_; };
  auto a_free = [&](int s_) { return bar0 + 8u * (V4_NSA + s_); };
  auto b_full = [&](int s_) { return bar0 + 8u * (2 * V4_NSA + s_); };
  auto b_free = [&](int s_) { return bar0 + 8u * (2 * V4_NSA + NSB + s_); };
  auto ready = [&](int k) { return bar0 + 8u * (2 * V4_NSA + 2 * NSB + k); };
  const uint32_t h_done = bar0 + 8u * (2 * V4_NSA + 2 * NSB + V4_NR);          // head b (and, without ROT, head a) has read
  const uint32_t h_done_a = h_done + 8u;                                       // ROT: head a has read its block
  constexpr bool EARLY = ROT == 1 || ROT == 2;     // the next tile's input chunk is handed over before this tile's heads
  constexpr bool ALT = ROT == 3;                   // the two producer warpgroups take alternate A chunks (one ring stage each)
  // accumulator blocks of tile `it`: P = layer-1 block a, then [mu; lv] block a; Q = the same for b; R = layer 2
  auto acc_p = [&](int it_) { return ROT == 2 ? (uint32_t)(128 * ((3 - it_ % 3) % 3)) : (uint32_t)V4_ACC1A; };
  auto acc_q = [&](int it_) { return ROT == 2 ? (uint32_t)(128 * ((4 - it_ % 3) % 3)) : (uint32_t)V4_ACC1B; };
  auto acc_r = [&](int it_) { return ROT == 2 ? (uint32_t)(128 * ((5 - it_ % 3) % 3)) : (uint32_t)V4_ACC2; };

  const int ntiles = (a.n + TILE - 1) / TILE;
  int my_tiles = 0;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) ++my_tiles;
  // Prologue: the first weight chunks and the first input rows are requested BEFORE the parameter loads, the TMEM
  // allocation and the CTA-wide barrier, so that their DRAM / L2 latency runs under those (at 65536 samples a CTA has only
  // three or four tiles: every microsecond in front of the first MMA is 1.5 % of the call).
  // (16 NCH values: this thread's 16 columns of every input chunk, input 32 ch + 16 half + k at 16 ch + k)
  float xn[ALT ? 32 : 16 * NCH];
  if (warp < 8) {
    const int half_ = warp >> 2;
    if (ALT) {                                      // warpgroup h hands over the input chunk of tiles h, h + 2, ...: whole rows
      const int tile_ = blockIdx.x + half_ * gridDim.x, env_ = tile_ * TILE + (tid & 127);
#pragma unroll
      for (int k = 0; k < (ALT ? 32 : 0); ++k) xn[k] = (tile_ < ntiles && env_ < a.n) ? a.s[(size_t)k * a.ld + env_] : 0.f;
    } else {
      const int env_ = blockIdx.x * TILE + (tid & 127);
#pragma unroll
      for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const int r = KC * ch + 16 * half_ + k;
          xn[16 * ch + k] = (env_ < a.n && (IN == 0 || r < nin)) ? a.s[(size_t)r * a.ld + env_] : 0.f;
        }
    }
  }
  int q_first = 0;                                                  // weight chunks already requested (copy thread only)
  if (tid == 288) {
    for (int s_ = 0; s_ < NSB; ++s_) { mbar_init(b_full(s_), 1); mbar_init(b_free(s_), 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const int total = my_tiles * BCH;
    for (; q_first < NSB && q_first < total; ++q_first) {
      mbar_expect_tx(b_full(q_first), V4_STAGE_B);
      const uint8_t* src = reinterpret_cast<const uint8_t*>(a.image) + (size_t)q_first * V4_STAGE_B;
      const uint32_t dst = smem_u32(ring + q_first * V4_STAGE_B);
#pragma unroll
      for (int p = 0; p < 4; ++p) bulk_g2s(dst + p * (V4_STAGE_B / 4), src + p * (V4_STAGE_B / 4), V4_STAGE_B / 4, b_full(q_first));
    }
  }
  for (int i = tid; i < V2_NPAR; i += 320) par[i] = a.params[i];
  if (tid < KIN) {
    const bool in_ = IN == 0 || tid < nin;                            // padding columns: mean 0, 1 / std 0
    s_mean[tid] = in_ ? a.mean[tid] : 0.f;
    s_inv[tid] = in_ ? 1.0f / a.stdv[tid] : 0.f;
  }
  if (tid == 0) {
    for (int s_ = 0; s_ < V4_NSA; ++s_) { mbar_init(a_full(s_), ALT ? 128 : 256); mbar_init(a_free(s_), 1); }
    for (int k = 0; k < V4_NR; ++k) mbar_init(ready(k), 1);
    mbar_init(h_done, 256);
    mbar_init(h_done_a, 256);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 9) {
    // ===================================================== weight-copy issuer: 18 (20) chunks of 32 KB per tile, MMA order
    if (tid == 288) {
      const int total = my_tiles * BCH;
      for (int q = q_first; q < total; ++q) {
        const int st = q % NSB, use = q / NSB;
        if (use > 0) mbar_wait(b_free(st), (uint32_t)(use - 1) & 1u);
        mbar_expect_tx(b_full(st), V4_STAGE_B);
        const uint8_t* src = reinterpret_cast<const uint8_t*>(a.image) + (size_t)(q % BCH) * V4_STAGE_B;
        const uint32_t dst = smem_u32(ring + st * V4_STAGE_B);
#pragma unroll
        for (int p = 0; p < 4; ++p) bulk_g2s(dst + p * (V4_STAGE_B / 4), src + p * (V4_STAGE_B / 4), V4_STAGE_B / 4, b_full(st));
      }
    }
  } else if (warp == 8) {
    // ===================================================== MMA issuer
    // One thread issues 216 MMAs per tile, and its own instruction stream is what paces them if it is not kept short: a
    // back-to-back M128 x N128 x K8 TF32 MMA takes 64 cycles (tools/micro/umma_rate.cu, SS and TS alike), but with the
    // stage index a run-time value every shared-memory descriptor cost four dependent uniform-datapath instructions and
    // an MMA went out every 92 cycles.  18 weight chunks per tile is a multiple of the six stages (20 of the five with two
    // input chunks), so with the tile body unrolled the stage of every chunk is a compile-time constant and a descriptor
    // is ONE add: (ring address >> 4) + (constant offset | the constant leading-byte-offset field); the A chunks alternate
    // between two TMEM stages whose order flips from tile to tile when a tile has an odd number of them (13 with one
    // input chunk), kept as two registers that are swapped.
    if (elect_one_sync()) {
      static_assert(BCH % NSB == 0, "stage bookkeeping of the unrolled tile body");
      const uint32_t idesc = idesc_tf32(TILE, 128);
      constexpr uint32_t LBO16 = 128, SBO16 = 8;                        // 2048 B and 128 B in 16-byte units
      constexpr uint32_t DESC_HI = SBO16 | (1u << 14);                  // bits 32..45 stride byte offset, bit 46 version 1
      const uint32_t ring16 = smem_u32(ring) >> 4;                      // < 2^14: the address field cannot overflow
      auto bdesc = [&](uint32_t off16) { return ((uint64_t)DESC_HI << 32) | (uint64_t)(ring16 + (off16 + (LBO16 << 16))); };
      uint32_t a_st[2] = {tmem + V4_AR, tmem + V4_AR + 64};             // TMEM stage of this tile's even / odd A chunks
      uint32_t a_fu[2] = {a_full(0), a_full(1)}, a_fr[2] = {a_free(0), a_free(1)};
      int ga = 0;
      for (int it = 0; it < my_tiles; ++it) {
        const uint32_t P = tmem + acc_p(it), Q = tmem + acc_q(it), R = tmem + acc_r(it);
        // (parity of the uses of a weight stage before this tile: BCH / NSB uses per tile)
        const uint32_t itp = (BCH / NSB) % 2 ? (uint32_t)it & 1u : 0u;
        // B chunk q of the tile (stage q % NSB, its (BCH / NSB it + q / NSB)-th use) against the A chunk in TMEM stage `ab`:
        // 4 k-steps x (lo.hi, hi.lo, hi.hi)
        // (the weights are waited for BEFORE the A chunk: they arrive chunks ahead, the A chunk is what the MMA pipe is
        // waiting for, and every mbarrier wait costs the issuing thread ~100 cycles even when the phase is long complete)
        auto wait_b = [&](int q) { mbar_wait(b_full(q % NSB), (itp ^ (uint32_t)(q / NSB)) & 1u); tc_fence_after(); };
        auto mma_chunk = [&](int q, uint32_t ab, uint32_t d, bool first) {
          const int sb = q % NSB;
#pragma unroll
          for (int j = 0; j < V4_KC / 8; ++j) {
            const uint64_t dbh = bdesc((uint32_t)(sb * (V4_STAGE_B / 16) + j * 2 * LBO16));
            const uint64_t dbl = bdesc((uint32_t)(sb * (V4_STAGE_B / 16) + V4_STAGE_B / 32 + j * 2 * LBO16));
            umma_tf32_ts(d, ab + 32 + 8 * j, dbh, idesc, (first && j == 0) ? 0u : 1u);
            umma_tf32_ts(d, ab + 8 * j, dbl, idesc, 1u);
            umma_tf32_ts(d, ab + 8 * j, dbh, idesc, 1u);
          }
          umma_commit(b_free(sb));
        };
        auto next_a = [&](int k) {                                      // A chunk k of the tile: wait, return its TMEM stage
          mbar_wait(a_fu[k & 1], (uint32_t)(ga >> 1) & 1u);
          tc_fence_after();
          ++ga;
          return a_st[k & 1];
        };
        // without ROT: P and Q are what the previous tile's heads read.  With ROT: P is the previous tile's layer-2 block,
        // read out before its last layer-3 chunk was issued; Q waits for head a, R for head b.
        // ROT 0: P and Q are what the previous tile's heads read, both released by h_done.
        // ROT 1: the same blocks, released one by one -- P by head a (h_done_a), Q by head b (h_done).
        // ROT 2: P is the previous tile's layer-2 block, read out before its last layer-3 chunk was issued; Q waits for
        //        head a, R for head b.
        if ((ROT == 0 || ROT == 3) && it > 0) { mbar_wait(h_done, (uint32_t)(it - 1) & 1u); tc_fence_after(); }
        if (ROT == 1 && it > 0) { mbar_wait(h_done_a, (uint32_t)(it - 1) & 1u); tc_fence_after(); }
        uint32_t ab;
#pragma unroll
        for (int k = 0; k < NCH; ++k) {                                 // A0 (A0, A1) = x -> layer-1 blocks a and b
          wait_b(2 * k);
          ab = next_a(k);
          mma_chunk(2 * k, ab, P, k == 0);
          if (k == NCH - 1) umma_commit(ready(V4_R1A));
          wait_b(2 * k + 1);
          if (ROT == 2 && it > 0) { mbar_wait(h_done_a, (uint32_t)(it - 1) & 1u); tc_fence_after(); }
          if (ROT == 1 && it > 0) { mbar_wait(h_done, (uint32_t)(it - 1) & 1u); tc_fence_after(); }
          mma_chunk(2 * k + 1, ab, Q, k == 0);
          umma_commit(a_fr[k & 1]);
        }
        umma_commit(ready(V4_R1B));
        if (ROT == 2 && it > 0) { mbar_wait(h_done, (uint32_t)(it - 1) & 1u); tc_fence_after(); }
#pragma unroll
        for (int c = 0; c < 8; ++c) {                                   // A1..A8 (A2..A9) -> layer 2
          wait_b(2 * NCH + c);
          ab = next_a(NCH + c);
          mma_chunk(2 * NCH + c, ab, R, c == 0);
          umma_commit(a_fr[(NCH + c) & 1]);
        }
        umma_commit(ready(V4_R2));
#pragma unroll
        for (int c = 0; c < 4; ++c) {                                   // A9..A12 (A10..A13) -> [mu; lv] blocks a and b
          wait_b(2 * NCH + 8 + 2 * c);
          ab = next_a(NCH + 8 + c);
          mma_chunk(2 * NCH + 8 + 2 * c, ab, P, c == 0);
          if (c == 3) umma_commit(ready(V4_R3A));
          wait_b(2 * NCH + 9 + 2 * c);
          mma_chunk(2 * NCH + 9 + 2 * c, ab, Q, c == 0);
          umma_commit(a_fr[(NCH + 8 + c) & 1]);
        }
        umma_commit(ready(V4_R3B));
        if constexpr (ACH % V4_NSA == 1) {                              // the next tile's even chunks live in the other stage
          { const uint32_t t_ = a_st[0]; a_st[0] = a_st[1]; a_st[1] = t_; }
          { const uint32_t t_ = a_fu[0]; a_fu[0] = a_fu[1]; a_fu[1] = t_; }
          { const uint32_t t_ = a_fr[0]; a_fr[0] = a_fr[1]; a_fr[1] = t_; }
        }
      }
    }
  } else {
    // ===================================================== producers / epilogue: 2 warpgroups, thread t and t + 128 = sample t
    const int half = warp >> 2, row = tid & 127;                       // a warp may touch TMEM lanes 32 (warp % 4) ..
    const uint32_t lane_addr = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const float bd = par[V2_NPAR - 1];
    int ga = 0;
    // A chunk is handed over in two steps: put() splits it and issues the TMEM stores; publish() -- wait for the stores,
    // arrive on a_full -- is made by the NEXT put() after its own split, so the store latency sits under that arithmetic
    // instead of in front of the MMA (per-chunk producer latency, not the MMA pipe, bounded this kernel: 13 chunks x
    // ~0.8 us against 7 us of MMA per tile).  publish() must be called by hand before waiting on anything the pending chunk
    // feeds (an accumulator-complete barrier of its own layer).
    int pending = -1;
    auto publish = [&]() {
      if (pending >= 0) {
        tmem_wait_st();
        tc_fence_before();
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a_full(pending)) : "memory");
        pending = -1;
      }
    };
    auto put = [&](const float (&act_in)[16]) {                        // this thread's 16 of the chunk's 32 columns
      float hi[16], lo[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) { hi[i] = tf32_rna(act_in[i]); lo[i] = act_in[i] - hi[i]; }
      publish();
      if (ga >= V4_NSA) { mbar_wait(a_free(ga % V4_NSA), (uint32_t)(ga / V4_NSA - 1) & 1u); tc_fence_after(); }
      const uint32_t at = lane_addr + V4_AR + (ga % V4_NSA) * 64 + 16 * half;
      tmem_st16(at, hi);
      tmem_st16(at + 32, lo);
      pending = ga % V4_NSA;
      ++ga;
    };
    // four chunks out of one accumulator block: all four loads in flight, then bias + relu + put chunk by chunk
    auto put_block = [&](uint32_t acc, const float* bias) {
      uint32_t r[4][16];
#pragma unroll
      for (int c = 0; c < 4; ++c) tmem_ld16_nowait(lane_addr + acc + c * V4_KC + 16 * half, r[c]);
#pragma unroll
      for (int c = 0; c < 4; ++c) tmem_ld_wait(r[c]);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float h[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) h[i] = __uint_as_float(r[c][i]);
        bias_relu16(h, bias + c * V4_KC + 16 * half);
        put(h);
        // the first chunk of a block is what the idle MMA pipe is waiting for, and behind the last one comes a wait and
        // a round of loads, not arithmetic: those two are handed over at once
        if (c == 0 || c == 3) publish();
      }
    };
    auto wait_ready = [&](int k, int it) { mbar_wait(ready(k), (uint32_t)it & 1u); tc_fence_after(); };
    auto load_row = [&](int tile_, float (&raw)[16 * NCH]) {
      const int env_ = tile_ * TILE + row;
#pragma unroll
      for (int ch = 0; ch < NCH; ++ch)
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const int r = KC * ch + 16 * half + k;
          raw[16 * ch + k] = (tile_ < ntiles && env_ < a.n && (IN == 0 || r < nin)) ? a.s[(size_t)r * a.ld + env_] : 0.f;
        }
    };
    auto put_input = [&](int tile_) {                                   // A0 (A0, A1) of tile_ from the prefetched row
      const bool live_ = tile_ * TILE + row < a.n;
#pragma unroll
      for (int ch = 0; ch < NCH; ++ch) {
        float x[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const int r = KC * ch + 16 * half + k;
          x[k] = live_ ? (xn[16 * ch + k] - s_mean[r]) * s_inv[r] : 0.f;
        }
        put(x);
      }
    };
    int it = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const int env = tile * TILE + row;
      const bool live = env < a.n;
      const uint32_t P = acc_p(it), Q = acc_q(it), R = acc_r(it);
      if constexpr (ALT) {
        // Chunk k of the tile is the (13 it + k)-th of the kernel and lives in ring stage (13 it + k) & 1: warpgroup `half`
        // produces the chunks of stage `half`, all 32 columns of its row -- every second chunk, so that it has TWO chunks'
        // MMA time for the hand-over chain (a_free -> tcgen05.st -> wait::st -> a_full) that bounds layer 2 when both
        // warpgroups work on every chunk.
        const int par = (half + it) & 1;                                // this tile: k = par, par + 2, ...
        auto put32 = [&](const float (&act)[32]) {
          if (ga > 0) { mbar_wait(a_free(half), (uint32_t)(ga - 1) & 1u); tc_fence_after(); }   // ga: this stage's uses
          const uint32_t at = lane_addr + V4_AR + half * 64;
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            float hi[16], lo[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) { hi[i] = tf32_rna(act[16 * g + i]); lo[i] = act[16 * g + i] - hi[i]; }
            tmem_st16(at + 16 * g, hi);
            tmem_st16(at + 32 + 16 * g, lo);
          }
          tmem_wait_st();
          tc_fence_before();
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a_full(half)) : "memory");
          ++ga;
        };
        if (par == 0) {                                                 // k = 0: the input chunk
          float x[32];
#pragma unroll
          for (int k = 0; k < 32; ++k) x[k] = live ? (xn[k % (ALT ? 32 : 16)] - s_mean[k]) * s_inv[k] : 0.f;
          put32(x);
          const int tile_ = tile + 2 * (int)gridDim.x, env_ = tile_ * TILE + row;   // this warpgroup's next input chunk
#pragma unroll
          for (int k = 0; k < (ALT ? 32 : 0); ++k) xn[k] = (tile_ < ntiles && env_ < a.n) ? a.s[(size_t)k * a.ld + env_] : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 6; ++j) {                                   // k = 2 j + 1 (par = 1) or 2 j + 2 (par = 0)
          const int blk = j >> 1;                                       // 0: layer-1 block a, 1: block b, 2: layer 2
          const int c = 2 * (j & 1) + (par ^ 1);                        // chunk of the block
          if ((j & 1) == 0) wait_ready(blk == 0 ? V4_R1A : blk == 1 ? V4_R1B : V4_R2, it);
          float h[32];
          tmem_ld32(lane_addr + (blk == 0 ? P : blk == 1 ? Q : R) + c * V4_KC, h);
          const float* bias = (blk == 2 ? b2 : b1 + blk * 128) + c * V4_KC;
          float h0[16], h1[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) { h0[i] = h[i]; h1[i] = h[16 + i]; }
          bias_relu16(h0, bias);
          bias_relu16(h1, bias + 16);
#pragma unroll
          for (int i = 0; i < 16; ++i) { h[i] = h0[i]; h[16 + i] = h1[i]; }
          put32(h);
        }
      } else {
      if (!EARLY || it == 0) {
        put_input(tile);                                                // A0
        publish();
        load_row(tile + gridDim.x, xn);
      }
#pragma unroll 1
      for (int blk = 0; blk < 2; ++blk) {                               // A1..A8: relu(layer 1 + b1)
        wait_ready(blk == 0 ? V4_R1A : V4_R1B, it);                     // (A4 may be pending here: R1B does not need it)
        put_block(blk == 0 ? P : Q, b1 + blk * 128);
      }
      publish();                                                        // A8: layer 2 cannot complete without it
      wait_ready(V4_R2, it);
      put_block(R, b2);                                                 // A9..A12: relu(layer 2 + b2)
      if (EARLY && tile + (int)gridDim.x < ntiles) {                    // the next tile's A0, ahead of this tile's heads
        put_input(tile + gridDim.x);
        load_row(tile + 2 * gridDim.x, xn);
      }
      publish();                                                        // A12 (or the next A0)
      }
      float dval = 0.f, klv = 0.f;
#pragma unroll 1
      for (int hb = 0; hb < 2; ++hb) {                                  // heads: this thread's 32 of the block's 64 latents
        float e[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) e[i] = (a.eps && live) ? a.eps[(size_t)(64 * hb + 32 * half + i) * a.ld + env] : 0.f;
        wait_ready(hb == 0 ? V4_R3A : V4_R3B, it);
        const uint32_t acc = lane_addr + (hb == 0 ? P : Q);
        float mu[32], lv[32];
        tmem_ld32(acc + 32 * half, mu);
        tmem_ld32(acc + 64 + 32 * half, lv);
        if (EARLY && hb == 0) {                                         // block P has been read (tmem_ld32 waits for its data)
          tc_fence_before();
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(h_done_a) : "memory");
        }
        const float4* bm4 = reinterpret_cast<const float4*>(b3 + 128 * hb + 32 * half);
        const float4* bl4 = reinterpret_cast<const float4*>(b3 + 128 * hb + 64 + 32 * half);
        const float4* wv4 = reinterpret_cast<const float4*>(wd + 64 * hb + 32 * half);
#pragma unroll
        for (int i4 = 0; i4 < 8; ++i4) {
          const float4 bm_ = bm4[i4], bl_ = bl4[i4], wv_ = wv4[i4];
          const float bmv[4] = {bm_.x, bm_.y, bm_.z, bm_.w}, blv[4] = {bl_.x, bl_.y, bl_.z, bl_.w};
          const float wvv[4] = {wv_.x, wv_.y, wv_.z, wv_.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int i = 4 * i4 + k;
            const float m = mu[i] + bmv[k], l = lv[i] + blv[k];
            const float sd = expf(0.5f * l);
            dval = fmaf(wvv[k], fmaf(sd, e[i], m), dval);
            if (KL) klv += fmaf(m, m, fmaf(sd, sd, -l)) - 1.f;       // VDBLoss.kl_divergence, math.py:83-86
          }
        }
      }
      tc_fence_before();
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(h_done) : "memory");   // ACC1a / ACC1b may be overwritten
      // the two halves of a sample meet: half 1 hands its partial sums to half 0
      if (half == 1) { red[row] = dval; red[128 + row] = klv; }
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (half == 0 && live) {
        dval += red[row] + bd;
        const float one_minus_p = 1.f / (1.f + expf(dval));
        if (a.reward) a.reward[env] = -logf(one_minus_p + 1e-8f);
        if (a.d_out) a.d_out[env] = dval;
        if (KL) a.kl_out[env] = 0.5f * (klv + red[128 + row]);
      }
      asm volatile("bar.sync 2, 256;" ::: "memory");                     // red[] may be rewritten by the next tile
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

}  // namespace om

using namespace om;

struct OmDisc {
  DiscShape sh;
  int n_in;                     // 32: every kernel; otherwise the default kernels only (image4 + params2 / image + params)
  float* image = nullptr;
  float* params = nullptr;
  float* image2 = nullptr;      // VAIL: chunk image / parameters of disc_vail2_kernel
  float* params2 = nullptr;
  float* image3 = nullptr;      // VAIL: chunk image / parameters of disc_vail3_kernel (A operand in TMEM)
  float* params3 = nullptr;
  float* image4 = nullptr;      // VAIL: chunk image of disc_vail4_kernel (one CTA per SM, A in TMEM); parameters = params2
};

static void split_tf32(float x, float* hi, float* lo) {
  uint32_t u;
  std::memcpy(&u, &x, 4);
  u = (u + 0x1000u) & 0xFFFFE000u;                 // cvt.rna.tf32.f32: nearest, ties away from zero
  std::memcpy(hi, &u, 4);
  *lo = x - *hi;
}

// one A chunk: rows [r0, r0+rows) x columns [k0, k0+32) of a row-major [*, ldw] matrix, as two B sub-chunks of 16
// columns, each a hi image [4][rows][4] followed by its lo image
static void append_chunk(std::vector<float>& img, const float* w, int ldw, int r0, int rows, int k0) {
  for (int hb = 0; hb < KC / KB; ++hb) {
    const size_t base = img.size();
    img.resize(base + (size_t)rows * KB * 2);
    float* hi = img.data() + base;
    float* lo = hi + (size_t)rows * KB;
    for (int kc = 0; kc < KB / 4; ++kc)
      for (int r = 0; r < rows; ++r)
        for (int e = 0; e < 4; ++e)
          split_tf32(w[(size_t)(r0 + r) * ldw + k0 + hb * KB + kc * 4 + e], hi + ((size_t)kc * rows + r) * 4 + e,
                     lo + ((size_t)kc * rows + r) * 4 + e);
  }
}

extern "C" int om_disc_create(const OmDiscDesc* d, OmDisc** out) {
  OM_REQUIRE(d && out, "om_disc_create: null argument");
  OM_REQUIRE(d->n_in >= 1 && d->n_in <= DISC_MAX_IN, "om_disc_create: n_in must be 1..%d, got %d", DISC_MAX_IN, d->n_in);
  const bool vail = d->kind == 0;
  OM_REQUIRE(d->kind == 0 || d->kind == 1, "om_disc_create: kind must be 0 (VAIL) or 1 (GAIL)");
  OM_REQUIRE((vail && d->n_h1 == 256 && d->n_h2 == 128 && d->z_size == 128) || (!vail && d->n_h1 == 512 && d->n_h2 == 256),
             "om_disc_create: only the reference shapes are built (VAIL n_in-256-128-z128-1, GAIL n_in-512-256-1)");
  OM_REQUIRE(d->w1 && d->b1 && d->w2 && d->b2 && d->wd && d->bd, "om_disc_create: null weights");
  OM_REQUIRE(!vail || (d->wmu && d->bmu && d->wlv && d->blv), "om_disc_create: VAIL needs mu / logvar layers");
  const int n1 = d->n_h1, n2 = d->n_h2, z = vail ? d->z_size : 0;
  // W1 in whole 32-column input chunks, the padding columns zero.  The earlier kernels, reachable through the
  // disc_vail2 / disc_pg2 knobs only, take 32 inputs: their images are built for that width alone.
  const int n_in = d->n_in, nch = ceil_div(n_in, KC), kin = KC * nch;
  const bool all_kernels = n_in == DISC_IN;
  std::vector<float> w1((size_t)n1 * kin, 0.f);
  for (int r = 0; r < n1; ++r) std::memcpy(&w1[(size_t)r * kin], d->w1 + (size_t)r * n_in, sizeof(float) * n_in);
  std::vector<float> img;
  if (!vail || all_kernels) {
    for (int nb = 0; nb < n1 / 256; ++nb) {
      for (int ch = 0; ch < nch; ++ch) append_chunk(img, w1.data(), kin, nb * 256, 256, ch * KC);
      for (int c = 0; c < 8; ++c) append_chunk(img, d->w2, n1, 0, n2, nb * 256 + c * KC);
    }
  }
  if (vail && all_kernels) {
    std::vector<float> w3((size_t)2 * z * n2);                 // [mu; logvar] stacked: 2z rows x n2
    std::memcpy(w3.data(), d->wmu, sizeof(float) * z * n2);
    std::memcpy(w3.data() + (size_t)z * n2, d->wlv, sizeof(float) * z * n2);
    for (int c = 0; c < n2 / KC; ++c) append_chunk(img, w3.data(), n2, 0, 2 * z, c * KC);
  }
  std::vector<float> par;
  par.insert(par.end(), d->b1, d->b1 + n1);
  par.insert(par.end(), d->b2, d->b2 + n2);
  if (vail) {
    par.insert(par.end(), d->bmu, d->bmu + z);
    par.insert(par.end(), d->blv, d->blv + z);
  }
  par.insert(par.end(), d->wd, d->wd + (vail ? z : n2));
  par.push_back(d->bd[0]);
  // ---- 2-CTA-per-SM VAIL variant: 16-column chunks, every B block 128 rows, [mu; logvar] rows interleaved per 64
  std::vector<float> img2, par2;
  if (vail) {
    std::vector<float> w3i((size_t)2 * z * n2), b3i(2 * z);
    for (int hb = 0; hb < 2; ++hb)
      for (int r = 0; r < 64; ++r) {
        std::memcpy(&w3i[(size_t)(128 * hb + r) * n2], d->wmu + (size_t)(64 * hb + r) * n2, sizeof(float) * n2);
        std::memcpy(&w3i[(size_t)(128 * hb + 64 + r) * n2], d->wlv + (size_t)(64 * hb + r) * n2, sizeof(float) * n2);
        b3i[128 * hb + r] = d->bmu[64 * hb + r];
        b3i[128 * hb + 64 + r] = d->blv[64 * hb + r];
      }
    auto chunk16 = [&](const float* w, int ldw, int r0, int k0) {          // 128 rows x 16 columns: hi image, lo image
      const size_t base = img2.size();
      img2.resize(base + (size_t)V2_ROWS * V2_KC * 2);
      float* hi = img2.data() + base;
      float* lo = hi + (size_t)V2_ROWS * V2_KC;
      for (int kc = 0; kc < V2_KC / 4; ++kc)
        for (int r = 0; r < V2_ROWS; ++r)
          for (int e = 0; e < 4; ++e)
            split_tf32(w[(size_t)(r0 + r) * ldw + k0 + kc * 4 + e], hi + ((size_t)kc * V2_ROWS + r) * 4 + e,
                       lo + ((size_t)kc * V2_ROWS + r) * 4 + e);
    };
    if (all_kernels) {
      for (int blk = 0; blk < 2; ++blk) {
        for (int c = 0; c < 2; ++c) chunk16(d->w1, DISC_IN, 128 * blk, 16 * c);
        for (int c = 0; c < 8; ++c) chunk16(d->w2, n1, 0, 128 * blk + 16 * c);
      }
      for (int hb = 0; hb < 2; ++hb)
        for (int c = 0; c < 8; ++c) chunk16(w3i.data(), n2, 128 * hb, 16 * c);
    }
    par2.insert(par2.end(), d->b1, d->b1 + n1);
    par2.insert(par2.end(), d->b2, d->b2 + n2);
    par2.insert(par2.end(), b3i.begin(), b3i.end());
    par2.insert(par2.end(), d->wd, d->wd + z);
    par2.push_back(d->bd[0]);
  }
  // ---- VAIL with the A operand in TMEM (disc_vail3_kernel): 64-row blocks of layer 1 and of [mu; logvar] (rows
  //      interleaved per 32), 128-row chunks of layer 2, all 16 columns wide, in the kernel's issue order
  std::vector<float> img3, par3;
  if (vail && all_kernels) {
    std::vector<float> w3i((size_t)2 * z * n2), b3i(2 * z);
    for (int hb = 0; hb < 4; ++hb)
      for (int r = 0; r < 32; ++r) {
        std::memcpy(&w3i[(size_t)(64 * hb + r) * n2], d->wmu + (size_t)(32 * hb + r) * n2, sizeof(float) * n2);
        std::memcpy(&w3i[(size_t)(64 * hb + 32 + r) * n2], d->wlv + (size_t)(32 * hb + r) * n2, sizeof(float) * n2);
        b3i[64 * hb + r] = d->bmu[32 * hb + r];
        b3i[64 * hb + 32 + r] = d->blv[32 * hb + r];
      }
    auto chunk = [&](const float* w, int ldw, int r0, int rows, int k0) {       // rows x 16 columns: hi image, lo image
      const size_t base = img3.size();
      img3.resize(base + (size_t)rows * V3_KC * 2);
      float* hi = img3.data() + base;
      float* lo = hi + (size_t)rows * V3_KC;
      for (int kc = 0; kc < V3_KC / 4; ++kc)
        for (int r = 0; r < rows; ++r)
          for (int e = 0; e < 4; ++e)
            split_tf32(w[(size_t)(r0 + r) * ldw + k0 + kc * 4 + e], hi + ((size_t)kc * rows + r) * 4 + e,
                       lo + ((size_t)kc * rows + r) * 4 + e);
    };
    for (int blk = 0; blk < 4; ++blk) {
      for (int c = 0; c < 2; ++c) chunk(d->w1, DISC_IN, 64 * blk, 64, 16 * c);
      for (int c = 0; c < 4; ++c) chunk(d->w2, n1, 0, 128, 64 * blk + 16 * c);
    }
    for (int hb = 0; hb < 4; ++hb)
      for (int c = 0; c < 8; ++c) chunk(w3i.data(), n2, 64 * hb, 64, 16 * c);
    if (img3.size() * sizeof(float) != (size_t)V3_IMAGE_BYTES) return fail("om_disc_create: internal image size mismatch");
    par3.insert(par3.end(), d->b1, d->b1 + n1);
    par3.insert(par3.end(), d->b2, d->b2 + n2);
    par3.insert(par3.end(), b3i.begin(), b3i.end());
    par3.insert(par3.end(), d->wd, d->wd + z);
    par3.push_back(d->bd[0]);
  }
  // ---- VAIL, one CTA per SM, A operand in TMEM (disc_vail4_kernel): 2 nch + 16 chunks of 128 rows x 32 columns in MMA
  //      order; the [mu; logvar] rows interleaved per 64 exactly as for disc_vail2_kernel (whose parameter block it shares)
  std::vector<float> img4;
  if (vail) {
    std::vector<float> w3i((size_t)2 * z * n2);
    for (int hb = 0; hb < 2; ++hb)
      for (int r = 0; r < 64; ++r) {
        std::memcpy(&w3i[(size_t)(128 * hb + r) * n2], d->wmu + (size_t)(64 * hb + r) * n2, sizeof(float) * n2);
        std::memcpy(&w3i[(size_t)(128 * hb + 64 + r) * n2], d->wlv + (size_t)(64 * hb + r) * n2, sizeof(float) * n2);
      }
    auto chunk32 = [&](const float* w, int ldw, int r0, int k0) {          // 128 rows x 32 columns: hi image, lo image
      const size_t base = img4.size();
      img4.resize(base + (size_t)128 * V4_KC * 2);
      float* hi = img4.data() + base;
      float* lo = hi + (size_t)128 * V4_KC;
      for (int kc = 0; kc < V4_KC / 4; ++kc)
        for (int r = 0; r < 128; ++r)
          for (int e = 0; e < 4; ++e)
            split_tf32(w[(size_t)(r0 + r) * ldw + k0 + kc * 4 + e], hi + ((size_t)kc * 128 + r) * 4 + e,
                       lo + ((size_t)kc * 128 + r) * 4 + e);
    };
    for (int ch = 0; ch < nch; ++ch) {
      chunk32(w1.data(), kin, 0, KC * ch);
      chunk32(w1.data(), kin, 128, KC * ch);
    }
    for (int c = 0; c < 8; ++c) chunk32(d->w2, n1, 0, 32 * c);
    for (int c = 0; c < 4; ++c) {
      chunk32(w3i.data(), n2, 0, 32 * c);
      chunk32(w3i.data(), n2, 128, 32 * c);
    }
  }
  OmDisc* h = new OmDisc();
  h->sh = DiscShape{d->kind, n1, n2, z};
  h->n_in = n_in;
  cudaError_t e = cudaSuccess;
  auto upload = [&](const std::vector<float>& v, float** dst) {           // an image not built stays null
    if (e == cudaSuccess && !v.empty()) e = cudaMalloc(dst, v.size() * sizeof(float));
    if (e == cudaSuccess && !v.empty()) e = cudaMemcpy(*dst, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice);
  };
  upload(img, &h->image);
  upload(par, &h->params);
  upload(img2, &h->image2);
  upload(par2, &h->params2);
  upload(img3, &h->image3);
  upload(par3, &h->params3);
  upload(img4, &h->image4);
  if (e != cudaSuccess) {
    if (h->image) cudaFree(h->image);
    if (h->params) cudaFree(h->params);
    if (h->image2) cudaFree(h->image2);
    if (h->params2) cudaFree(h->params2);
    if (h->image3) cudaFree(h->image3);
    if (h->params3) cudaFree(h->params3);
    if (h->image4) cudaFree(h->image4);
    delete h;
    return fail("om_disc_create: device upload failed: %s (no CPU path)", cudaGetErrorString(e));
  }
  *out = h;
  return 0;
}

extern "C" void om_disc_destroy(OmDisc* h) {
  if (!h) return;
  if (h->image) cudaFree(h->image);
  cudaFree(h->params);
  if (h->image2) cudaFree(h->image2);
  if (h->params2) cudaFree(h->params2);
  if (h->image3) cudaFree(h->image3);
  if (h->params3) cudaFree(h->params3);
  if (h->image4) cudaFree(h->image4);
  delete h;
}

extern "C" int om_disc_reward(const OmDisc* h, const float* s, const float* mean, const float* stdv, const float* eps, int n,
                              int ld, float* reward, float* d_out, void* stream) {
  OM_REQUIRE(reward || n == 0, "om_disc_reward: null argument");
  return om_disc_forward(h, s, mean, stdv, eps, n, ld, reward, d_out, nullptr, stream);
}

extern "C" int om_disc_forward(const OmDisc* h, const float* s, const float* mean, const float* stdv, const float* eps, int n,
                               int ld, float* reward, float* d_out, float* kl_out, void* stream) {
  OM_REQUIRE(h, "om_disc_forward: null discriminator");
  OM_REQUIRE(n >= 0 && ld >= n, "om_disc_forward: need 0 <= n <= ld");
  if (n == 0) return 0;
  OM_REQUIRE(s && mean && stdv && (reward || d_out || kl_out), "om_disc_forward: null argument");
  OM_REQUIRE(!kl_out || h->sh.kind == 0, "om_disc_forward: the KL term exists for the variational (VAIL) network only");
  int dev = 0, sms = 0;
  OM_CUDA_OK(cudaGetDevice(&dev));
  OM_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int ntiles = ceil_div(n, TILE);
  const int grid = ntiles < sms ? ntiles : sms;                  // persistent: one CTA per SM
  const size_t smem = 2 * STAGE_A_BYTES + NSB * STAGE_B2_BYTES + (DISC_MAX_PAR + 4) * sizeof(float) + 12 * 8 + 16;
  DiscArgs a{h->sh, h->image, h->params, s, mean, stdv, eps, reward, d_out, kl_out, n, ld};
  cudaStream_t st = (cudaStream_t)stream;
  if (h->n_in != DISC_IN) {
    // another input width: the default kernels, built for one or two input chunks
    const bool knob = h->sh.kind == 0 ? !(g_knobs.disc_vail2 < 0 || g_knobs.disc_vail2 == 4) : g_knobs.disc_pg2 == 0;
    OM_REQUIRE(!knob, "om_disc_forward: the kernel variant the disc_vail2 / disc_pg2 knob selects takes %d inputs only, "
               "this network has %d", DISC_IN, h->n_in);
    DiscArgsIn aw;
    static_cast<DiscArgs&>(aw) = a;
    aw.n_in = h->n_in;
    const bool two_ch = h->n_in > KC;
    if (h->sh.kind == 0) {
      aw.image = h->image4;
      aw.params = h->params2;
      const size_t smem4 = v4_smem(two_ch ? 2 : 1);
      auto kern = two_ch ? (kl_out ? disc_vail4_kernel<true, 0, 2> : disc_vail4_kernel<false, 0, 2>)
                         : (kl_out ? disc_vail4_kernel<true, 0, 1> : disc_vail4_kernel<false, 0, 1>);
      OM_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4));
      kern<<<grid, 320, smem4, st>>>(aw);
    } else {
      const size_t smem_pg2 = smem + 2 * 128 * sizeof(float);         // the standardiser slots lie inside DISC_MAX_PAR
      auto kern = two_ch ? disc_reward_pg2_kernel<512, 256, false, false, 2> : disc_reward_pg2_kernel<512, 256, false, false, 1>;
      OM_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pg2));
      kern<<<grid, 320, smem_pg2, st>>>(aw);
    }
    OM_LAUNCHED();
    return 0;
  }
  // VAIL: two CTAs per SM.  (The two-producer-group kernel below is 3 % faster at 65536 samples when timed alone -- 73.4
  // vs 76.3 us -- but 15 % slower inside bench.py's process, after the large-buffer measurements: 88.8 us; the two-CTA
  // kernel reads 76-78 us in both settings, so it stays the default.)
  int two = h->sh.kind == 0;
  if (g_knobs.disc_vail2 >= 0) two = h->sh.kind == 0 && g_knobs.disc_vail2 != 0;           // tuning / test hook: force either
  // VAIL default: disc_vail4_kernel (one CTA per SM, A operand in TMEM): 69 us at 65536 samples / 796 us at 1 M against 74 /
  // 815 for the two-CTA shared-memory kernel (knob 1), 82 / 975 for the two-CTA TMEM kernel (knob 3), 72 / 841 for the
  // two-producer-group shared-memory kernel (knob 0)
  if (h->sh.kind == 0 && (g_knobs.disc_vail2 == 4 || g_knobs.disc_vail2 == 5 || g_knobs.disc_vail2 == 6 || g_knobs.disc_vail2 == 7 ||
                            g_knobs.disc_vail2 < 0)) {
    const size_t smem4 = v4_smem(1);
    const int rot = g_knobs.disc_vail2 == 5 ? 2 : g_knobs.disc_vail2 == 6 ? 1 : g_knobs.disc_vail2 == 7 ? 3 : 0;
    DiscArgs a4 = a;
    a4.image = h->image4;
    a4.params = h->params2;
    auto kern = rot == 3 ? (kl_out ? disc_vail4_kernel<true, 3> : disc_vail4_kernel<false, 3>)
              : rot == 2 ? (kl_out ? disc_vail4_kernel<true, 2> : disc_vail4_kernel<false, 2>)
              : rot == 1 ? (kl_out ? disc_vail4_kernel<true, 1> : disc_vail4_kernel<false, 1>)
                         : (kl_out ? disc_vail4_kernel<true, 0> : disc_vail4_kernel<false, 0>);
    OM_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4));
    kern<<<grid, 320, smem4, st>>>(a4);
    OM_LAUNCHED();
    return 0;
  }
  if (h->sh.kind == 0 && g_knobs.disc_vail2 == 3) {            // A operand in TMEM (opt-in: measured slower, see the kernel)
    const size_t smem3 = V3_NSB * V3_STAGE_B + (V3_NPAR + 3 + 2 * DISC_IN) * sizeof(float) + (2 * V3_NSA + 2 * V3_NSB) * 8 + 16;
    const int grid3 = ntiles < 2 * sms ? ntiles : 2 * sms;
    DiscArgs a3 = a;
    a3.image = h->image3;
    a3.params = h->params3;
    auto kern = kl_out ? disc_vail3_kernel<true> : disc_vail3_kernel<false>;
    OM_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem3));
    kern<<<grid3, 192, smem3, st>>>(a3);
    OM_LAUNCHED();
    return 0;
  }
  if (two) {
    const size_t smem2 = V2_NS * V2_STAGE_BYTES + (V2_NPAR + 3 + 2 * DISC_IN) * sizeof(float) + 3 * V2_NS * 8 + 16;
    const int grid2 = ntiles < 2 * sms ? ntiles : 2 * sms;
    DiscArgs a2 = a;
    a2.image = h->image2;
    a2.params = h->params2;
    auto kern = kl_out ? disc_vail2_kernel<true> : disc_vail2_kernel<false>;
    OM_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
    kern<<<grid2, 192, smem2, st>>>(a2);
    OM_LAUNCHED();
    return 0;
  }
  int pg2 = 1;                                                      // two producer warpgroups per CTA
  if (g_knobs.disc_pg2 >= 0) pg2 = g_knobs.disc_pg2 != 0;                        // tuning / test hook
  if (pg2) {
    const size_t smem_pg2 = smem + 2 * 128 * sizeof(float);
    if (h->sh.kind == 0) {
      auto kern = kl_out ? disc_reward_pg2_kernel<256, 128, true, true> : disc_reward_pg2_kernel<256, 128, true, false>;
      OM_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pg2));
      kern<<<grid, 320, smem_pg2, st>>>(a);
    } else {
      OM_CUDA_OK(cudaFuncSetAttribute(disc_reward_pg2_kernel<512, 256, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_pg2));
      disc_reward_pg2_kernel<512, 256, false, false><<<grid, 320, smem_pg2, st>>>(a);
    }
    OM_LAUNCHED();
    return 0;
  }
  if (h->sh.kind == 0) {
    auto kern = kl_out ? disc_reward_kernel<256, 128, true, true> : disc_reward_kernel<256, 128, true, false>;
    OM_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, 192, smem, st>>>(a);
  } else {
    OM_CUDA_OK(cudaFuncSetAttribute(disc_reward_kernel<512, 256, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    disc_reward_kernel<512, 256, false, false><<<grid, 192, smem, st>>>(a);
  }
  OM_LAUNCHED();
  return 0;
}
