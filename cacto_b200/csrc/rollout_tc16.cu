// rollout_tc16.cu -- K1 on tcgen05 with fp16 operand splitting, persistent CTAs and two free-running tile pipelines.
//
// Same fused actor + dynamics rollout as rollout.cu / rollout_tc.cu (RL.py:197-233, NeuralNetwork.py:51-63,130-138,
// environment.py:80-91).  The 256x256 hidden layer runs on tcgen05.mma kind::f16 (fp32 accumulation in TMEM) with
//     a' = S_a a = a_hi + a_lo,   w' = S_w w = w_hi + w_lo      (each part fp16: 11 significant bits)
//     a' w' ~= a_hi w_hi + a_hi w_lo + a_lo w_hi                (error ~2^-21 relative, the class of 3xTF32)
// at the fp16 rate, i.e. twice the tf32 rate of rollout_tc.cu.  S_a = 32 is folded into the shared-memory copy of
// (W1, b1) (LeakyReLU is positively homogeneous, power-of-two scaling is exact); S_w = 2^s brings max|W2| into
// [2^13, 2^14) so that the low parts stay fp16-normal; the epilogue multiplies the accumulator by 1 / (S_a S_w).
// Range limit of this engine: a hidden activation beyond +-2047 overflows its fp16 high part -> the action becomes
// non-finite -> the rollout is flagged failed (success = 0); the 'fma' engine has no such limit.
// Systems: the five with at most 8 inputs and 3 actions (single / double integrator, car, car_park, manipulator); UR5
// (13 inputs, 6 actions) runs on the 3xTF32 kernel of rollout_tc.cu, where its fp64 dynamics, not the actor, set the time.
//
// One persistent CTA per SM owns a contiguous range of 128-rollout tiles and runs two independent tile pipelines
// ("slots") that share the tensor pipe and one W2 stream:
//   warps 0-3 / 4-7  workers of slot 0 / 1 (128 threads per tile).  Shared-memory bandwidth is the scarce resource of this
//                    kernel (ncu: LSU + tensor-core wavefronts at 82 % of the data pipe with one thread per row), so both
//                    worker phases are register-tiled over rows to amortise the broadcast loads of the small weights:
//                    * layer 1 (K = ns, CUDA cores, packed FFMA2): per 16-unit K-chunk a thread computes 4 rows x 4 units
//                      (one LDS.128 of W1 per input serves 4 rows), LeakyReLU, hi/lo split, 8-byte stores into the slot's
//                      A stage (UMMA K-major no-swizzle layout, conflict-free);
//                    * epilogue: tcgen05.ld.16x256b hands a thread 4 rows x 2 columns per 8-column block, so one load of
//                      (b2, W3) per column pair serves 4 rows; bias + LeakyReLU + layer 3 as per-thread partial sums, then a
//                      two-stage shuffle butterfly leaves every thread with the 3 actions of ONE row;
//                    * that thread advances the fp64 dynamics of its row, stores the SoA trajectory and publishes the
//                      normalised fp32 state for the next layer-1 pass (8 KB exchange buffer + one 128-thread barrier).
//   warp 8 / 9       MMA issuer of slot 0 / 1 (one lane): 3 x tcgen05.mma M128 N256 K16 per chunk; tcgen05.commit
//                    recycles the A stage, publishes the accumulator and releases the W2 ring slot.
//   warp 10          TMA producer (one lane): streams the pre-split W2 image (16 chunks x 16 KB) from L2 into a
//                    T16_RING-slot ring with cp.async.bulk; both slots consume every chunk.
// Slot 1 starts its steps 8 chunks (half a step) after slot 0 -- its K-chunks are visited in the rotated order
// 8..15,0..7, accumulation is commutative -- so that the epilogue + dynamics of one slot overlaps the MMAs of the other.
#include <cuda_fp16.h>
#include "common.cuh"
#include "mlp.cuh"
#include "systems.cuh"

namespace cacto {

constexpr int T16_TILE = 128;                      // rollouts per UMMA tile (M)
constexpr int T16_SLOTS = 2;                       // tile pipelines per CTA (2 x 256 TMEM columns)
constexpr int T16_WORKERS = T16_TILE * T16_SLOTS;  // 256 worker threads
constexpr int T16_THREADS = T16_WORKERS + 96;      // + 2 issuer warps + producer warp
constexpr int T16_KC = 16;                         // hidden units per K-chunk = one kind::f16 UMMA k-step
constexpr int T16_NCHUNK = ACTOR_H / T16_KC;       // 16
constexpr int T16_HALF = T16_NCHUNK / 2;           // slot 1 lags by half a step
constexpr int T16_STAGES = 4;                      // A stages per slot (divides T16_NCHUNK: stage and phase of a chunk are compile-time in the issuer)
constexpr int T16_RING = 8;                        // W2 ring slots = half a step: ring slot and phase of a chunk are compile-time in the issuer
constexpr int T16_A_IMG = T16_TILE * T16_KC * 2;   // bytes of one A image (hi or lo): 4 KB
constexpr int T16_B_IMG = ACTOR_H * T16_KC * 2;    // bytes of one W2 image (hi or lo) of a chunk: 8 KB
constexpr int T16_IMG_BYTES = T16_NCHUNK * 2 * T16_B_IMG;   // 256 KB
constexpr int T16_TRAILER = 64;                    // [0] u32 max|W2| bits, [1] f32 1/(S_a S_w), [2] f32 S_w
constexpr int T16_MAXT = 512;                      // tiles per CTA that the per-tile horizon table holds
constexpr int T16_MAX_NS = 8;                      // inputs a row publishes in the state exchange (layer-1 register tile)
constexpr int T16_MAX_NA = 3;                      // actions the epilogue's head table holds
constexpr float T16_SA = 32.f;

template <int NS>
struct Tc16Smem {
  alignas(1024) unsigned char B[T16_RING][2 * T16_B_IMG];              // W2 ring: [slot][hi | lo]           128 KB
  alignas(1024) unsigned char A[T16_SLOTS][T16_STAGES][2 * T16_A_IMG]; // A stages: [slot][stage][hi | lo]    64 KB
  alignas(16) float W1[NS][ACTOR_H];                                   // S_a * W1                           3-7 KB
  alignas(16) float b1[ACTOR_H];                                       // S_a * b1
  alignas(16) float head[ACTOR_H / 2][8];   // per column pair (c, c+1): b2 | W3[.][0] | W3[.][1] | W3[.][2]    4 KB
  alignas(16) float4 xn[T16_SLOTS][T16_MAX_NS / 4][T16_TILE];          // normalised fp32 states of the step (row -> layer-1 threads) 8 KB
  float b3[8];
  // the issuer handles K-chunks in pairs: W2 ring slots and A stages are released (and W2 is loaded) two at a time
  uint64_t b_full[T16_RING / 2], b_empty[T16_RING / 2];
  uint64_t a_full[T16_SLOTS][T16_STAGES], a_empty[T16_SLOTS][T16_STAGES / 2], d_full[T16_SLOTS], start1;
  uint32_t tmem_base;
  int tile_tmax[T16_MAXT];
};

__device__ __forceinline__ void t16_mbar_init(uint64_t* b, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count));
}
__device__ __forceinline__ void t16_mbar_arrive(uint64_t* b) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ bool t16_mbar_try(uint32_t mb, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(mb), "r"(parity)
      : "memory");
  return done != 0;
}
#ifndef T16_WAIT_HINT_NS
#define T16_WAIT_HINT_NS 20000
#endif
__device__ __noinline__ void t16_mbar_wait_slow(uint32_t mb, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  unsigned long long t0 = 0;
  while (true) {
    // try_wait with a time hint suspends the thread in hardware (ns): waiting roles do not steal issue slots
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(mb), "r"(parity), "r"((uint32_t)T16_WAIT_HINT_NS)
        : "memory");
    if (done) break;
    if ((++spins & 1023u) == 0) {              // fail loudly instead of hanging the GPU: trap after 4 s
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000ull) __trap();
    }
  }
}
__device__ __forceinline__ void t16_mbar_wait(uint64_t* b, uint32_t parity) {
  const uint32_t mb = smem_u32(b);
  if (!t16_mbar_try(mb, parity)) t16_mbar_wait_slow(mb, parity);     // the common case (already complete) is one instruction
}
// one lane of a converged warp (the MMA / TMA roles run warp-converged on warp-uniform values so that the compiler keeps the
// UMMA descriptors and barrier addresses in uniform registers instead of wrapping every instruction in a per-lane loop)
__device__ __forceinline__ bool t16_elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void t16_commit(uint64_t* b) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(b)) : "memory");
}
// K-major, no swizzle: 16-byte units of 8 consecutive k; 8 rows x 16 B = one 128-byte core matrix; consecutive 8-row
// groups are SBO = 128 B apart, the next k-unit is LBO = (rows / 8) * 128 B away.
__device__ __forceinline__ uint64_t t16_desc(uint32_t saddr, uint32_t lbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t)(128u >> 4) << 32) | ((uint64_t)1 << 46);
}
__device__ __forceinline__ void t16_umma(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
__host__ __device__ constexpr int t16_b_offset(int n, int kk) {       // byte offset of B[n][kk] inside one chunk image
  return (kk >> 3) * (ACTOR_H / 8) * 128 + (n >> 3) * 128 + (n & 7) * 16 + (kk & 7) * 2;
}

// packed fp32 pairs (Blackwell FFMA2 / FMUL2: two lanes per issue slot)
__device__ __forceinline__ uint64_t pk(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void upk(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {      // (lo, hi) -> f16x2, lo in the low half
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// ---------------------------------------------------------------------------------------------------------------
// W2 image: max|W2| -> S_w, then per chunk [hi image | lo image] of B[n][kk] = S_w W2[16 kc + kk][n].
__global__ void __launch_bounds__(256) k_tc16_absmax(const float* __restrict__ actor, int ns, int na, unsigned char* __restrict__ img) {
  const ActorLayout L(ns, na);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t m = (i < ACTOR_H * ACTOR_H) ? (__float_as_uint(actor[L.W2 + i]) & 0x7fffffffu) : 0u;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<uint32_t*>(img + T16_IMG_BYTES), m);
}

__device__ __forceinline__ float t16_w_scale(uint32_t maxbits) {
  const int e = (int)(maxbits >> 23);                  // biased exponent of max|W2|
  if (e == 0 || e == 255) return 1.f;                  // zero / subnormal / non-finite weights: no scaling
  int s = 13 - (e - 127);
  s = max(-60, min(60, s));
  return __uint_as_float((uint32_t)(s + 127) << 23);
}

__global__ void __launch_bounds__(256) k_tc16_prepare(const float* __restrict__ actor, int ns, int na, unsigned char* __restrict__ img) {
  const ActorLayout L(ns, na);
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ACTOR_H * ACTOR_H) return;
  const float sw = t16_w_scale(*reinterpret_cast<const uint32_t*>(img + T16_IMG_BYTES));
  const int k = i / ACTOR_H, n = i - k * ACTOR_H;          // coalesced read of W2[k][n]
  const float w = actor[L.W2 + i] * sw;
  const __half hi = __float2half_rn(w);
  const __half lo = __float2half_rn(w - __half2float(hi));
  const int kc = k / T16_KC, kk = k - kc * T16_KC;
  unsigned char* base = img + (size_t)kc * 2 * T16_B_IMG + t16_b_offset(n, kk);
  *reinterpret_cast<__half*>(base) = hi;
  *reinterpret_cast<__half*>(base + T16_B_IMG) = lo;
  if (i == 0) {
    float* tr = reinterpret_cast<float*>(img + T16_IMG_BYTES);
    tr[1] = 1.f / (T16_SA * sw);
    tr[2] = sw;
  }
}

#ifdef T16_TRACE   // debug builds only (profiles/scripts/): per-role event timeline of CTA 0 (code in the low byte, clock64 above)
__device__ long long* g_t16_trace = nullptr;
constexpr int T16_TRACE_N = 8192;
#define T16_EV(role, code)                                                                                       \
  do {                                                                                                           \
    if (blockIdx.x == 0 && g_t16_trace != nullptr && trace_n < T16_TRACE_N)                                      \
      g_t16_trace[(role) * T16_TRACE_N + trace_n++] = (clock64() << 8) | (long long)(code);                      \
  } while (0)
#else
#define T16_EV(role, code) do { } while (0)
#endif

// ---------------------------------------------------------------------------------------------------------------
// tcgen05.ld.16x256b.x2: 16 TMEM lanes x 16 columns.  Register 4k + 2rh + e of thread t holds lane (t / 4 + 8 rh),
// column 8k + 2 (t % 4) + e  (k = 0..1; layout verified on B200 with profiles/scripts/ldtm_test.cu).
#define T16_LDTM_16x256_X2(v, taddr)                                                                     \
  asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"                 \
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]) \
               : "r"(taddr))

template <int SYS>
__global__ void __launch_bounds__(T16_THREADS, 1) k_rollout_tc16(const __grid_constant__ cacto_sys_params P, const float* __restrict__ actor,
                                                                 const unsigned char* __restrict__ w2img, const double* __restrict__ ics,
                                                                 const int32_t* __restrict__ horizon, int T_max, double* __restrict__ states,
                                                                 double* __restrict__ controls, int32_t* __restrict__ flags,
                                                                 double* __restrict__ rewards, int64_t B, int ntiles) {
  constexpr int NX = SysDims<SYS>::NX, NA = SysDims<SYS>::NA, NS = NX + 1;
  constexpr int WORKERS = T16_WORKERS, THREADS = T16_THREADS;
  static_assert(NS <= T16_MAX_NS, "the state exchange and the layer-1 register tile hold at most 8 inputs");
  static_assert(NA <= T16_MAX_NA, "the epilogue's head table holds at most 3 actions");
  using Smem = Tc16Smem<NS>;
  static_assert(T16_NCHUNK % T16_STAGES == 0 && T16_NCHUNK % T16_RING == 0 && T16_HALF % T16_RING == 0, "compile-time stage / ring indices");
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
  const ActorLayout L(NS, NA);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;      // warp: provably warp-uniform
  const bool worker = tid < WORKERS;
  // contiguous, balanced tile range of this CTA; slot m takes tiles tile_lo + m, tile_lo + m + 2, ...
  const int tile_lo = (int)(((int64_t)blockIdx.x * ntiles) / gridDim.x), tile_hi = (int)(((int64_t)(blockIdx.x + 1) * ntiles) / gridDim.x);
  const int my_tiles = tile_hi - tile_lo;

  // ---- one-time setup: small weights to shared memory (layer 1 pre-scaled by S_a), barriers, TMEM, per-tile horizons
  for (int i = tid; i < NS * ACTOR_H; i += THREADS) sm.W1[i / ACTOR_H][i % ACTOR_H] = T16_SA * actor[L.W1 + i];
  for (int c = tid; c < ACTOR_H; c += THREADS) {
    sm.b1[c] = T16_SA * actor[L.b1 + c];
    float* h = &sm.head[c >> 1][c & 1];
    h[0] = actor[L.b2 + c];
#pragma unroll
    for (int j = 0; j < 3; ++j) h[2 + 2 * j] = (j < NA) ? actor[L.W3 + c * NA + j] : 0.f;
  }
  if (tid < 8) sm.b3[tid] = tid < NA ? actor[L.b3 + tid] : 0.f;
  for (int i = tid; i < my_tiles; i += THREADS) sm.tile_tmax[i] = 0;
  if (tid == 0) {
    for (int s = 0; s < T16_RING / 2; ++s) { t16_mbar_init(&sm.b_full[s], 1); t16_mbar_init(&sm.b_empty[s], 2); }
    for (int m = 0; m < T16_SLOTS; ++m) {
      for (int s = 0; s < T16_STAGES; ++s) t16_mbar_init(&sm.a_full[m][s], T16_TILE / 2);
      for (int s = 0; s < T16_STAGES / 2; ++s) t16_mbar_init(&sm.a_empty[m][s], 1);
      t16_mbar_init(&sm.d_full[m], 1);
    }
    t16_mbar_init(&sm.start1, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == WORKERS / 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sm.tmem_base)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  __syncthreads();
  for (int64_t i = tid; i < (int64_t)my_tiles * T16_TILE; i += THREADS) {
    const int64_t b = (int64_t)tile_lo * T16_TILE + i;
    if (b < B) atomicMax(&sm.tile_tmax[i / T16_TILE], min(max(horizon[b], 0), T_max));
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = sm.tmem_base;
  const float inv_scale = reinterpret_cast<const float*>(w2img + T16_IMG_BYTES)[1];

  // steps of each slot, and the chunk range [g_begin, g_end) of the W2 stream that slot m consumes
  int N[T16_SLOTS] = {0, 0};
  for (int i = 0; i < my_tiles; ++i) N[i & 1] += sm.tile_tmax[i];
  const int off1 = N[0] > 0 ? T16_HALF : 0;
  const int g_begin[T16_SLOTS] = {0, off1}, g_end[T16_SLOTS] = {T16_NCHUNK * N[0], off1 + T16_NCHUNK * N[1]};
  const int g_total = max(g_end[0], g_end[1]);

  if (worker) {
    // =================================================================== workers
    const int m = tid / T16_TILE, w = (tid % T16_TILE) >> 5;          // slot; warp within the slot = TMEM lane quadrant
    const int l4 = lane >> 2, l3 = lane & 3;
    // epilogue / dynamics: after the butterfly this thread owns row 32 w + l4 + 8 isel of the tile
    const int isel = 2 * (lane & 1) + ((lane >> 1) & 1);
    const int row = 32 * w + l4 + 8 * isel;
    // layer 1: warps (0,1) of the slot produce the even chunks, warps (2,3) the odd ones; warp w computes the 8 units of
    // k-unit w & 1 for the rows lane + 32 i (i = 0..3): W1 loads are warp-uniform, the 16-byte A stores conflict-free
    const int l1_par = w >> 1, l1_ku = w & 1;
    unsigned char* const a_dst0 = &sm.A[m][0][0] + l1_ku * (T16_TILE / 8) * 128 + (lane >> 3) * 128 + (lane & 7) * 16;   // row lane; row lane + 32 i: + 512 i
    const uint32_t d_taddr = tmem + ((uint32_t)(32 * w) << 16) + (uint32_t)(m * ACTOR_H);
    const uint64_t inv2 = pk(inv_scale, inv_scale), alpha2 = pk(LEAKY_ALPHA, LEAKY_ALPHA);
    int q = 0, dstep = 0;                       // chunks produced / steps finished by this slot so far
#ifdef T16_TRACE
    int trace_n = 0;
    const bool tr = (tid % T16_TILE) == 0;
#define WEV(code) do { if (tr) T16_EV(m, code); } while (0)
#else
#define WEV(code) do { } while (0)
#endif
    if (m == 1 && N[0] > 0 && N[1] > 0) t16_mbar_wait(&sm.start1, 0);
    for (int ti = m; ti < my_tiles; ti += T16_SLOTS) {
      const int tmax = sm.tile_tmax[ti];
      const int64_t b = (int64_t)(tile_lo + ti) * T16_TILE + row;
      const bool owner = b < B;
      double x[NS];
      int h = 0, ok = 1;
      if (owner) {
#pragma unroll
        for (int j = 0; j < NS; ++j) {
          x[j] = ics[b * NS + j];
          states[(int64_t)j * B + b] = x[j];
        }
        h = min(max(horizon[b], 0), T_max);
      }
      for (int t = 0; t < tmax; ++t) {
        const bool live = owner && ok && t < h;
        WEV(1);                                  // step start
        // ---- publish the normalised state of my row, fetch those of my four layer-1 rows
        {
          float xo[T16_MAX_NS];
#pragma unroll
          for (int j = 0; j < T16_MAX_NS; ++j) xo[j] = 0.f;
#pragma unroll
          for (int j = 0; j < NS; ++j) xo[j] = live ? normalize_component(P, j, (float)x[j]) : 0.f;
#pragma unroll
          for (int v = 0; v < T16_MAX_NS / 4; ++v) sm.xn[m][v][row] = make_float4(xo[4 * v], xo[4 * v + 1], xo[4 * v + 2], xo[4 * v + 3]);
        }
        asm volatile("bar.sync %0, 128;" ::"r"(1 + m) : "memory");
        float xn[4][NS];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
          for (int v = 0; v < T16_MAX_NS / 4; ++v) {
            const float4 f = sm.xn[m][v][lane + 32 * i];
            if (4 * v + 0 < NS) xn[i][(4 * v + 0) % NS] = f.x;
            if (4 * v + 1 < NS) xn[i][(4 * v + 1) % NS] = f.y;
            if (4 * v + 2 < NS) xn[i][(4 * v + 2) % NS] = f.z;
            if (4 * v + 3 < NS) xn[i][(4 * v + 3) % NS] = f.w;
          }
        }
        // ---- layer 1 into the A stages: every other chunk, 4 rows x 8 units per thread
#pragma unroll 1
        for (int kc = l1_par; kc < T16_NCHUNK; kc += 2) {
          const int qc = q + kc;                                          // this chunk's index in the slot's chunk sequence
          const int ci = (g_begin[m] + kc) & (T16_NCHUNK - 1);            // slot 1 visits the chunks in rotated order
          const int st = qc % T16_STAGES;
          const int c = ci * T16_KC + 8 * l1_ku;
          const ulonglong2 bA = *reinterpret_cast<const ulonglong2*>(&sm.b1[c]), bB = *reinterpret_cast<const ulonglong2*>(&sm.b1[c + 4]);
          unsigned char* dst = a_dst0 + st * (2 * T16_A_IMG);
          auto finish_row = [&](int i, const uint64_t (&z)[4]) {              // LeakyReLU, hi / lo split, 16-byte stores of row lane + 32 i
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int p = 0; p < 4; ++p) {
              float z0, z1, s0, s1;
              upk(z[p], z0, z1);
              upk(mul2(z[p], alpha2), s0, s1);
              const float a0 = fmaxf(z0, s0), a1 = fmaxf(z1, s1);          // LeakyReLU(0.3) = max(z, 0.3 z)
              const float h0 = __uint_as_float(__float_as_uint(a0) & 0xffffe000u), h1 = __uint_as_float(__float_as_uint(a1) & 0xffffe000u);
              hi[p] = pack_h2(h0, h1);
              lo[p] = pack_h2(a0 - h0, a1 - h1);
            }
            *reinterpret_cast<uint4*>(dst + 512 * i) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(dst + 512 * i + T16_A_IMG) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          };
          // all of W1's chunk columns in registers (8 registers per input), rows one after the other
          ulonglong2 wA[NS], wB[NS];
#pragma unroll
          for (int j = 0; j < NS; ++j) {
            wA[j] = *reinterpret_cast<const ulonglong2*>(&sm.W1[j][c]);
            wB[j] = *reinterpret_cast<const ulonglong2*>(&sm.W1[j][c + 4]);
          }
          WEV(2);                                  // chunk: W1 loaded, about to wait for the stage
          if (qc >= T16_STAGES) t16_mbar_wait(&sm.a_empty[m][st >> 1], (uint32_t)((qc / T16_STAGES - 1) & 1));   // stage pair (st >> 1) of chunk pair qc / 2
          WEV(3);                                  // stage free
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            uint64_t z[4] = {bA.x, bA.y, bB.x, bB.y};
#pragma unroll
            for (int j = 0; j < NS; ++j) {
              const uint64_t xj = pk(xn[i][j], xn[i][j]);
              z[0] = fma2(xj, wA[j].x, z[0]); z[1] = fma2(xj, wA[j].y, z[1]);
              z[2] = fma2(xj, wB[j].x, z[2]); z[3] = fma2(xj, wB[j].y, z[3]);
            }
            finish_row(i, z);
          }
#ifndef T16_EXP_NO_FENCE      // timing experiment only
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy stores -> visible to the UMMA (async proxy)
#endif
          t16_mbar_arrive(&sm.a_full[m][st]);
          WEV(4);                                // chunk published
        }
        q += T16_NCHUNK;
        WEV(5);                                  // waiting for the accumulator
        // ---- epilogue: per 16-column block a thread holds 4 rows x 2 column pairs; scale + bias, LeakyReLU, layer 3 as
        //      per-thread partial sums (even / odd column lanes of the packed accumulators); next block's TMEM load in flight
        t16_mbar_wait(&sm.d_full[m], (uint32_t)(dstep & 1));
        ++dstep;
        WEV(6);                                  // accumulator ready
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        uint64_t acc2[4][NA];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < NA; ++j) acc2[i][j] = pk(0.f, 0.f);
        uint32_t va[2][8], vb[2][8];
        T16_LDTM_16x256_X2(va[0], d_taddr);
        T16_LDTM_16x256_X2(va[1], d_taddr + (16u << 16));
        auto consume = [&](const uint32_t (&v)[2][8], int c0) {
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            const int pair = (c0 + 8 * k) / 2 + l3;
            const ulonglong2 hA = *reinterpret_cast<const ulonglong2*>(&sm.head[pair][0]);   // b2 pair | W3[.][0] pair
            const ulonglong2 hB = *reinterpret_cast<const ulonglong2*>(&sm.head[pair][4]);   // W3[.][1] pair | W3[.][2] pair
#pragma unroll
            for (int i = 0; i < 4; ++i) {                                     // row l4 + 8 i: half hl = i / 2, row half rh = i % 2
              const uint32_t* r = &v[i >> 1][4 * k + 2 * (i & 1)];
              const uint64_t zz = fma2(pk(__uint_as_float(r[0]), __uint_as_float(r[1])), inv2, hA.x);
              float z0, z1, s0, s1;
              upk(zz, z0, z1);
              upk(mul2(zz, alpha2), s0, s1);
              const uint64_t hv = pk(fmaxf(z0, s0), fmaxf(z1, s1));
              acc2[i][0] = fma2(hv, hA.y, acc2[i][0]);
              if (NA > 1) acc2[i][1] = fma2(hv, hB.x, acc2[i][1]);
              if (NA > 2) acc2[i][2] = fma2(hv, hB.y, acc2[i][2]);
            }
          }
        };
#pragma unroll 1
        for (int c0 = 0; c0 < ACTOR_H; c0 += 32) {
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          T16_LDTM_16x256_X2(vb[0], d_taddr + (uint32_t)(c0 + 16));
          T16_LDTM_16x256_X2(vb[1], d_taddr + (16u << 16) + (uint32_t)(c0 + 16));
          consume(va, c0);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (c0 + 32 < ACTOR_H) {
            T16_LDTM_16x256_X2(va[0], d_taddr + (uint32_t)(c0 + 32));
            T16_LDTM_16x256_X2(va[1], d_taddr + (16u << 16) + (uint32_t)(c0 + 32));
          }
          consume(vb, c0 + 16);
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");    // my TMEM reads precede the next step's MMAs (ordered via a_full)
        WEV(7);                                  // epilogue done
        // ---- butterfly over the 4 lanes that share these rows: 4 rows x NA partial sums -> the NA actions of row `row`
        float act[NA];
        {
          float p[4][NA];
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < NA; ++j) {
              float e, o;
              upk(acc2[i][j], e, o);
              p[i][j] = e + o;
            }
          const bool odd = lane & 1, up = lane & 2;
          float s1[2][NA];
#pragma unroll
          for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int j = 0; j < NA; ++j) {
              const float send = odd ? p[r][j] : p[r + 2][j];                // even lanes keep rows 0,1; odd lanes keep rows 2,3
              const float keep = odd ? p[r + 2][j] : p[r][j];
              s1[r][j] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
            }
#pragma unroll
          for (int j = 0; j < NA; ++j) {
            const float send = up ? s1[0][j] : s1[1][j];
            const float keep = up ? s1[1][j] : s1[0][j];
            act[j] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
          }
        }
        // ---- dynamics of my row
        if (live) {
          double u[NA], xnext[NS];
#pragma unroll
          for (int j = 0; j < NA; ++j) {
            u[j] = (double)(sm.b3[j] + act[j]);
            controls[((int64_t)t * NA + j) * B + b] = u[j];
          }
          if (rewards != nullptr) rewards[(int64_t)t * B + b] = sys_reward<SYS, double>(P, P.w_running, x, u, false);
          sys_step<SYS, double>(P, x, u, xnext);
          xnext[NX] = x[NX] + P.dt;
          bool nan = false;
#pragma unroll
          for (int j = 0; j < NS; ++j) {
            x[j] = xnext[j];
            nan |= (xnext[j] != xnext[j]);
            states[((int64_t)(t + 1) * NS + j) * B + b] = xnext[j];
          }
          if (nan) ok = 0;
          if (rewards != nullptr && t + 1 == h && !nan)
            rewards[(int64_t)(t + 1) * B + b] = sys_reward<SYS, double>(P, P.w_terminal, x, (const double*)nullptr, false);
        }
        WEV(8);                                  // dynamics done
      }
      if (owner) flags[b] = ok;
    }
  } else if (warp < WORKERS / 32 + T16_SLOTS) {
    // =================================================================== MMA issuer of slot m (warp-converged, one elected lane issues)
    const int m = warp - WORKERS / 32, o = 1 - m;
    const int gb = __shfl_sync(0xffffffffu, g_begin[m], 0), ge = __shfl_sync(0xffffffffu, g_end[m], 0);
    const int ob = __shfl_sync(0xffffffffu, g_begin[o], 0), oe = __shfl_sync(0xffffffffu, g_end[o], 0);
    constexpr uint32_t idesc = (1u << 4) | ((uint32_t)(ACTOR_H >> 3) << 17) | ((uint32_t)(T16_TILE >> 4) << 24);   // f16 x f16 -> f32, K-major
    constexpr uint32_t lboA = (T16_TILE / 8) * 128, lboB = (ACTOR_H / 8) * 128;
    const uint32_t d = tmem + (uint32_t)(m * ACTOR_H);
    const uint32_t a_base = smem_u32(&sm.A[m][0][0]), b_base = smem_u32(&sm.B[0][0]);
    const uint32_t pb0 = (uint32_t)(gb / T16_RING) & 1u;             // ring phase of this slot's first chunk (gb is 0 or T16_HALF, a multiple of T16_RING)
#ifdef T16_TRACE
    int trace_n = 0;
#endif
    // K-chunks are issued in pairs (one fence / elect / two commits per 6 UMMAs): the issuer warp shares its scheduler with two
    // busy worker warps and retires an instruction only every ~24 cycles, so its instruction count per chunk IS its chunk time.
    // The barrier polls of pair kp + 1 are issued before the UMMA block of pair kp.
    constexpr int NPAIR = T16_NCHUNK / 2, RPAIR = T16_RING / 2, SPAIR = T16_STAGES / 2;
    bool rdy_b = t16_mbar_try(smem_u32(&sm.b_full[0]), pb0);
    bool rdy_a0 = t16_mbar_try(smem_u32(&sm.a_full[m][0]), 0u), rdy_a1 = t16_mbar_try(smem_u32(&sm.a_full[m][1]), 0u);
    for (int g0 = gb; g0 < ge; g0 += T16_NCHUNK) {                // one step: stages, ring slots and parities are compile-time
#pragma unroll
      for (int kp = 0; kp < NPAIR; ++kp) {
        const int st = (2 * kp) % T16_STAGES, rp = kp % RPAIR;
        const int g = g0 + 2 * kp;
        T16_EV(2 + m, 1);
        if (!rdy_b) t16_mbar_wait_slow(smem_u32(&sm.b_full[rp]), pb0 ^ (uint32_t)((kp / RPAIR) & 1));
        T16_EV(2 + m, 2);                        // W2 chunk pair present
        if (!rdy_a0) t16_mbar_wait_slow(smem_u32(&sm.a_full[m][st]), (uint32_t)((kp / SPAIR) & 1));
        if (!rdy_a1) t16_mbar_wait_slow(smem_u32(&sm.a_full[m][st + 1]), (uint32_t)((kp / SPAIR) & 1));
        T16_EV(2 + m, 3);                        // A chunk pair present
        {
          const int kn = (kp + 1) % NPAIR, sn = (2 * kn) % T16_STAGES;   // next pair (of the next step when kp = 7: same parities)
          rdy_b = t16_mbar_try(smem_u32(&sm.b_full[kn % RPAIR]), pb0 ^ (uint32_t)((kn / RPAIR) & 1));
          rdy_a0 = t16_mbar_try(smem_u32(&sm.a_full[m][sn]), (uint32_t)((kn / SPAIR) & 1));
          rdy_a1 = t16_mbar_try(smem_u32(&sm.a_full[m][sn + 1]), (uint32_t)((kn / SPAIR) & 1));
        }
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (t16_elect_one()) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const uint32_t a0 = a_base + (uint32_t)(st + h) * (2 * T16_A_IMG), b0 = b_base + (uint32_t)(2 * rp + h) * (2 * T16_B_IMG);
            const uint64_t ah = t16_desc(a0, lboA), al = t16_desc(a0 + T16_A_IMG, lboA);
            const uint64_t bh = t16_desc(b0, lboB), bl = t16_desc(b0 + T16_B_IMG, lboB);
            t16_umma(d, ah, bh, idesc, (kp == 0 && h == 0) ? 0u : 1u);
#ifndef T16_EXP_ONE_UMMA      // timing experiment only: hi x hi alone (results lose the low parts)
            t16_umma(d, ah, bl, idesc, 1u);
            t16_umma(d, al, bh, idesc, 1u);
#endif
          }
          t16_commit(&sm.a_empty[m][st >> 1]);                       // the A stage pair may be overwritten once these MMAs are done
          if (kp == NPAIR - 1) t16_commit(&sm.d_full[m]);
          t16_commit(&sm.b_empty[rp]);                               // my share of the ring slot pair
          if (g < ob || g >= oe) t16_commit(&sm.b_empty[rp]);        // ... and the other slot's when it does not consume these chunks
          if (kp == T16_HALF / 2 - 1 && m == 0 && g0 == 0) t16_commit(&sm.start1);   // slot 1 starts half a step behind
        }
        __syncwarp();
        T16_EV(2 + m, 8);
      }
    }
  } else {
    // =================================================================== TMA producer (warp-converged, one elected lane issues)
    constexpr uint32_t bytes = 4 * T16_B_IMG;                      // hi + lo images of two consecutive chunks: 32 KB, contiguous in the image and in the ring
    const int gt = __shfl_sync(0xffffffffu, g_total, 0) / 2;       // chunk pairs (the ranges are multiples of T16_HALF)
    int rp = 0, rphase = 0, kp = 0;
    for (int g = 0; g < gt; ++g) {
      if (g >= T16_RING / 2) t16_mbar_wait(&sm.b_empty[rp], (uint32_t)(rphase ^ 1));
      if (t16_elect_one()) {
        const uint32_t mb = smem_u32(&sm.b_full[rp]);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(&sm.B[2 * rp][0])),
                     "l"(w2img + (size_t)kp * bytes), "r"(bytes), "r"(mb)
                     : "memory");
      }
      __syncwarp();
      if (++rp == T16_RING / 2) { rp = 0; rphase ^= 1; }
      if (++kp == T16_NCHUNK / 2) kp = 0;
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == WORKERS / 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

template <int SYS>
static int launch_rollout_tc16(const cacto_sys_params& P, const float* actor, const unsigned char* w2img, const double* ics, const int32_t* horizon,
                               int T_max, double* states, double* controls, int32_t* flags, double* rewards, int64_t B, cudaStream_t st) {
  auto k = k_rollout_tc16<SYS>;
  const size_t sm = sizeof(Tc16Smem<SysDims<SYS>::NX + 1>);
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
  if (e != cudaSuccess) return (int)e;
  int dev = 0, num_sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
  const int64_t ntiles = (B + T16_TILE - 1) / T16_TILE;
  if (ntiles > (int64_t)1 << 30) return CACTO_E_SIZE;
  // one persistent CTA per SM (two tiles in flight each); more CTAs only when a CTA's tile table would overflow
  int64_t grid = (ntiles + T16_SLOTS - 1) / T16_SLOTS;
  if (grid > num_sms) grid = num_sms;
  if ((ntiles + grid - 1) / grid > T16_MAXT) grid = (ntiles + T16_MAXT - 1) / T16_MAXT;
  k<<<(unsigned)grid, T16_THREADS, sm, st>>>(P, actor, w2img, ics, horizon, T_max, states, controls, flags, rewards, B, (int)ntiles);
  CACTO_LAUNCH_CHECK();
  return 0;
}

}  // namespace cacto

using namespace cacto;

#ifdef T16_TRACE
extern "C" int cacto_debug_t16_trace(long long* buf) { return (int)cudaMemcpyToSymbol(cacto::g_t16_trace, &buf, sizeof(buf)); }
extern "C" int cacto_debug_t16_trace_n(void) { return cacto::T16_TRACE_N; }
#endif

extern "C" int64_t cacto_actor_tc16_image_bytes(void) { return T16_IMG_BYTES + T16_TRAILER; }

extern "C" int cacto_actor_tc16_prepare(const float* actor_params, int32_t ns, int32_t na, void* w2img, void* stream) {
  if (!actor_params || !w2img) return CACTO_E_ARG;
  if (ns < 2 || ns > CACTO_MAX_NS || na < 1 || na > CACTO_MAX_NA) return CACTO_E_SIZE;
  if (reinterpret_cast<uintptr_t>(w2img) & 127) return CACTO_E_ALIGN;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned char* img = static_cast<unsigned char*>(w2img);
  cudaError_t e = cudaMemsetAsync(img + T16_IMG_BYTES, 0, T16_TRAILER, st);
  if (e != cudaSuccess) return (int)e;
  k_tc16_absmax<<<(ACTOR_H * ACTOR_H + 255) / 256, 256, 0, st>>>(actor_params, ns, na, img);
  CACTO_LAUNCH_CHECK();
  k_tc16_prepare<<<(ACTOR_H * ACTOR_H + 255) / 256, 256, 0, st>>>(actor_params, ns, na, img);
  CACTO_LAUNCH_CHECK();
  return 0;
}

extern "C" int cacto_rollout_tc16(const cacto_sys_params* p, const float* actor_params, const void* w2img, const double* ics,
                                  const int32_t* horizon, int32_t T_max, double* states, double* controls, int32_t* flags,
                                  double* rewards, int64_t B, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (p->system < CACTO_SINGLE_INTEGRATOR || p->system > CACTO_MANIPULATOR) return CACTO_E_SYSTEM;   // UR5: cacto_rollout_tc
  if (B < 0 || T_max < 0) return CACTO_E_SIZE;
  if (B == 0) return 0;
  if (!actor_params || !w2img || !ics || !horizon || !states || !flags || (T_max > 0 && !controls)) return CACTO_E_ARG;
  if ((reinterpret_cast<uintptr_t>(w2img) & 127) || (reinterpret_cast<uintptr_t>(actor_params) & 15)) return CACTO_E_ALIGN;
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned char* img = static_cast<const unsigned char*>(w2img);
  switch (p->system) {
    case CACTO_SINGLE_INTEGRATOR: return launch_rollout_tc16<CACTO_SINGLE_INTEGRATOR>(*p, actor_params, img, ics, horizon, T_max, states, controls, flags, rewards, B, st);
    case CACTO_DOUBLE_INTEGRATOR: return launch_rollout_tc16<CACTO_DOUBLE_INTEGRATOR>(*p, actor_params, img, ics, horizon, T_max, states, controls, flags, rewards, B, st);
    case CACTO_CAR: return launch_rollout_tc16<CACTO_CAR>(*p, actor_params, img, ics, horizon, T_max, states, controls, flags, rewards, B, st);
    case CACTO_CAR_PARK: return launch_rollout_tc16<CACTO_CAR_PARK>(*p, actor_params, img, ics, horizon, T_max, states, controls, flags, rewards, B, st);
    case CACTO_MANIPULATOR: return launch_rollout_tc16<CACTO_MANIPULATOR>(*p, actor_params, img, ics, horizon, T_max, states, controls, flags, rewards, B, st);
    default: return CACTO_E_SYSTEM;
  }
}
