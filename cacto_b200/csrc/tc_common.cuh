// tc_common.cuh -- building blocks of the tensor-core (tcgen05) update kernels of update_tc.cu.
//
// Arithmetic: every dense layer of the large-batch Sobolev update (NeuralNetwork.py:150-232) is a 128-row tile GEMM on
// tcgen05.mma kind::f16 with fp16 operand splitting -- the scheme of rollout_tc16.cu:
//     a' = 2^p a = a_hi + a_lo,  w' = 2^s w = w_hi + w_lo,   a' w' ~= a_hi w_hi + a_hi w_lo + a_lo w_hi   (fp32 accumulation in TMEM)
// with power-of-two scales (exact): per weight matrix from max|W| (prepare kernel), per ROW of the activation tile from a bound
// on the row's magnitude (the thread that owns the row knows it), so that no operand leaves the fp16 range however the
// network was trained.  Relative error of a product ~2^-21; a CPU emulation of the split with these scales stays within the fp32
// error per layer on trained networks (tests/test_trained_nets.py).  The engine as a whole does not: on the reference's trained
// double-integrator actor its actions are ~35x and its dW3 ~22x the fp32 oracle's distance from fp64 (dW3 1.07e-4, just past the
// 1e-4 parity gate; tests/test_gpu_trained_nets.py K_TC).  The source of that excess is not located yet.
//
// Kernel skeleton ("chain kernel"): a persistent CTA walks a list of jobs (one 128-row tile each); per job a chain of layers
//     [epilogue threads write the A image of layer l] -> a_full -> [issuer: UMMAs over the K-chunks of W_l] -> d_full ->
//     [epilogue threads read the accumulator from TMEM, apply the layer's functor, write side outputs + the next A image]
// with three roles: 16 epilogue warps (warp w owns TMEM lanes 32 (w & 3).. and the 16-column chunks c with (c & 3) == w >> 2),
// one MMA-issuer warp and one TMA-producer warp that streams the pre-split weight images (16 KB chunks, cp.async.bulk) from L2
// through a ring of shared-memory slots, running ahead of the issuer across layers and jobs.
#pragma once
#include <cuda_fp16.h>
#include "common.cuh"
#include "mlp.cuh"

namespace cacto {
namespace tcu {

constexpr int TILE = 128;                       // rows of a tile = UMMA M
constexpr int EPI_WARPS = 16, EPI_THREADS = EPI_WARPS * 32;
constexpr int THREADS = EPI_THREADS + 64;       // + issuer warp + producer warp
constexpr int CHUNK_ELEMS = 4096;               // N * kc of one weight chunk
constexpr int CHUNK_BYTES = 4 * CHUNK_ELEMS;    // hi + lo fp16 images: 16 KB
constexpr int LBO_A = (TILE / 8) * 128;         // k-unit stride of a 128-row K-major image: 2048 B
constexpr int MAX_LAYERS = 6;
constexpr int A_GROUP_K = 64, A_GROUPS = 4;     // the A image of a layer is published in groups of 64 k-values (<= 256 / 64 groups)
constexpr int ACC_COLS = 256;                   // TMEM columns of one accumulator; consecutive layers alternate between two
constexpr float SIN_SCALE = 8192.f;             // |sin|, |cos| <= 1 -> |a'| <= 2^13

struct LayerSeq {        // the layers of one chain, in issue order; K, N multiples of 16, N <= 256
  int n;
  int K[MAX_LAYERS], N[MAX_LAYERS];
};
__host__ __device__ __forceinline__ int layer_kc(int K, int N) { const int kc = CHUNK_ELEMS / N; return kc > K ? K : kc; }   // k-values per chunk
__host__ __device__ __forceinline__ int64_t stream_bytes(const LayerSeq& L) {
  int64_t b = 0;
  for (int l = 0; l < L.n; ++l) b += (int64_t)L.K[l] * L.N[l] * 4;
  return b;
}
// byte offset of B[n][kk] inside the hi image of one chunk of a layer with N outputs (K-major, no swizzle: 16-byte units of 8
// consecutive k; 8 rows x 16 B = one core matrix; 8-row groups 128 B apart; k-units (N / 8) * 128 B apart)
__host__ __device__ __forceinline__ int b_offset(int N, int n, int kk) { return (kk >> 3) * (N / 8) * 128 + (n >> 3) * 128 + (n & 7) * 16 + (kk & 7) * 2; }

#ifdef TCU_TRACE   // debug builds only (profiles/scripts/tcu_trace.py): event timeline of CTA 0 -- role 0: epilogue thread 0, role 1: issuer
__device__ long long* g_tcu_trace = nullptr;
constexpr int TCU_TRACE_N = 4096;
#define TCU_EV(role, code)                                                                                        \
  do {                                                                                                            \
    if (blockIdx.x == 0 && g_tcu_trace != nullptr && (threadIdx.x & 31) == 0 && tcu_trace_n < TCU_TRACE_N)        \
      g_tcu_trace[(role) * TCU_TRACE_N + tcu_trace_n++] = (clock64() << 8) | (long long)(code);                   \
  } while (0)
#define TCU_TRACE_DECL int tcu_trace_n = 0
#else
#define TCU_EV(role, code) do { } while (0)
#define TCU_TRACE_DECL do { } while (0)
#endif

// ---------------------------------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count)); }
__device__ __forceinline__ void mbar_arrive(uint64_t* b) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory"); }
__device__ __forceinline__ bool mbar_try(uint32_t mb, uint32_t parity) {
  uint32_t done;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(mb), "r"(parity) : "memory");
  return done != 0;
}
__device__ __noinline__ void mbar_wait_slow(uint32_t mb, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  unsigned long long t0 = 0;
  while (true) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(mb), "r"(parity), "r"(20000u) : "memory");
    if (done) break;
    if ((++spins & 1023u) == 0) {                    // fail loudly instead of hanging the GPU: trap after 4 s
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000ull) __trap();
    }
  }
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
  const uint32_t mb = smem_u32(b);
  if (!mbar_try(mb, parity)) mbar_wait_slow(mb, parity);
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void umma_commit(uint64_t* b) { asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(b)) : "memory"); }
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t)(128u >> 4) << 32) | ((uint64_t)1 << 46);
}
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(da), "l"(db),
               "r"(idesc), "r"(accumulate)
               : "memory");
}
__device__ __forceinline__ uint32_t umma_idesc(int N) { return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(TILE >> 4) << 24); }   // f16 x f16 -> f32, K-major
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, %0;" ::"n"(EPI_THREADS) : "memory"); }     // the 512 epilogue threads only
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {      // (lo, hi) -> f16x2, lo in the low half
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// 16 consecutive accumulator columns of the thread's TMEM lane
__device__ __forceinline__ void ldtm16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]),
        "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// 2^e with m 2^e in [2^13, 2^14) for a finite m > 0 (1 for m = 0 / non-finite): the scale that puts a row (or a matrix) of
// largest magnitude m at the top of the fp16 range with 2 bits of headroom; `inv` receives 2^-e.
__host__ __device__ __forceinline__ float pow2_scale(float m, float& inv) {
#ifdef __CUDA_ARCH__
  const uint32_t bits = __float_as_uint(m);
#else
  uint32_t bits;
  memcpy(&bits, &m, 4);
#endif
  const int e = (int)((bits >> 23) & 0xff);
  if (e == 0 || e == 255) { inv = 1.f; return 1.f; }
  int s = 13 - (e - 127);
  s = s > 100 ? 100 : (s < -100 ? -100 : s);
  const uint32_t sb = (uint32_t)(s + 127) << 23, ib = (uint32_t)(127 - s) << 23;
#ifdef __CUDA_ARCH__
  inv = __uint_as_float(ib);
  return __uint_as_float(sb);
#else
  float r;
  memcpy(&r, &sb, 4);
  memcpy(&inv, &ib, 4);
  return r;
#endif
}

// x rounded to 11 significant bits (nearest, ties away from zero; exactly representable in fp16 when in range): with truncation
// instead the dropped a_lo w_lo term of the split product is 4 x larger (2^-20 instead of 2^-22 relative)
__device__ __forceinline__ float hi11(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }

// hi / lo fp16 split of a scaled pair: hi = RN_fp16(a) (11 significant bits), lo = RN_fp16(a - hi) -- the subtraction is exact in
// fp32.  Packed fp32x2 multiply / subtract and the f16x2 conversions: 6 instructions per pair (the integer rounding trick of hi11
// plus scalar arithmetic took 10; the chunk passes of the chain kernels are issue-bound).
__device__ __forceinline__ void split_pair(float x0, float x1, float scale, uint32_t& h, uint32_t& l) {
  uint64_t a, d;
  asm("{\n\t.reg .b64 x, s;\n\tmov.b64 x, {%1, %2};\n\tmov.b64 s, {%3, %3};\n\tmul.rn.f32x2 %0, x, s;\n\t}" : "=l"(a) : "f"(x0), "f"(x1), "f"(scale));
  float a0, a1, h0, h1;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(a));
  h = pack_h2(a0, a1);
  asm("{\n\t.reg .b16 lo, hi;\n\tmov.b32 {lo, hi}, %2;\n\tcvt.f32.f16 %0, lo;\n\tcvt.f32.f16 %1, hi;\n\t}" : "=f"(h0), "=f"(h1) : "r"(h));
  asm("{\n\t.reg .b64 hh, m1;\n\tmov.b64 hh, {%2, %3};\n\tmov.b64 m1, {%4, %4};\n\tfma.rn.f32x2 %0, hh, m1, %1;\n\t}" : "=l"(d) : "l"(a), "f"(h0), "f"(h1), "f"(-1.f));
  float d0, d1;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d0), "=f"(d1) : "l"(d));
  l = pack_h2(d0, d1);
}
// ... of 8 scaled values -> one 16-byte unit of each image
__device__ __forceinline__ void split8(const float* x, float scale, uint4& hi, uint4& lo) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int p = 0; p < 4; ++p) split_pair(x[2 * p], x[2 * p + 1], scale, h[p], l[p]);
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// ---------------------------------------------------------------------------------------------------- workspace layout
// Per-sample tensors of width W (a multiple of 4) live as [tile][W / 4][128 rows][4]: the thread that owns row r of a tile moves
// float4 number (tile * W/4 + c4) * 128 + r -- a warp touches 512 contiguous bytes -- and the weight-gradient kernel finds the
// 8 consecutive samples of a feature group (one fp16 k-unit) in 128 contiguous bytes.
__device__ __forceinline__ float4* ws4(float* base, int W, int64_t tile, int col, int row) {
  return reinterpret_cast<float4*>(base) + ((tile * (W >> 2) + (col >> 2)) * TILE + row);
}
__device__ __forceinline__ const float4* ws4(const float* base, int W, int64_t tile, int col, int row) {
  return reinterpret_cast<const float4*>(base) + ((tile * (W >> 2) + (col >> 2)) * TILE + row);
}
__device__ __forceinline__ void ws_store16(float* base, int W, int64_t tile, int col, int row, const float* v) {
#pragma unroll
  for (int i = 0; i < 4; ++i) *ws4(base, W, tile, col + 4 * i, row) = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}
__device__ __forceinline__ void ws_load16(const float* base, int W, int64_t tile, int col, int row, float* v) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float4 f = *ws4(base, W, tile, col + 4 * i, row);
    v[4 * i] = f.x; v[4 * i + 1] = f.y; v[4 * i + 2] = f.z; v[4 * i + 3] = f.w;
  }
}

// ---------------------------------------------------------------------------------------------------- shared state of a chain kernel
template <int A_K, int RING>
struct ChainSmem {
  static constexpr int A_IMG = TILE * A_K * 2;                       // bytes of the hi (or lo) A image for K <= A_K
  alignas(1024) unsigned char ring[RING][CHUNK_BYTES];
  alignas(1024) unsigned char a_hi[A_IMG];
  alignas(1024) unsigned char a_lo[A_IMG];
  alignas(16) float rowx[2][4][TILE];                                // per-row exchange between the 4 column groups (double-buffered)
  alignas(16) float colsum[640];                                     // per-CTA column sums (bias / head gradients), flushed at the end
  uint64_t w_full[RING], w_empty[RING], a_full[A_GROUPS], d_full;
  uint32_t tmem_base;
};

// what an epilogue thread knows about itself
struct Epi {
  int warp, lane, q, cgp, row;        // TMEM lane quadrant, column group, row within the tile
  uint32_t taddr;                     // TMEM address of (row, column 0) of the accumulator being consumed (set by wait_acc)
  uint32_t tbase;                     // ... of accumulator buffer 0
  uint32_t layers_done;               // accumulators consumed so far (phase of d_full, accumulator buffer = parity)
  uint32_t xbuf;                      // parity of the row-exchange buffer
};

template <typename SM>
__device__ __forceinline__ void chain_setup(SM& sm, int tid, int warp) {
  if (tid == 0) {
    for (int s = 0; s < (int)(sizeof(sm.w_full) / 8); ++s) { mbar_init(&sm.w_full[s], 1); mbar_init(&sm.w_empty[s], 1); }
    for (int g = 0; g < A_GROUPS; ++g) mbar_init(&sm.a_full[g], EPI_THREADS);
    mbar_init(&sm.d_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < 640; i += THREADS) sm.colsum[i] = 0.f;
  if (warp == EPI_WARPS) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sm.tmem_base)), "r"(2 * ACC_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
}
template <typename SM>
__device__ __forceinline__ void chain_teardown(SM& sm, int warp) {
  tc_fence_before();
  __syncthreads();
  if (warp == EPI_WARPS) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(sm.tmem_base), "r"(2 * ACC_COLS));
}
__device__ __forceinline__ Epi epi_init(int tid, uint32_t tmem) {
  Epi e;
  e.warp = tid >> 5; e.lane = tid & 31; e.q = e.warp & 3; e.cgp = e.warp >> 2; e.row = 32 * e.q + e.lane;
  e.tbase = tmem + ((uint32_t)(32 * e.q) << 16);
  e.taddr = e.tbase;
  e.layers_done = 0; e.xbuf = 0;
  return e;
}
// The A image of the next layer reaches the issuer in groups of A_GROUP_K k-values: the issuer starts the UMMAs of a K-chunk as
// soon as its groups are complete, while the epilogue threads are still producing the later ones (the accumulators of consecutive
// layers alternate between two TMEM buffers, so the running UMMAs never touch the one being read).  Every epilogue thread
// arrives exactly once per layer on EACH of the A_GROUPS barriers -- publish_a_group(g) as soon as its share of group g is
// written, publish_a_from(g) for all remaining groups -- so that all of them flip once per layer whatever the layer's width.
template <typename SM>
__device__ __forceinline__ void publish_a_group(SM& sm, int g) {
  fence_async_smem();
  tc_fence_before();
  mbar_arrive(&sm.a_full[g]);
}
template <typename SM>
__device__ __forceinline__ void publish_a_from(SM& sm, int g0) {
  fence_async_smem();
  tc_fence_before();
  for (int g = g0; g < A_GROUPS; ++g) mbar_arrive(&sm.a_full[g]);
}
// the whole A image of the next layer is complete (and my TMEM reads of the previous accumulator are done)
template <typename SM>
__device__ __forceinline__ void publish_a(SM& sm) { publish_a_from(sm, 0); }
template <typename SM>
__device__ __forceinline__ void wait_acc(SM& sm, Epi& e) {
  mbar_wait(&sm.d_full, e.layers_done & 1u);
  e.taddr = e.tbase + (e.layers_done & 1u) * (uint32_t)ACC_COLS;
  ++e.layers_done;
  tc_fence_after();
}
// combine a per-thread value over the 4 column-group threads that share a row
template <typename SM>
__device__ __forceinline__ float row_max4(SM& sm, Epi& e, float m) {
  float (*x)[TILE] = sm.rowx[e.xbuf];
  e.xbuf ^= 1u;
  x[e.cgp][e.row] = m;
  epi_bar();
  return fmaxf(fmaxf(x[0][e.row], x[1][e.row]), fmaxf(x[2][e.row], x[3][e.row]));
}
template <typename SM>
__device__ __forceinline__ float row_sum4(SM& sm, Epi& e, float m) {
  float (*x)[TILE] = sm.rowx[e.xbuf];
  e.xbuf ^= 1u;
  x[e.cgp][e.row] = m;
  epi_bar();
  return (x[0][e.row] + x[1][e.row]) + (x[2][e.row] + x[3][e.row]);
}
// 16 values of my row (columns k0 .. k0 + 15 of the next layer's input) -> the A image
template <typename SM>
__device__ __forceinline__ void put_a16(SM& sm, const Epi& e, int k0, const float* v, float scale) {
  const int off = (k0 >> 3) * LBO_A + (e.row >> 3) * 128 + (e.row & 7) * 16;
  uint4 hi, lo;
  split8(v, scale, hi, lo);
  *reinterpret_cast<uint4*>(sm.a_hi + off) = hi;
  *reinterpret_cast<uint4*>(sm.a_lo + off) = lo;
  split8(v + 8, scale, hi, lo);
  *reinterpret_cast<uint4*>(sm.a_hi + off + LBO_A) = hi;
  *reinterpret_cast<uint4*>(sm.a_lo + off + LBO_A) = lo;
}
// max |accumulator| over the thread's 16-column chunks of an N-column layer (pass 1 of a row-scaled epilogue)
template <int N>
__device__ __forceinline__ float acc_absmax(const Epi& e) {
  float m = 0.f;
#pragma unroll 1
  for (int ch = e.cgp; ch < N / 16; ch += 4) {
    float v[16];
    ldtm16(e.taddr + (uint32_t)(16 * ch), v);
#pragma unroll
    for (int i = 0; i < 16; ++i) m = fmaxf(m, fabsf(v[i]));
  }
  return m;
}
// column sums over the 32 rows of a warp for 16 columns (butterfly: 16 shuffles), added into colsum[c0 .. c0 + 15].  DET: colsum
// belongs to this warp alone (a per-quadrant copy, update_tc.cu), so each lane adds its column with a plain read-modify-write.
template <bool DET = false>
__device__ __forceinline__ void warp_colsum16(float* colsum, int c0, const float* v, int lane) {
  float a[8];
  {
    const bool up = lane & 16;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float send = up ? v[i] : v[i + 8], keep = up ? v[i + 8] : v[i];
      a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
  }
  float b[4];
  {
    const bool up = lane & 8;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float send = up ? a[i] : a[i + 4], keep = up ? a[i + 4] : a[i];
      b[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
  }
  float c[2];
  {
    const bool up = lane & 4;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const float send = up ? b[i] : b[i + 2], keep = up ? b[i + 2] : b[i];
      c[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
  }
  const bool up = lane & 2;
  float d = (up ? c[1] : c[0]) + __shfl_xor_sync(0xffffffffu, up ? c[0] : c[1], 2);
  d += __shfl_xor_sync(0xffffffffu, d, 1);
  // lane holds column 8 [lane & 16] + 4 [lane & 8] + 2 [lane & 4] + [lane & 2]
  if ((lane & 1) == 0) {
    float* p = &colsum[c0 + ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1)];
    if constexpr (DET) *p += d;
    else atomicAdd(p, d);
  }
}
__device__ __forceinline__ void amax_update(uint32_t* slot, float m, int lane) {      // slot = max over the tensor of |x| (bit pattern)
  uint32_t b = __float_as_uint(m) & 0x7fffffffu;
  b = __reduce_max_sync(0xffffffffu, b);
  if (lane == 0 && b != 0u) atomicMax(slot, b);
}

// ---------------------------------------------------------------------------------------------------- issuer / producer roles
// One layer sequence of one job: waits for the A image, walks the K-chunks of every layer in ring order.
struct RingState {
  int slot;
  uint32_t phase;
  uint32_t layers;      // layers issued so far (phase of a_full)
};
template <int RING, typename SM>
__device__ __forceinline__ void issue_job(SM& sm, const LayerSeq& L, RingState& rs, uint32_t tmem, int& tcu_trace_n) {
  const uint32_t a_hi = smem_u32(sm.a_hi), a_lo = smem_u32(sm.a_lo), ring = smem_u32(&sm.ring[0][0]);
  for (int l = 0; l < L.n; ++l) {
    const int K = L.K[l], N = L.N[l], kc = layer_kc(K, N), nch = K / kc;
    const uint32_t idesc = umma_idesc(N), lboB = (uint32_t)(N / 8) * 128u, b_lo = (uint32_t)(N * kc * 2);
    const uint32_t par = rs.layers & 1u, d = tmem + par * (uint32_t)ACC_COLS;      // a_full phase and accumulator buffer of this layer
    ++rs.layers;
    int groups = 0;                        // A groups waited for so far
    for (int c = 0; c < nch; ++c) {
      const int need = ((c + 1) * kc - 1) / A_GROUP_K + 1;      // groups that hold the k-values of this chunk
      for (; groups < need; ++groups) mbar_wait(&sm.a_full[groups], par);
      if (c == 0) TCU_EV(1, 1);            // first A group present
      mbar_wait(&sm.w_full[rs.slot], rs.phase);
      if (c == 0) TCU_EV(1, 2);            // first weight chunk present
      tc_fence_after();
      if (elect_one()) {
        const uint32_t b0 = ring + (uint32_t)rs.slot * CHUNK_BYTES;
        for (int ks = 0; ks < kc / 16; ++ks) {
          const uint32_t ao = (uint32_t)((c * kc + 16 * ks) >> 3) * LBO_A, bo = b0 + (uint32_t)ks * 2u * lboB;
          const uint64_t ah = umma_desc(a_hi + ao, LBO_A), al = umma_desc(a_lo + ao, LBO_A);
          const uint64_t bh = umma_desc(bo, lboB), bl = umma_desc(bo + b_lo, lboB);
          umma_f16(d, ah, bh, idesc, (c == 0 && ks == 0) ? 0u : 1u);
          umma_f16(d, ah, bl, idesc, 1u);
          umma_f16(d, al, bh, idesc, 1u);
        }
        umma_commit(&sm.w_empty[rs.slot]);
        if (c == nch - 1) umma_commit(&sm.d_full);
      }
      __syncwarp();
      if (c == nch - 1) TCU_EV(1, 3);      // layer issued
      if (++rs.slot == RING) { rs.slot = 0; rs.phase ^= 1u; }
    }
  }
}
template <int RING, typename SM>
__device__ __forceinline__ void produce_job(SM& sm, const LayerSeq& L, const unsigned char* __restrict__ stream, RingState& rs) {
  const unsigned char* src = stream;
  for (int l = 0; l < L.n; ++l) {
    const int K = L.K[l], N = L.N[l], kc = layer_kc(K, N), nch = K / kc;
    const uint32_t bytes = (uint32_t)(N * kc * 4);
    for (int c = 0; c < nch; ++c) {
      mbar_wait(&sm.w_empty[rs.slot], rs.phase ^ 1u);          // fresh barrier: the wait on the preceding phase returns at once
      if (elect_one()) {
        const uint32_t mb = smem_u32(&sm.w_full[rs.slot]);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(&sm.ring[rs.slot][0])),
                     "l"(src), "r"(bytes), "r"(mb)
                     : "memory");
      }
      __syncwarp();
      src += bytes;
      if (++rs.slot == RING) { rs.slot = 0; rs.phase ^= 1u; }
    }
  }
}

}  // namespace tcu
}  // namespace cacto
