// update_tc.cu -- K3 at large batch (B >= ~2 k: BASELINE configs 2, 3, 5) on tcgen05 tensor cores.
//
// Same arithmetic as update.cu -- NN.compute_critic_grad (NeuralNetwork.py:150-178) as the sweeps F / G / A / B of SURVEY.md
// A.3 and NN.compute_actor_grad (:180-232, A.4) -- organised layer by layer over 128-sample tiles instead of sample-tile by
// sample-tile: every dense layer is a tile GEMM on tcgen05.mma kind::f16 with fp16 operand splitting (tc_common.cuh), the
// per-sample intermediates (sin z, cos z, g, delta, a, extra, e: ~10 KB per sample) go through a caller-owned workspace in a
// tile-major layout that both the sweeps (thread per row) and the weight-gradient GEMMs (reduction over samples) read as
// contiguous 16-byte vectors, and the weight gradients are batch-reduction GEMMs (one accumulator per 128 x N block of dW in
// TMEM, ~150 CTAs, 16-byte vector reductions into the gradient block) instead of one atomic per weight and 16 samples.
//
//   k_tc_prepare      weight images: per matrix max|W| -> power-of-two scale -> hi / lo fp16 images in UMMA layout, 16 KB chunks
//   k_tc_critic_fwd   forward sweeps: target critic at s_next / s, critic at s (keeps sin, cos), critic at s' (actor step)
//   k_tc_critic_bwd   G sweep (dV/ds through the net + Sobolev loss seeds), GP (dV/ds' -> dQ/da for the actor), B sweep
//   k_tc_critic_adj   A sweep (adjoint through G: second-order terms)
//   k_tc_actor_fwd    actor forward (keeps h1, h2);   k_tc_actor_env  s' = f(s, a), ds'/da, dr/da per sample (fp64)
//   k_tc_actor_bwd    actor backward;                 k_tc_wgrad      all weight gradients of a step in one launch
#include <string.h>
#include "common.cuh"
#include "det.cuh"
#include "mlp.cuh"
#include "systems.cuh"
#include "tc_common.cuh"

namespace cacto {
using namespace tcu;

constexpr int CWT = CR_H1 + CR_H2 + CR_H3 + CR_H4;    // 384 hidden units of the critic
__host__ __device__ __forceinline__ constexpr int kofs(int l) { return l == 0 ? 0 : (l == 1 ? CR_H1 : (l == 2 ? CR_H1 + CR_H2 : CR_H1 + CR_H2 + CR_H3)); }

// sin / cos of the SIREN layers -- what the forward sweeps spend their time on (96 evaluations per thread and job).
// sinf / sincosf inline a Payne-Hanek slow path (local-memory loops) at every call site: with 96 call sites per sweep the
// kernel outgrew the instruction cache (ncu, first version: 45 us per 128-row forward sweep).  Fast path: k = rint(x / pi) by the
// magic-number trick (no float <-> int conversions, which run at a quarter of the FMA rate), Cody-Waite reduction r = x - k pi
// in three FMAs (exact products for |k| < 2^15), minimax polynomials r P(r^2) (degree 9) and Q(r^2) (degree 10) on [-pi/2, pi/2]
// (max abs error 1.7e-7, measured against fp64 over |x| < 60: profiles/scripts/sincos_fit.py), sign (-1)^k by an XOR.  Arguments
// beyond 1e5 -- never produced by a SIREN with finite weights of sane size -- take the accurate library routine out of line.
__device__ __noinline__ float2 sincos_slow(float x) {
  float2 r;
  sincosf(x, &r.x, &r.y);
  return r;
}
__device__ __forceinline__ float reduce_pi(float x, uint32_t& sign) {
  const float t = fmaf(x, 0.318309886f, 12582912.f);          // 1.5 * 2^23: the integer part lands in the low mantissa bits
  const float k = t - 12582912.f;
  sign = __float_as_uint(t) << 31;                            // parity of k
  float r = fmaf(k, -3.140625f, x);
  r = fmaf(k, -9.67502593994140625e-4f, r);
  return fmaf(k, -1.509957990978376432e-7f, r);
}
__device__ __forceinline__ float sin_poly(float r, float r2) {
  float p = fmaf(r2, 2.605224915696493e-06f, -0.00019809075291124477f);
  p = fmaf(r2, p, 0.008333051063441448f);
  p = fmaf(r2, p, -0.16666657991913642f);
  p = fmaf(r2, p, 0.9999999957328009f);
  return r * p;
}
__device__ __forceinline__ float cos_poly(float r2) {
  float p = fmaf(r2, -2.605149521781454e-07f, 2.4760161353683747e-05f);
  p = fmaf(r2, p, -0.001388836140030791f);
  p = fmaf(r2, p, 0.041666636258075075f);
  p = fmaf(r2, p, -0.4999999935847215f);
  return fmaf(r2, p, 0.9999999997806525f);
}
__device__ __forceinline__ void sincos_fast(float x, float& s, float& c) {
  uint32_t sg;
  const float r = reduce_pi(x, sg), r2 = r * r;
  s = __uint_as_float(__float_as_uint(sin_poly(r, r2)) ^ sg);
  c = __uint_as_float(__float_as_uint(cos_poly(r2)) ^ sg);
}
__device__ __forceinline__ float sin_fast(float x) {
  uint32_t sg;
  const float r = reduce_pi(x, sg);
  return __uint_as_float(__float_as_uint(sin_poly(r, r * r)) ^ sg);
}

__device__ __forceinline__ float slog_tc(float x) { return x > 0.f ? logf(fmaxf(x, 1e-7f) + 1.f) : -logf(fmaxf(-x, 1e-7f) + 1.f); }
__device__ __forceinline__ float slog_grad_tc(float x) { return fabsf(x) >= 1e-7f ? 1.f / (fabsf(x) + 1.f) : 0.f; }

// indices into the per-update absmax table (bit patterns; zeroed by k_tc_prepare)
enum { AM_XN = 0, AM_A0, AM_AA, AM_DL, AM_EE, AM_XNA, AM_H1, AM_H2, AM_E2, AM_E1, AM_D3, AM_VB, AM_COUNT = 16 };

// Device pointers into the caller's workspace (cacto_update_tc_workspace_bytes).  "ws4" tensors use the tile-major layout of
// tc_common.cuh; "rows" tensors are per-row scalars [tiles * 128]; "rm" tensors are row-major [B][width].
struct TcWs {
  float *XN, *CS, *SN, *GG, *DL, *A0, *AA, *EX, *EE;            // critic step (ws4; widths 16, 384, 384, 256, 384, 16, 256, 384, 384)
  float *VTN, *VBAR, *EXMAX;                                    // rows; EXMAX: [4][tiles * 128]
  float *VB4;                                                   // ws4, width 4: vbar in column 0
  float *XNA, *H1, *H2, *CSP, *D3, *E2, *E1;                    // actor step (ws4; widths 16, 256, 256, 384, 16, 256, 256)
  float *ACT, *SP, *FU, *DRDA;                                  // rm: [B][na], [B][ns], [B][ns * na], [B][na]
  float *PART;                                                  // [WG_MAX_CTAS][128][256] partial weight-gradient blocks
  unsigned char *S_tf, *S_cf, *S_cb, *S_af, *S_ab;              // weight streams: target fwd, critic fwd / bwd, actor fwd / bwd
  float *US;                                                    // [5][8] unscale 2^-s per stream and layer
  uint32_t* amax;                                               // [AM_COUNT]
  int64_t tiles;
};
enum { ST_TF = 0, ST_CF, ST_CB, ST_AF, ST_AB };
constexpr int WG_MAX_CTAS = 192;

// ---- deterministic variants (DET = true; cacto_*_grad_tc_det).  The bias / head column sums and the loss are the only cross-warp and
// cross-CTA float sums of the chain kernels (the weight matrices already go through the fixed-order k_tc_wgrad_reduce).  With DET
// every epilogue quadrant q sums into its own copy colq[q] of the column sums (behind the chain's shared state, TC_DET_SMEM bytes;
// one warp per entry), the loss per warp into lossw[warp]; at the end the CTA writes (colq[0] + colq[1]) + (colq[2] + colq[3]) and
// the warp-ordered loss into its slice of a partials region -- every entry of the slice, so the region needs no clearing -- and
// k_tc_det_reduce adds the slices of each region into grad in slice order.  Slice layout (TC_DET_SLICE floats), critic: [0, 384) d b_l
// at kofs(l), [384, 512) d w5, 512 d b5, TC_DET_LOSS the loss; actor: [0, 256) d b2, [256, 512) d b1, [512, 512 + na) d b3.
constexpr int TC_DET_SLICE = (int)det_tc_slice, TC_DET_LOSS = 640, TC_DET_COLS = 640;
constexpr size_t TC_DET_SMEM = (4 * TC_DET_COLS + EPI_WARPS) * sizeof(float);
template <typename SM>
__device__ __forceinline__ float* det_colq(unsigned char* smem_raw) { return reinterpret_cast<float*>(smem_raw + sizeof(SM)); }
template <typename SM>
__device__ __forceinline__ void det_clear(unsigned char* smem_raw, int tid) {        // before chain_setup (whose barrier publishes it)
  float* q = det_colq<SM>(smem_raw);
  for (int i = tid; i < 4 * TC_DET_COLS + EPI_WARPS; i += THREADS) q[i] = 0.f;
}
// epilogue threads, after the epi_bar that ends the jobs: column sums [0, n) go to slice entries [dst, dst + n)
template <typename SM>
__device__ __forceinline__ void det_flush(unsigned char* smem_raw, float* slice, int n, int dst, bool loss, int tid) {
  const float* q = det_colq<SM>(smem_raw);
  for (int i = tid; i < TC_DET_SLICE; i += EPI_THREADS) {
    float v = 0.f;
    const int k = i - dst;
    if (k >= 0 && k < n) v = (q[k] + q[TC_DET_COLS + k]) + (q[2 * TC_DET_COLS + k] + q[3 * TC_DET_COLS + k]);
    if (i == TC_DET_LOSS && loss) {
      for (int w = 0; w < EPI_WARPS; ++w) v += q[4 * TC_DET_COLS + w];
    }
    slice[i] = v;
  }
}

static LayerSeq seq_critic_fwd() { LayerSeq L = {4, {16, CR_H1, CR_H2, CR_H3}, {CR_H1, CR_H2, CR_H3, CR_H4}}; return L; }
static LayerSeq seq_critic_bwd(int n) { LayerSeq L = {n, {CR_H4, CR_H3, CR_H2, CR_H1}, {CR_H3, CR_H2, CR_H1, 16}}; return L; }
static LayerSeq seq_actor_fwd() { LayerSeq L = {3, {16, ACTOR_H, ACTOR_H}, {ACTOR_H, ACTOR_H, 16}}; return L; }
static LayerSeq seq_actor_bwd() { LayerSeq L = {2, {16, ACTOR_H}, {ACTOR_H, ACTOR_H}}; return L; }

// ================================================================================================== weight images
struct PrepJob {
  const float* W;        // row-major [in][out] (Keras kernel)
  int in, out;           // real sizes
  int K, N;              // padded GEMM sizes of the image
  int fwd;               // 1: B[n][k] = W[k][n] (x W);  0: B[n][k] = W[n][k] (delta W^T)
  unsigned char* dst;    // K * N * 4 bytes: chunks of [hi | lo]
  float* unscale;        // receives 2^-s
};
struct PrepTable {
  int n;
  PrepJob j[16];
  int cta0[17];          // CTAs [cta0[j], cta0[j + 1]) convert the 16-byte units of job j (1024 units each)
  uint32_t* zero;        // words cleared by block 0 (absmax table)
  int nzero;
};

__global__ void __launch_bounds__(512) k_tc_prepare(const PrepTable T) {
  __shared__ uint32_t wmax[16];
  pdl_wait();
  int ji = 0;
  while (ji + 1 < T.n && (int)blockIdx.x >= T.cta0[ji + 1]) ++ji;
  const PrepJob& J = T.j[ji];
  const int tid = threadIdx.x, part = blockIdx.x - T.cta0[ji];
  if (blockIdx.x == 0)
    for (int i = tid; i < T.nzero; i += 512) T.zero[i] = 0u;
  // every CTA of a job scans the whole matrix for max|W| (L2-resident, <= 64 K floats)
  uint32_t m = 0;
  {
    const int n4 = (J.in * J.out) >> 2;                      // every layer block starts 16-byte aligned and holds a multiple of 4 floats ...
    const float4* w4 = reinterpret_cast<const float4*>(J.W);
#pragma unroll 8
    for (int i = tid; i < n4; i += 512) {
      const float4 w = __ldg(w4 + i);
      m = max(max(m, __float_as_uint(w.x) & 0x7fffffffu), max(__float_as_uint(w.y) & 0x7fffffffu, max(__float_as_uint(w.z) & 0x7fffffffu, __float_as_uint(w.w) & 0x7fffffffu)));
    }
    for (int i = 4 * n4 + tid; i < J.in * J.out; i += 512) m = max(m, __float_as_uint(__ldg(J.W + i)) & 0x7fffffffu);   // ... except actor W3 with odd na
  }
  m = __reduce_max_sync(0xffffffffu, m);
  if ((tid & 31) == 0) wmax[tid >> 5] = m;
  __syncthreads();
  m = wmax[0];
#pragma unroll
  for (int i = 1; i < 16; ++i) m = max(m, wmax[i]);
  float inv;
  const float s = pow2_scale(__uint_as_float(m), inv);
  if (tid == 0 && part == 0) *J.unscale = inv;
  const int K = J.K, N = J.N, kc = layer_kc(K, N), KU = K / 8;
  const int chunk_bytes = N * kc * 4, lo_off = N * kc * 2;
  // one 16-byte unit (8 consecutive k of one n) per thread and step
  for (int it = part * 1024 + tid; it < min(N * KU, part * 1024 + 1024); it += 512) {
    int n, u;
    float x[8];
    if (J.fwd) {              // source contiguous in n: consecutive threads take consecutive n
      u = it / N; n = it - u * N;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int k = 8 * u + i;
        x[i] = (k < J.in && n < J.out) ? __ldg(J.W + (int64_t)k * J.out + n) : 0.f;
      }
    } else {                  // source contiguous in k: consecutive threads take consecutive k-units
      n = it / KU; u = it - n * KU;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int k = 8 * u + i;
        x[i] = (n < J.in && k < J.out) ? __ldg(J.W + (int64_t)n * J.out + k) : 0.f;
      }
    }
    uint32_t h[4], l[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const float a0 = x[2 * p] * s, a1 = x[2 * p + 1] * s;
      const __half2 hh = __floats2half2_rn(a0, a1);
      const float2 hf = __half22float2(hh);
      const __half2 ll = __floats2half2_rn(a0 - hf.x, a1 - hf.y);
      h[p] = *reinterpret_cast<const uint32_t*>(&hh);
      l[p] = *reinterpret_cast<const uint32_t*>(&ll);
    }
    const int k0 = 8 * u;
    unsigned char* base = J.dst + (size_t)(k0 / kc) * chunk_bytes + b_offset(N, n, k0 % kc);
    *reinterpret_cast<uint4*>(base) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(base + lo_off) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}
static void prep_finish(PrepTable& T) {
  T.cta0[0] = 0;
  for (int j = 0; j < T.n; ++j) T.cta0[j + 1] = T.cta0[j] + (T.j[j].N * T.j[j].K / 8 + 1023) / 1024;
}

// ================================================================================================== critic forward sweeps
enum { FWD_TGT_NEXT = 0, FWD_TGT_S = 1, FWD_F = 2, FWD_FP = 3 };
struct FwdArgs {
  int nkinds, kind[4];
  const float* critic;         // parameter blocks (biases, w5, b5 are read from here)
  const float* target;
  const float* state;          // [B][ns]
  const float* state_next;     // [B][ns]
  float* V_out;                // [B]  (FWD_F)
  float* Vt_out;               // [B]  (FWD_TGT_S)
  int64_t B;
};

typedef ChainSmem<128, 6> CriticSmemTc;
typedef ChainSmem<256, 5> ActorSmemTc;

// 16 sines (and cosines) at once: one range check for the whole group keeps the fast path free of branches and calls
template <bool WITH_COS>
__device__ __forceinline__ void sincos16(const float* z, float* s, float* c) {
  float zm = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) zm = fmaxf(zm, fabsf(z[i]));
  if (zm > 1.0e5f || !(zm == zm)) {
    // (unrolled with scalar temporaries: a rolled loop would index z / s / c dynamically and push all three arrays -- the fast
    // path's too -- into local memory)
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const float2 r = sincos_slow(z[i]);
      s[i] = r.x;
      if (WITH_COS) c[i] = r.y;
    }
    return;
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    if (WITH_COS) sincos_fast(z[i], s[i], c[i]);
    else s[i] = sin_fast(z[i]);
  }
}
// max |accumulator| over the thread's 16-column chunks of an N-column layer (pass 1 of a row-scaled epilogue)
__device__ __forceinline__ float acc_absmax_n(const Epi& e, int N) {
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

// normalised state row -> A image (K = 16), optional ws copy; returns the row's unscale factor to ALL threads of the row
template <typename SM>
__device__ __forceinline__ float state_prologue(SM& sm, Epi& e, const cacto_sys_params& P, const float* __restrict__ src, int64_t b, bool valid, float* XNp,
                                                int64_t tile, uint32_t* amax_slot) {
  float inv = 0.f;
  if (e.cgp == 0) {
    float x[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) x[j] = 0.f;
    float m = 0.f;
    if (valid) {
#pragma unroll
      for (int j = 0; j < CACTO_MAX_NS; ++j)          // (static indices: x stays in registers)
        if (j < P.ns) {
          x[j] = normalize_component(P, j, src[b * P.ns + j]);
          m = fmaxf(m, fabsf(x[j]));
        }
    }
    const float s = pow2_scale(m, inv);
    put_a16(sm, e, 0, x, s);
    if (XNp != nullptr) {
      ws_store16(XNp, 16, tile, 0, e.row, x);
      amax_update(amax_slot, m, e.lane);
    }
  }
  return row_max4(sm, e, inv);        // inv > 0 from column group 0, 0 from the others
}

// The forward sweep is bound by the sine / cosine evaluations (96 per thread and job): ONE copy of the chunk loop serves the four
// layers and the four job kinds (runtime widths and flags) -- the first version instantiated it 12 times, 11 k instructions that
// the instruction cache could not hold (ncu: stall_no_instruction second only to the scoreboard).
__global__ void __launch_bounds__(THREADS, 1) k_tc_critic_fwd(const __grid_constant__ cacto_sys_params P, const FwdArgs A, const TcWs ws, const LayerSeq L,
                                                              int njobs) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  CriticSmemTc& sm = *reinterpret_cast<CriticSmemTc*>(smem_raw);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  chain_setup(sm, tid, warp);
  pdl_wait();            // everything above overlaps the tail of the preceding kernel (programmatic dependent launch)
  const uint32_t tmem = sm.tmem_base;
  const CriticLayout CL(P.ns);
  const int ntiles = (int)ws.tiles;
  if (warp < EPI_WARPS) {
    Epi e = epi_init(tid, tmem);
    TCU_TRACE_DECL;
#define FEV(code) do { if (tid == 0) TCU_EV(0, code); } while (0)
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) {
      const int kslot = job / ntiles;
      const int kind = kslot == 0 ? A.kind[0] : (kslot == 1 ? A.kind[1] : A.kind[2]);
      const int64_t tile = job - kslot * ntiles, b = tile * TILE + e.row;
      const bool valid = b < A.B;
      const bool tgt = kind <= FWD_TGT_S;
      const float* par = tgt ? A.target : A.critic;
      const float* US = ws.US + 8 * (tgt ? ST_TF : ST_CF);
      const float* src = kind == FWD_TGT_NEXT ? A.state_next : (kind == FWD_FP ? ws.SP : A.state);
      FEV(10);
      const float rinv = state_prologue(sm, e, P, src, b, valid, kind == FWD_F ? ws.XN : nullptr, tile, ws.amax + AM_XN);
      publish_a(sm);
      float* SNp = kind == FWD_F ? ws.SN : nullptr;
      float* CSp = kind == FWD_F ? ws.CS : (kind == FWD_FP ? ws.CSP : nullptr);
      const float* w5 = kind == FWD_FP ? nullptr : par + CL.W[4];
      float vpart = 0.f;
#pragma unroll 1
      for (int l = 0; l < 4; ++l) {
        const int N = l < 2 ? CR_H1 : CR_H3, col0 = kofs(l);
        const float us = (l == 0 ? rinv : 1.f / SIN_SCALE) * __ldg(US + l);
        const float* bias = par + (l == 0 ? CL.b[0] : (l == 1 ? CL.b[1] : (l == 2 ? CL.b[2] : CL.b[3])));
        FEV(30);
        wait_acc(sm, e);
        FEV(31);
#pragma unroll 1
        for (int ch = e.cgp; ch < N / 16; ch += 4) {
          float v[16], s[16], c[16];
          ldtm16(e.taddr + (uint32_t)(16 * ch), v);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float4 bb = __ldg(reinterpret_cast<const float4*>(bias + 16 * ch) + i);
            v[4 * i] = fmaf(v[4 * i], us, bb.x); v[4 * i + 1] = fmaf(v[4 * i + 1], us, bb.y);
            v[4 * i + 2] = fmaf(v[4 * i + 2], us, bb.z); v[4 * i + 3] = fmaf(v[4 * i + 3], us, bb.w);
          }
          if (CSp != nullptr) sincos16<true>(v, s, c);          // the target sweeps need no cosines
          else sincos16<false>(v, s, c);
          if (SNp != nullptr) ws_store16(SNp, CWT, tile, col0 + 16 * ch, e.row, s);
          if (CSp != nullptr) ws_store16(CSp, CWT, tile, col0 + 16 * ch, e.row, c);
          if (l < 3) {
            put_a16(sm, e, 16 * ch, s, SIN_SCALE);
            publish_a_group(sm, ch >> 2);             // the next layer's UMMAs start on this 64-column group
          } else if (w5 != nullptr) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 ww = __ldg(reinterpret_cast<const float4*>(w5 + 16 * ch) + i);
              vpart = fmaf(s[4 * i], ww.x, vpart); vpart = fmaf(s[4 * i + 1], ww.y, vpart);
              vpart = fmaf(s[4 * i + 2], ww.z, vpart); vpart = fmaf(s[4 * i + 3], ww.w, vpart);
            }
          }
        }
        FEV(32);
        if (l < 3) publish_a_from(sm, N / A_GROUP_K);
        FEV(33);
      }
      if (kind != FWD_FP) {
        const float V = row_sum4(sm, e, vpart) + __ldg(par + CL.b[4]);
        if (e.cgp == 0 && valid) {
          if (kind == FWD_TGT_NEXT) ws.VTN[b] = V;
          else if (kind == FWD_TGT_S) A.Vt_out[b] = V;
          else A.V_out[b] = V;
        }
      }
    }
  } else if (warp == EPI_WARPS) {
    RingState rs = {0, 0u, 0u};
    int tcu_trace_n = 0;
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) issue_job<6>(sm, L, rs, tmem, tcu_trace_n);
  } else {
    RingState rs = {0, 0u, 0u};
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) {
      const int kslot = job / ntiles;
      const int kind = kslot == 0 ? A.kind[0] : (kslot == 1 ? A.kind[1] : A.kind[2]);
      produce_job<6>(sm, L, kind <= FWD_TGT_S ? ws.S_tf : ws.S_cf, rs);
    }
  }
  chain_teardown(sm, warp);
}

// ================================================================================================== critic backward-direction sweeps
enum { BWD_G = 0, BWD_GP = 1, BWD_B = 2 };
struct BwdArgs {
  const float* critic;
  float w_S;
  int sobolev, mc;
  const float* prtg;  const float* dVdx;  const float* done;  const float* weights;   // critic step inputs [B], [B][ns], [B], [B]
  const float* V;               // [B] from the forward sweep
  float inv_B;
  float* rtg_out;  float* loss_out;
  float* grad;                  // critic gradient block (BWD_B: biases, w5, b5) / actor gradient block (BWD_GP: b3)
  int64_t B;
};

// These sweeps do little arithmetic per element; what they wait for is the workspace (cos z, extra, g, sin z: L2 / HBM latency)
// and the accumulator.  Every layer therefore issues the loads of ALL its workspace operands before it waits for the MMAs
// (they do not depend on them), so that the two latencies overlap instead of adding up.
// DET: A.grad is the kernel's partials region; CTA j writes slice j.
template <int MODE, bool DET = false>
__global__ void __launch_bounds__(THREADS, 1) k_tc_critic_bwd(const __grid_constant__ cacto_sys_params P, const BwdArgs A, const TcWs ws, const LayerSeq L,
                                                              int njobs) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  CriticSmemTc& sm = *reinterpret_cast<CriticSmemTc*>(smem_raw);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  if constexpr (DET) det_clear<CriticSmemTc>(smem_raw, tid);
  chain_setup(sm, tid, warp);
  pdl_wait();            // everything above overlaps the tail of the preceding kernel (programmatic dependent launch)
  const uint32_t tmem = sm.tmem_base;
  const CriticLayout CL(P.ns);
  const ActorLayout AL(P.ns, P.na);
  if (warp < EPI_WARPS) {
    Epi e = epi_init(tid, tmem);
    float* const colsum = DET ? det_colq<CriticSmemTc>(smem_raw) + TC_DET_COLS * e.q : sm.colsum;
    TCU_TRACE_DECL;
#define EEV(code) do { if (tid == 0) TCU_EV(0, code); } while (0)
    const float* US = ws.US + 8 * ST_CB;
    const float* w5 = A.critic + CL.W[4];
    const float* CSsrc = MODE == BWD_GP ? ws.CSP : ws.CS;
    const bool sob = MODE == BWD_B && A.sobolev;
    float w5max;
    {
      const float4 w = __ldg(reinterpret_cast<const float4*>(w5) + e.lane);         // 128 output weights: 4 per lane
      const uint32_t mb = __float_as_uint(fmaxf(fmaxf(fabsf(w.x), fabsf(w.y)), fmaxf(fabsf(w.z), fabsf(w.w))));
      w5max = __uint_as_float(__reduce_max_sync(0xffffffffu, mb));
    }
    float lsum = 0.f;
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) {
      const int64_t tile = job, b = tile * TILE + e.row;
      const bool valid = b < A.B;
      const float vz = valid ? 1.f : 0.f;
      float rinv;            // unscale of the current A image's row
      EEV(10);               // job start
      // ---- first operand (K = 128): delta_4 = w5 * cos z_4 (G, GP)  /  e_4 = vbar w5 cos z_4 + extra_4 (B)
      if (MODE != BWD_B) {
        const float s = pow2_scale(w5max, rinv);
        float c[2][16];
#pragma unroll
        for (int j = 0; j < 2; ++j) ws_load16(CSsrc, CWT, tile, kofs(3) + 16 * (e.cgp + 4 * j), e.row, c[j]);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int ch = e.cgp + 4 * j;
#pragma unroll
          for (int i = 0; i < 16; ++i) c[j][i] *= vz * __ldg(w5 + 16 * ch + i);
          if (MODE == BWD_G) ws_store16(ws.DL, CWT, tile, kofs(3) + 16 * ch, e.row, c[j]);
          put_a16(sm, e, 16 * ch, c[j], s);
        }
        if (MODE == BWD_G) amax_update(ws.amax + AM_DL, vz * w5max, e.lane);
      } else {
        // all workspace operands of the two chunks are requested before anything waits: extra_4, cos z_4; sin z_4 follows as soon
        // as the registers of cos z_4 are free
        float ev[2][16], c[2][16];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          ws_load16(ws.CS, CWT, tile, kofs(3) + 16 * (e.cgp + 4 * j), e.row, c[j]);
          if (sob) ws_load16(ws.EX, CWT, tile, kofs(3) + 16 * (e.cgp + 4 * j), e.row, ev[j]);
        }
        // value part of the loss (NeuralNetwork.py:157-158, 167-173): y, vbar; one thread per row, shared with the row's other threads
        float vb = 0.f;
        if (e.cgp == 0 && valid) {
          const float pr = A.prtg[b], wt = A.weights[b], Vb = A.V[b];
          const float dn = A.mc ? 0.f : A.done[b], vt = A.mc ? 0.f : ws.VTN[b];
          const float y = A.mc ? pr : pr + (1.f - dn) * vt;
          A.rtg_out[b] = y;
          const float er = y - Vb, k = A.sobolev ? A.w_S : 1.f, wk = wt * k * A.inv_B;
          vb = -2.f * wk * er;
          lsum += wk * er * er;
        }
        vb = row_sum4(sm, e, vb);           // vbar may be negative: exchanged as a sum (the other column groups contribute 0)
        float m = 0.f;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int ch = e.cgp + 4 * j;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            ev[j][i] = vz * (vb * __ldg(w5 + 16 * ch + i) * c[j][i] + (sob ? ev[j][i] : 0.f));
            m = fmaxf(m, fabsf(ev[j][i]));
          }
          ws_store16(ws.EE, CWT, tile, kofs(3) + 16 * ch, e.row, ev[j]);
          warp_colsum16<DET>(colsum, kofs(3) + 16 * ch, ev[j], e.lane);           // d b_4
        }
        // d w5 += sum_s vbar h_4 is a batch reduction like the other weight gradients: vbar goes to the workspace as a 4-wide
        // tensor (column 0) and k_tc_wgrad pairs it with sin z_4
        if (e.cgp == 0) {
          *ws4(ws.VB4, 4, tile, 0, e.row) = make_float4(vz * vb, 0.f, 0.f, 0.f);
          amax_update(ws.amax + AM_VB, vz * fabsf(vb), e.lane);
        }
        if (e.cgp == 0) {                                          // d b5 = sum vbar
          float t = vb;
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
          if (e.lane == 0) {
            if constexpr (DET) colsum[CWT + CR_H4] += t;
            else atomicAdd(&sm.colsum[CWT + CR_H4], t);
          }
        }
        amax_update(ws.amax + AM_EE, m, e.lane);
        m = row_max4(sm, e, m);
        const float s = pow2_scale(m, rinv);
#pragma unroll
        for (int j = 0; j < 2; ++j) put_a16(sm, e, 16 * (e.cgp + 4 * j), ev[j], s);
      }
      EEV(11);               // first operand written
      publish_a(sm);
      EEV(12);

      // ---- hidden layers 3, 2, 1 (outputs of widths 128, 64, 64 at column offsets kofs(2), kofs(1), kofs(0))
#pragma unroll 1
      for (int li = 0; li < 3; ++li) {
        const int lo = 2 - li, N = li == 0 ? CR_H3 : CR_H2, nch = N / 64, col0 = kofs(lo);
        // fetched ahead of the accumulator: cos z of the thread's chunks; with a single chunk (64-wide layers) its extra too (in c[1])
        float c[2][16];
        ws_load16(CSsrc, CWT, tile, col0 + 16 * e.cgp, e.row, c[0]);
        if (nch == 2) ws_load16(CSsrc, CWT, tile, col0 + 16 * (e.cgp + 4), e.row, c[1]);
        else if (sob) ws_load16(ws.EX, CWT, tile, col0 + 16 * e.cgp, e.row, c[1]);
        float xmax = 0.f;
        if (sob) xmax = ws.EXMAX[(int64_t)lo * ws.tiles * TILE + tile * TILE + e.row];
        EEV(20);             // operand loads issued
        wait_acc(sm, e);
        EEV(21);             // accumulator ready
        const float us = rinv * __ldg(US + li);
        const float mraw = acc_absmax_n(e, N);
        EEV(22);             // pass 1 done
        const float m = row_max4(sm, e, mraw * us + xmax);
        EEV(23);             // row exchange done
        float rnew;
        const float s = pow2_scale(m, rnew);
        float mx = 0.f;
#pragma unroll
        for (int j = 0; j < 2; ++j)
          if (j < nch) {
            const int ch = e.cgp + 4 * j;
            float v[16], x[16];
            if (sob) {
              if (nch == 1) {
#pragma unroll
                for (int i = 0; i < 16; ++i) x[i] = c[1][i];
              } else {
                ws_load16(ws.EX, CWT, tile, col0 + 16 * ch, e.row, x);
              }
            }
            ldtm16(e.taddr + (uint32_t)(16 * ch), v);
            if (MODE == BWD_B) {
#pragma unroll
              for (int i = 0; i < 16; ++i) v[i] = vz * (v[i] * us * c[j][i] + (sob ? x[i] : 0.f));
              ws_store16(ws.EE, CWT, tile, col0 + 16 * ch, e.row, v);
              warp_colsum16<DET>(colsum, col0 + 16 * ch, v, e.lane);                   // d b_l
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) v[i] *= us;
              if (MODE == BWD_G) ws_store16(ws.GG, 256, tile, col0 + 16 * ch, e.row, v);
#pragma unroll
              for (int i = 0; i < 16; ++i) v[i] *= vz * c[j][i];
              if (MODE == BWD_G) ws_store16(ws.DL, CWT, tile, col0 + 16 * ch, e.row, v);
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) mx = fmaxf(mx, fabsf(v[i]));
            if (!(MODE == BWD_B && lo == 0)) {
              put_a16(sm, e, 16 * ch, v, s);
              publish_a_group(sm, j);
            }
          }
        if (MODE == BWD_G) amax_update(ws.amax + AM_DL, mx, e.lane);
        if (MODE == BWD_B) amax_update(ws.amax + AM_EE, mx, e.lane);
        rinv = rnew;
        EEV(24);             // chunks done
        if (!(MODE == BWD_B && lo == 0)) publish_a_from(sm, nch);
        EEV(25);
      }

      if (MODE != BWD_B) {
        // ---- input layer: g_0 = delta_1 W1^T (N = 16 >= ns), one thread per row
        wait_acc(sm, e);
        if (e.cgp == 0) {
          float g0[16];
          ldtm16(e.taddr, g0);
          const float us = rinv * __ldg(US + 3);
#pragma unroll
          for (int j = 0; j < 16; ++j) g0[j] *= us;
          if (MODE == BWD_G) {
            // Sobolev loss and its seeds (NeuralNetwork.py:162-173; SURVEY.md A.3 step 3)
            float a0[16];
            float m = 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) a0[j] = 0.f;
            if (valid) {
              const float wn = A.weights[b] * A.inv_B / (float)P.nx;
#pragma unroll
              for (int j = 0; j < CACTO_MAX_NS - 1; ++j)
                if (j < P.nx) {
                  const float D = normalize_scale(P, j);
                  const float gs = D * g0[j];
                  const float diff = slog_tc(A.dVdx[b * P.ns + j]) - slog_tc(gs);
                  a0[j] = D * (-2.f * wn * diff * slog_grad_tc(gs));
                  lsum += wn * diff * diff;
                  m = fmaxf(m, fabsf(a0[j]));
                }
            }
            ws_store16(ws.A0, 16, tile, 0, e.row, a0);
            amax_update(ws.amax + AM_A0, m, e.lane);
          } else {
            // dQ/da = dV/ds' . ds'/da + dr/da; upstream gradient on the actor output = -dQ/da / B (NeuralNetwork.py:206-228)
            float d3[16];
            float m = 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) d3[j] = 0.f;
            if (valid) {
              const int ns = P.ns, na = P.na;
              float gs[CACTO_MAX_NS];                                        // dV/ds' in raw state units (one division per state, not per (state, action))
#pragma unroll
              for (int k = 0; k < CACTO_MAX_NS; ++k) gs[k] = k < ns ? normalize_scale(P, k) * g0[k] : 0.f;
#pragma unroll
              for (int j = 0; j < CACTO_MAX_NA; ++j)
                if (j < na) {
                  float qv = ws.DRDA[b * na + j];
#pragma unroll
                  for (int k = 0; k < CACTO_MAX_NS; ++k)
                    if (k < ns) qv = fmaf(gs[k], ws.FU[(b * ns + k) * na + j], qv);
                  d3[j] = -qv * A.inv_B;
                  m = fmaxf(m, fabsf(d3[j]));
                }
            }
            ws_store16(ws.D3, 16, tile, 0, e.row, d3);
            amax_update(ws.amax + AM_D3, m, e.lane);
            warp_colsum16<DET>(colsum, 0, d3, e.lane);                     // d b3
          }
        }
      }
    }
    // ---- per-CTA reductions -> global
    if (MODE == BWD_G || MODE == BWD_B) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, o);
      if constexpr (DET) {
        if (e.lane == 0) det_colq<CriticSmemTc>(smem_raw)[4 * TC_DET_COLS + e.warp] = lsum;
      } else {
        if (e.lane == 0 && lsum != 0.f && A.loss_out != nullptr) atomicAdd(A.loss_out, lsum);
      }
    }
    epi_bar();
    if constexpr (DET) {
      float* slice = A.grad + (int64_t)blockIdx.x * TC_DET_SLICE;
      if (MODE == BWD_B) det_flush<CriticSmemTc>(smem_raw, slice, CWT + CR_H4 + 1, 0, true, tid);
      else if (MODE == BWD_G) det_flush<CriticSmemTc>(smem_raw, slice, 0, 0, true, tid);
      else det_flush<CriticSmemTc>(smem_raw, slice, P.na, 2 * ACTOR_H, false, tid);
    } else if (MODE == BWD_B) {
      for (int i = tid; i < CWT + CR_H4 + 1; i += EPI_THREADS) {
        const float v = sm.colsum[i];
        if (v == 0.f) continue;
        if (i < CWT) {
          const int l = i < kofs(1) ? 0 : (i < kofs(2) ? 1 : (i < kofs(3) ? 2 : 3));
          atomicAdd(A.grad + CL.b[l] + (i - kofs(l)), v);
        } else if (i < CWT + CR_H4) {
          atomicAdd(A.grad + CL.W[4] + (i - CWT), v);
        } else {
          atomicAdd(A.grad + CL.b[4], v);
        }
      }
    } else if (MODE == BWD_GP) {
      if (tid < P.na && sm.colsum[tid] != 0.f) atomicAdd(A.grad + AL.b3 + tid, sm.colsum[tid]);
    }
  } else if (warp == EPI_WARPS) {
    RingState rs = {0, 0u, 0u};
    int tcu_trace_n = 0;
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) issue_job<6>(sm, L, rs, tmem, tcu_trace_n);
  } else {
    RingState rs = {0, 0u, 0u};
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) produce_job<6>(sm, L, ws.S_cb, rs);
  }
  chain_teardown(sm, warp);
}

// ================================================================================================== adjoint sweep (A)
template <bool DET = false>     // DET: grad is the kernel's partials region; CTA j writes slice j
__global__ void __launch_bounds__(THREADS, 1) k_tc_critic_adj(const __grid_constant__ cacto_sys_params P, const float* __restrict__ critic, float* __restrict__ grad,
                                                              const TcWs ws, const LayerSeq L, int njobs, int64_t B) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  CriticSmemTc& sm = *reinterpret_cast<CriticSmemTc*>(smem_raw);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  if constexpr (DET) det_clear<CriticSmemTc>(smem_raw, tid);
  chain_setup(sm, tid, warp);
  pdl_wait();            // everything above overlaps the tail of the preceding kernel (programmatic dependent launch)
  const uint32_t tmem = sm.tmem_base;
  const CriticLayout CL(P.ns);
  if (warp < EPI_WARPS) {
    Epi e = epi_init(tid, tmem);
    float* const colsum = DET ? det_colq<CriticSmemTc>(smem_raw) + TC_DET_COLS * e.q : sm.colsum;
    const float* US = ws.US + 8 * ST_CF;
    const float* w5 = critic + CL.W[4];
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) {
      const int64_t tile = job, b = tile * TILE + e.row;
      const float vz = b < B ? 1.f : 0.f;
      float rinv = 0.f;
      if (e.cgp == 0) {
        float a0[16];
        ws_load16(ws.A0, 16, tile, 0, e.row, a0);
        float m = 0.f;
#pragma unroll
        for (int j = 0; j < 16; ++j) m = fmaxf(m, fabsf(a0[j]));
        const float s = pow2_scale(m, rinv);
        put_a16(sm, e, 0, a0, s);
      }
      rinv = row_max4(sm, e, rinv);
      publish_a(sm);
#pragma unroll 1
      for (int l = 0; l < 4; ++l) {
        const int N = l < 2 ? CR_H1 : CR_H3, nch = N / 64, col0 = kofs(l);
        // operands of the layer, loaded before the accumulator is waited for: cos z_l and p = g_l sin z_l (g_4 = w5)
        float c[2][16], p[2][16];
#pragma unroll
        for (int j = 0; j < 2; ++j)
          if (j < nch) {
            const int ch = e.cgp + 4 * j;
            float g[16];
            ws_load16(ws.CS, CWT, tile, col0 + 16 * ch, e.row, c[j]);
            ws_load16(ws.SN, CWT, tile, col0 + 16 * ch, e.row, p[j]);
            if (l < 3) {
              ws_load16(ws.GG, 256, tile, col0 + 16 * ch, e.row, g);
#pragma unroll
              for (int i = 0; i < 16; ++i) p[j][i] *= g[i];
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) p[j][i] *= __ldg(w5 + 16 * ch + i);
            }
          }
        wait_acc(sm, e);
        const float us = rinv * __ldg(US + l);
        const float m = row_max4(sm, e, acc_absmax_n(e, N) * us);          // |a_l| = |t cos z| <= |t|
        float rnew;
        const float s = pow2_scale(m, rnew);
        float xm = 0.f, am = 0.f;
#pragma unroll
        for (int j = 0; j < 2; ++j)
          if (j < nch) {
            const int ch = e.cgp + 4 * j;
            float v[16];
            ldtm16(e.taddr + (uint32_t)(16 * ch), v);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float t = vz * v[i] * us;
              p[j][i] *= -t;                                   // extra_l = -t g_l sin z_l
              v[i] = t * c[j][i];                              // a_l = t cos z_l
              xm = fmaxf(xm, fabsf(p[j][i]));
              am = fmaxf(am, fabsf(v[i]));
            }
            ws_store16(ws.EX, CWT, tile, col0 + 16 * ch, e.row, p[j]);
            if (l < 3) {
              ws_store16(ws.AA, 256, tile, col0 + 16 * ch, e.row, v);
              put_a16(sm, e, 16 * ch, v, s);
              publish_a_group(sm, j);
            } else {
              warp_colsum16<DET>(colsum, 16 * ch, v, e.lane);                  // d w5 += sum_s a_4
            }
          }
        if (l < 3) amax_update(ws.amax + AM_AA, am, e.lane);
        xm = row_max4(sm, e, xm);
        if (e.cgp == 0) ws.EXMAX[(int64_t)l * ws.tiles * TILE + tile * TILE + e.row] = xm;
        rinv = rnew;
        if (l < 3) publish_a_from(sm, nch);
      }
    }
    epi_bar();
    if constexpr (DET) det_flush<CriticSmemTc>(smem_raw, grad + (int64_t)blockIdx.x * TC_DET_SLICE, CR_H4, CWT, false, tid);
    else if (tid < CR_H4 && sm.colsum[tid] != 0.f) atomicAdd(grad + CL.W[4] + tid, sm.colsum[tid]);
  } else if (warp == EPI_WARPS) {
    RingState rs = {0, 0u, 0u};
    int tcu_trace_n = 0;
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) issue_job<6>(sm, L, rs, tmem, tcu_trace_n);
  } else {
    RingState rs = {0, 0u, 0u};
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) produce_job<6>(sm, L, ws.S_cf, rs);
  }
  chain_teardown(sm, warp);
}

// ================================================================================================== actor forward / backward
// One LeakyReLU(0.3) layer of 256 units, forward: h = lrelu(acc * us + b); keeps h, next A image row-scaled by a bound on |z|.
template <typename SM>
__device__ __forceinline__ float actor_fwd_layer(SM& sm, Epi& e, float us, const float* __restrict__ bias, float* Hp, int64_t tile, uint32_t* amax_slot) {
  float m = 0.f;
#pragma unroll 1
  for (int ch = e.cgp; ch < ACTOR_H / 16; ch += 4) {
    float v[16];
    ldtm16(e.taddr + (uint32_t)(16 * ch), v);
#pragma unroll
    for (int i = 0; i < 16; ++i) m = fmaxf(m, fabsf(fmaf(v[i], us, __ldg(bias + 16 * ch + i))));
  }
  amax_update(amax_slot, m, e.lane);
  m = row_max4(sm, e, m);
  float rnew;
  const float s = pow2_scale(m, rnew);
#pragma unroll 1
  for (int ch = e.cgp; ch < ACTOR_H / 16; ch += 4) {
    float v[16], h[16];
    ldtm16(e.taddr + (uint32_t)(16 * ch), v);
#pragma unroll
    for (int i = 0; i < 16; ++i) h[i] = leaky(fmaf(v[i], us, __ldg(bias + 16 * ch + i)));
    ws_store16(Hp, ACTOR_H, tile, 16 * ch, e.row, h);
    put_a16(sm, e, 16 * ch, h, s);
    publish_a_group(sm, ch >> 2);                 // 256 columns = all A_GROUPS groups, one per iteration
  }
  return rnew;
}

__global__ void __launch_bounds__(THREADS, 1) k_tc_actor_fwd(const __grid_constant__ cacto_sys_params P, const float* __restrict__ actor,
                                                             const float* __restrict__ state, float* __restrict__ actions_out, const TcWs ws,
                                                             const LayerSeq L, int njobs, int64_t B) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  ActorSmemTc& sm = *reinterpret_cast<ActorSmemTc*>(smem_raw);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  chain_setup(sm, tid, warp);
  pdl_wait();            // everything above overlaps the tail of the preceding kernel (programmatic dependent launch)
  const uint32_t tmem = sm.tmem_base;
  const ActorLayout AL(P.ns, P.na);
  if (warp < EPI_WARPS) {
    Epi e = epi_init(tid, tmem);
    const float* US = ws.US + 8 * ST_AF;
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) {
      const int64_t tile = job, b = tile * TILE + e.row;
      const bool valid = b < B;
      float rinv = state_prologue(sm, e, P, state, b, valid, ws.XNA, tile, ws.amax + AM_XNA);
      publish_a(sm);
      wait_acc(sm, e);
      rinv = actor_fwd_layer(sm, e, rinv * US[0], actor + AL.b1, ws.H1, tile, ws.amax + AM_H1);      // (publishes the next A image group by group)
      wait_acc(sm, e);
      rinv = actor_fwd_layer(sm, e, rinv * US[1], actor + AL.b2, ws.H2, tile, ws.amax + AM_H2);
      wait_acc(sm, e);
      if (e.cgp == 0) {
        float a[16];
        ldtm16(e.taddr, a);
        const float us = rinv * US[2];
        if (valid) {
#pragma unroll
          for (int j = 0; j < CACTO_MAX_NA; ++j)
            if (j < P.na) {
              const float u = fmaf(a[j], us, __ldg(actor + AL.b3 + j));
              ws.ACT[b * P.na + j] = u;
              if (actions_out != nullptr) actions_out[b * P.na + j] = u;
            }
        }
      }
    }
  } else if (warp == EPI_WARPS) {
    RingState rs = {0, 0u, 0u};
    int tcu_trace_n = 0;
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) issue_job<5>(sm, L, rs, tmem, tcu_trace_n);
  } else {
    RingState rs = {0, 0u, 0u};
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) produce_job<5>(sm, L, ws.S_af, rs);
  }
  chain_teardown(sm, warp);
}

// per sample: s' = f(s, a) (fp64 arithmetic on the fp32-rounded inputs, quirk Q13), ds'/da (normalised, time row 0), dr/da
// (NeuralNetwork.py:188, 199-204) -- the per-sample block of k_actor_grad (update.cu)
template <int SYS>
__global__ void __launch_bounds__(128) k_tc_actor_env(const __grid_constant__ cacto_sys_params P, const float* __restrict__ state,
                                                      const double* __restrict__ term, const TcWs ws, int64_t B) {
  constexpr int NX = SysDims<SYS>::NX, NA = SysDims<SYS>::NA, NS = NX + 1;
  pdl_wait();
  const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double x[NS], u[NA], xn[NS], Fu[NX * NA];
#pragma unroll
  for (int j = 0; j < NS; ++j) x[j] = (double)state[b * NS + j];
  float uf[NA], g[NA];
#pragma unroll
  for (int j = 0; j < NA; ++j) {
    uf[j] = ws.ACT[b * NA + j];
    u[j] = (double)uf[j];
  }
  sys_step_Fu<SYS, double>(P, x, u, xn, Fu);
  xn[NX] = x[NX] + P.dt;
#pragma unroll
  for (int j = 0; j < NS; ++j) ws.SP[b * NS + j] = (float)xn[j];
#pragma unroll
  for (int i = 0; i < NX; ++i) {
    const double inv = P.normalize ? 1.0 / P.state_norm[i] : 1.0;
#pragma unroll
    for (int j = 0; j < NA; ++j) ws.FU[(b * NS + i) * NA + j] = (float)(Fu[i * NA + j] * inv);
  }
#pragma unroll
  for (int j = 0; j < NA; ++j) ws.FU[(b * NS + NX) * NA + j] = 0.f;
  const double tm = term[b];
  const float w6 = (float)(tm * P.w_terminal[6] + (1.0 - tm) * P.w_running[6]);     // NeuralNetwork.py:201
  sys_dr_da<SYS, float>(P, w6, uf, g);
#pragma unroll
  for (int j = 0; j < NA; ++j) ws.DRDA[b * NA + j] = g[j];
}

template <bool DET = false>     // DET: grad is the kernel's partials region; CTA j writes slice j
__global__ void __launch_bounds__(THREADS, 1) k_tc_actor_bwd(const __grid_constant__ cacto_sys_params P, float* __restrict__ grad, const TcWs ws,
                                                             const LayerSeq L, int njobs, int64_t B) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  ActorSmemTc& sm = *reinterpret_cast<ActorSmemTc*>(smem_raw);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  if constexpr (DET) det_clear<ActorSmemTc>(smem_raw, tid);
  chain_setup(sm, tid, warp);
  pdl_wait();            // everything above overlaps the tail of the preceding kernel (programmatic dependent launch)
  const uint32_t tmem = sm.tmem_base;
  const ActorLayout AL(P.ns, P.na);
  if (warp < EPI_WARPS) {
    Epi e = epi_init(tid, tmem);
    float* const colsum = DET ? det_colq<ActorSmemTc>(smem_raw) + TC_DET_COLS * e.q : sm.colsum;
    const float* US = ws.US + 8 * ST_AB;
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) {
      const int64_t tile = job, b = tile * TILE + e.row;
      const float vz = b < B ? 1.f : 0.f;
      float rinv = 0.f;
      if (e.cgp == 0) {
        float d3[16];
        ws_load16(ws.D3, 16, tile, 0, e.row, d3);
        float m = 0.f;
#pragma unroll
        for (int j = 0; j < 16; ++j) m = fmaxf(m, fabsf(d3[j]));
        const float s = pow2_scale(m, rinv);
        put_a16(sm, e, 0, d3, s);
      }
      rinv = row_max4(sm, e, rinv);
      publish_a(sm);
      // e2 = (d3 W3^T) * lrelu'(z2), then e1 = (e2 W2^T) * lrelu'(z1)
      for (int l = 0; l < 2; ++l) {
        float* Hp = l == 0 ? ws.H2 : ws.H1;
        float* Ep = l == 0 ? ws.E2 : ws.E1;
        // lrelu'(z) = 1 (h > 0) or 0.3: the signs of the 64 hidden units of this thread, fetched before the accumulator is waited for
        uint64_t pos = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float h[16];
          ws_load16(Hp, ACTOR_H, tile, 16 * (e.cgp + 4 * j), e.row, h);
#pragma unroll
          for (int i = 0; i < 16; ++i) pos |= (uint64_t)(h[i] > 0.f ? 1u : 0u) << (16 * j + i);
        }
        wait_acc(sm, e);
        const float us = rinv * __ldg(US + l);
        const float m = row_max4(sm, e, acc_absmax_n(e, ACTOR_H) * us);
        float rnew;
        const float s = pow2_scale(m, rnew);
        float mx = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int ch = e.cgp + 4 * j;
          float v[16];
          ldtm16(e.taddr + (uint32_t)(16 * ch), v);
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            v[i] *= vz * us * (((pos >> (16 * j + i)) & 1ull) ? 1.f : LEAKY_ALPHA);
            mx = fmaxf(mx, fabsf(v[i]));
          }
          ws_store16(Ep, ACTOR_H, tile, 16 * ch, e.row, v);
          warp_colsum16<DET>(colsum, l * ACTOR_H + 16 * ch, v, e.lane);        // d b2 | d b1
          if (l == 0) {
            put_a16(sm, e, 16 * ch, v, s);
            publish_a_group(sm, j);
          }
        }
        amax_update(ws.amax + (l == 0 ? AM_E2 : AM_E1), mx, e.lane);
        rinv = rnew;
      }
    }
    epi_bar();
    if constexpr (DET) {
      det_flush<ActorSmemTc>(smem_raw, grad + (int64_t)blockIdx.x * TC_DET_SLICE, 2 * ACTOR_H, 0, false, tid);
    } else {
      for (int i = tid; i < 2 * ACTOR_H; i += EPI_THREADS) {
        const float v = sm.colsum[i];
        if (v != 0.f) atomicAdd(grad + (i < ACTOR_H ? AL.b2 + i : AL.b1 + (i - ACTOR_H)), v);
      }
    }
  } else if (warp == EPI_WARPS) {
    RingState rs = {0, 0u, 0u};
    int tcu_trace_n = 0;
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) issue_job<5>(sm, L, rs, tmem, tcu_trace_n);
  } else {
    RingState rs = {0, 0u, 0u};
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) produce_job<5>(sm, L, ws.S_ab, rs);
  }
  chain_teardown(sm, warp);
}

// ================================================================================================== weight gradients
// dW[m][n] += sum over samples of X1[s][m] E1[s][n] (+ X2[s][m] E2[s][n]): UMMA M = 128 features (zero-padded), N outputs, K = samples.
// Operands come from ws4 tensors: the 8 consecutive samples of 4 features are 128 contiguous bytes = four fp16 k-units.
// A CTA owns (job, slice of the sample tiles); stages of 64 samples; both operand images are built by the 16 worker warps
// (scales from the per-tensor absmax table), one accumulator per term in TMEM (columns [0, N), [N, 2N)).
struct WgOperand { const float* p; int W, c0, amax; };      // ws4 tensor, its width, first column, absmax slot (-1: |x| <= 1)
struct WgJob {
  WgOperand X[2], E[2];
  int nterms, M, N, N_real, ld, ldn;   // M real features (<= 128), N padded outputs, N_real written outputs; out[m * ld + n * ldn]
  float* out;
};
struct WgTable {
  int njobs;
  WgJob j[8];
  int cta0[9];                         // CTAs [cta0[j], cta0[j + 1]) share the sample tiles of job j
};
constexpr int WG_KS = 64;                                   // samples per stage
constexpr int WG_LBO_A = LBO_A + 16;                        // padded k-unit strides: conflict-free 16-byte stores from consecutive k-units
constexpr int WG_A_IMG = (WG_KS / 8) * WG_LBO_A;            // bytes of the hi (or lo) A image of a stage
constexpr int WG_B_IMG = (WG_KS / 8) * ((256 / 8) * 128 + 16);
struct WgSmem {
  alignas(1024) unsigned char A[2][2][WG_A_IMG];            // [stage][hi | lo]
  alignas(1024) unsigned char Bm[2][2][WG_B_IMG];
  uint64_t full[2], empty[2], d_full;
  uint32_t tmem_base;
};

// Operand images of a stage, built with stmatrix.trans: a warp takes an 8-feature octet x 32 samples ("unit").  Lane t loads, for each
// of the four 8-sample octets, the feature PAIR t % 4 of sample t / 4 (8 bytes; the 8 lanes of a pair column read 8 consecutive
// rows of one ws4 group = one full 128-byte line), scales, splits into fp16 hi / lo, and holds exactly the m8n8 fragment
// (row = sample, column pair = feature pair) of four matrices; stmatrix.x4.trans writes them transposed -- memory row = feature,
// 8 consecutive samples = one 16-byte K-major unit (k = sample) -- 512 bytes per instruction.
// (First version: one thread gathered 8 samples x 4 features with eight 16-byte loads 128 bytes apart; every load instruction of a
// warp touched 32 lines, the small L1 beside 198 KB of shared memory thrashed, and the actor's dW2 took 315 us.  Second version:
// coalesced float4 loads and 2-byte scatter stores -- 96 STS.U16 per thread and stage, the issue slots and the shared-memory store
// wavefronts of the kernel.)
__device__ __forceinline__ void stsm_x4_trans(uint32_t addr, const uint32_t (&r)[4]) {
  asm volatile("stmatrix.sync.aligned.m8n8.x4.trans.shared.b16 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
}
__device__ __forceinline__ void wg_put_unit(const float2 (&f)[4], float scale, uint32_t hi_addr, uint32_t lo_addr) {
  uint32_t h[4], l[4];
#ifdef WG_EXP_NO_CONVERT      // timing experiment only: the loads stay alive through a never-true test
  if (f[0].x + f[1].x + f[2].x + f[3].x + f[0].y + f[1].y + f[2].y + f[3].y != 12345.678f) return;
#endif
#pragma unroll
  for (int m = 0; m < 4; ++m) split_pair(f[m].x, f[m].y, scale, h[m], l[m]);
  stsm_x4_trans(hi_addr, h);
  stsm_x4_trans(lo_addr, l);
}
// the feature pair (8 F + 2 pr, + 1) of sample `row` of a ws4 tensor; zero beyond its last column group
__device__ __forceinline__ float2 wg_load_pair(const WgOperand& O, int64_t tile, int feature, int row, int group_limit) {
  const int g = feature >> 2;
  if (g >= group_limit) return make_float2(0.f, 0.f);
#ifdef WG_EXP_NO_LOAD         // timing experiment only
  return make_float2(1e-3f * (float)row, 1e-3f * (float)feature);
#endif
  return __ldg(reinterpret_cast<const float2*>(ws4(O.p, O.W, tile, O.c0 + 4 * g, row)) + ((feature >> 1) & 1));
}

#ifdef TCU_TRACE   // events of the first CTA of the second-to-last job (a large one in both tables); codes 100+
#define WGEV(role, code)                                                                                                      \
  do {                                                                                                                        \
    if ((int)blockIdx.x == T.cta0[T.njobs - 2] && g_tcu_trace != nullptr && (threadIdx.x & 31) == 0 && tcu_trace_n < TCU_TRACE_N) \
      g_tcu_trace[(role) * TCU_TRACE_N + tcu_trace_n++] = (clock64() << 8) | (long long)(code);                               \
  } while (0)
#else
#define WGEV(role, code) do { } while (0)
#endif
__global__ void __launch_bounds__(THREADS, 1) k_tc_wgrad(const WgTable T, const TcWs ws) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  WgSmem& sm = *reinterpret_cast<WgSmem*>(smem_raw);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  int ji = 0;
  while (ji + 1 < T.njobs && (int)blockIdx.x >= T.cta0[ji + 1]) ++ji;
  const WgJob& J = T.j[ji];
  const int nct = T.cta0[ji + 1] - T.cta0[ji], ci = blockIdx.x - T.cta0[ji];
  // the CTAs of a job share its 64-sample half tiles ("units"); a stage = one term of one unit
  const int64_t units = ws.tiles * (TILE / WG_KS), u0 = units * ci / nct, u1 = units * (ci + 1) / nct;
  const int nstages = (int)(u1 - u0) * J.nterms;
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) { mbar_init(&sm.full[s], EPI_THREADS); mbar_init(&sm.empty[s], 1); }
    mbar_init(&sm.d_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EPI_WARPS) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sm.tmem_base)), "r"(256));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();
  const uint32_t tmem = sm.tmem_base;
  const int N = J.N, lboB = (N / 8) * 128 + 16;
  TCU_TRACE_DECL;
#ifdef WG_CTA_TIMES        // debug builds only: [start, end] of every CTA on the global timer (ns)
  if (tid == 0 && g_tcu_trace != nullptr) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g_tcu_trace[2 * blockIdx.x]));
#endif
  if (nstages > 0) {
    if (warp < EPI_WARPS) {
      if (tid == 0) WGEV(0, 100);
      float sx[2], se[2], unscale[2];
      for (int t = 0; t < J.nterms; ++t) {
        float ix, ie;
        sx[t] = pow2_scale(J.X[t].amax >= 0 ? __uint_as_float(ws.amax[J.X[t].amax]) : 1.f, ix);
        se[t] = pow2_scale(J.E[t].amax >= 0 ? __uint_as_float(ws.amax[J.E[t].amax]) : 1.f, ie);
        unscale[t] = ix * ie;
      }
      const int Mg = (J.M + 3) / 4;                       // feature groups of 4 that hold real features
      const int lane_ = tid & 31, srow = lane_ >> 2, pr = lane_ & 3;       // fragment coordinates: sample within the octet, feature pair
      const int smat = lane_ >> 3, srow8 = lane_ & 7;                      // stmatrix address duty: row srow8 of matrix smat
      const int n8 = N / 8, nB = 2 * n8;                                  // B units of a stage
      int st = 0;
      uint32_t ph = 0;
      bool zeroed = false;
      // stage k of this CTA = (unit u0 + k / nterms, term k % nterms).  All operand loads of a stage are
      // issued before its buffer is waited for (the MMAs of the stage two steps back).  The stage loop is memory-bound: in-kernel trace
      // (scratch build with -DTCU_TRACE) of a 96 KB stage = 4 k cycles until the loads are issued (LSU queue full: the SM's share of the
      // HBM bandwidth is 23 B / cycle) + 2.5 k cycles until the last value has arrived and is converted; issuing the next stage's loads
      // unit by unit between the conversions (tried) only moves the stall: a warp blocked on a load cannot convert either.
      float2 fa[2][4], fb[4][4];
      for (int k = 0; k < nstages; ++k) {
        const int t = J.nterms == 2 ? (k & 1) : 0;
        const int64_t unit_ = u0 + (J.nterms == 2 ? (k >> 1) : k), tile = unit_ >> 1;
        const int row0 = (int)(unit_ & 1) * WG_KS + srow;
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int unit = warp + EPI_WARPS * u, F = unit & 15, h = unit >> 4;
#pragma unroll
          for (int m = 0; m < 4; ++m) fa[u][m] = wg_load_pair(J.X[t], tile, 8 * F + 2 * pr, row0 + 32 * h + 8 * m, Mg);
        }
        const int egl = (J.E[t].W - J.E[t].c0 + 3) / 4;            // column groups of E that exist (a narrow E is zero-padded to N)
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int unit = warp + EPI_WARPS * u;
          if (unit < nB) {
            const int F = unit % n8, h = unit / n8;
#pragma unroll
            for (int m = 0; m < 4; ++m) fb[u][m] = wg_load_pair(J.E[t], tile, 8 * F + 2 * pr, row0 + 32 * h + 8 * m, egl);
          }
        }
        if (tid == 0) WGEV(0, 110);          // loads issued
        mbar_wait(&sm.empty[st], ph ^ 1u);
        if (tid == 0) WGEV(0, 111);          // stage buffer free
        const uint32_t ah = smem_u32(sm.A[st][0]), al = smem_u32(sm.A[st][1]), bh = smem_u32(sm.Bm[st][0]), bl = smem_u32(sm.Bm[st][1]);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int unit = warp + EPI_WARPS * u, F = unit & 15, h = unit >> 4;
          const uint32_t off = (uint32_t)((4 * h + smat) * WG_LBO_A + F * 128 + srow8 * 16);
          if (2 * F < Mg || !zeroed) wg_put_unit(fa[u], sx[t], ah + off, al + off);      // octets beyond M stay zero once written
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int unit = warp + EPI_WARPS * u;
          if (unit < nB) {
            const int F = unit % n8, h = unit / n8;
            const uint32_t off = (uint32_t)((4 * h + smat) * lboB + F * 128 + srow8 * 16);
            wg_put_unit(fb[u], se[t], bh + off, bl + off);
          }
        }
        if (st == 1) zeroed = true;          // both stage buffers hold zeros in the feature octets beyond M from now on
        fence_async_smem();
        mbar_arrive(&sm.full[st]);
        if (tid == 0) WGEV(0, 112);          // converted, published
        if (++st == 2) { st = 0; ph ^= 1u; }
      }
      // ---- epilogue: thread <-> feature row; 16-byte vector reductions into the gradient block
      mbar_wait(&sm.d_full, 0u);
      tc_fence_after();
      if (tid == 0) WGEV(0, 120);                // accumulators complete
      const int wq = warp & 3, cgp = warp >> 2, lane = tid & 31, m = 32 * wq + lane;
      const uint32_t taddr = tmem + ((uint32_t)(32 * wq) << 16);
      for (int ch = cgp; ch < N / 16; ch += 4) {
        float v[16], w[16];
        ldtm16(taddr + (uint32_t)(16 * ch), v);
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] *= unscale[0];
        if (J.nterms == 2) {
          ldtm16(taddr + (uint32_t)(N + 16 * ch), w);
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = fmaf(w[i], unscale[1], v[i]);
        }
        // the CTA's partial block [128][N] (plain 64-byte stores; k_tc_wgrad_reduce sums the slices of a job in a fixed order:
        // 16-byte vector reductions straight into dW ran at ~4 per ns chip-wide -- 317 us for the actor's 1.2 M -- and made the
        // gradient bits depend on the arrival order)
        // layout [column group of 4][feature row][4]: every store instruction of a warp writes 512 contiguous bytes
        float4* o = reinterpret_cast<float4*>(ws.PART + (int64_t)blockIdx.x * TILE * 256) + (4 * ch) * TILE + m;
#pragma unroll
        for (int i = 0; i < 4; ++i) o[i * TILE] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
      }
      if (tid == 0) WGEV(0, 121);                // partial block written
      tc_fence_before();
    } else if (warp == EPI_WARPS) {
      const uint32_t idesc = umma_idesc(N);
      int st = 0;
      uint32_t ph = 0;
      int k = 0;
      for (int64_t unit_ = u0; unit_ < u1; ++unit_)
        for (int t = 0; t < J.nterms; ++t, ++k) {
            mbar_wait(&sm.full[st], ph);
            tc_fence_after();
            WGEV(1, 130);                        // stage images present
            if (elect_one()) {
              const uint32_t a_hi = smem_u32(sm.A[st][0]), a_lo = smem_u32(sm.A[st][1]), b_hi = smem_u32(sm.Bm[st][0]), b_lo = smem_u32(sm.Bm[st][1]);
              const bool first = unit_ == u0;
#ifdef WG_EXP_NO_MMA           // timing experiment only
              for (int ks = 0; ks < (first ? 1 : 0); ++ks) {
#else
              for (int ks = 0; ks < WG_KS / 16; ++ks) {
#endif
                const uint64_t ah = umma_desc(a_hi + ks * 2 * WG_LBO_A, WG_LBO_A), al = umma_desc(a_lo + ks * 2 * WG_LBO_A, WG_LBO_A);
                const uint64_t bh = umma_desc(b_hi + ks * 2 * lboB, lboB), bl = umma_desc(b_lo + ks * 2 * lboB, lboB);
                const uint32_t d = tmem + (uint32_t)(t * N);
                umma_f16(d, ah, bh, idesc, (first && ks == 0) ? 0u : 1u);
                umma_f16(d, ah, bl, idesc, 1u);
                umma_f16(d, al, bh, idesc, 1u);
              }
              umma_commit(&sm.empty[st]);
              if (k == nstages - 1) umma_commit(&sm.d_full);
            }
            __syncwarp();
            if (++st == 2) { st = 0; ph ^= 1u; }
          }
    }
  }
  tc_fence_before();
  __syncthreads();
#ifdef WG_CTA_TIMES
  if (tid == 0 && g_tcu_trace != nullptr) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g_tcu_trace[2 * blockIdx.x + 1]));
#endif
  if (warp == EPI_WARPS) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(256));
}

// dW[m][n] += sum over the CTAs of the job of their partial blocks, in a fixed order (deterministic): WGR_LANES lanes per output
// float4 take every WGR_LANES-th slice, then a shuffle tree.  Consecutive lane groups take consecutive feature rows m of one column
// group (the partial blocks are [column group][m][4]: 16 contiguous bytes per row)
constexpr int WGR_LANES = 16, WGR_OUT = 256 / WGR_LANES;         // lanes per output, outputs per block
__global__ void __launch_bounds__(256) k_tc_wgrad_reduce(const WgTable T, const TcWs ws) {
  pdl_wait();
  const WgJob& J = T.j[blockIdx.y];
  const int n4 = J.N / 4, idx = blockIdx.x * WGR_OUT + (threadIdx.x / WGR_LANES), part = threadIdx.x % WGR_LANES;
  const bool live = idx < J.M * n4;
  const int cg = live ? idx / J.M : 0, m = live ? idx - cg * J.M : 0, c = 4 * cg;
  const int c0 = T.cta0[blockIdx.y], nct = T.cta0[blockIdx.y + 1] - c0;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (live && c < J.N_real) {
#pragma unroll 4
    // (every CTA of a job wrote its block: wg_assign never gives a job more CTAs than it has units.  An earlier version re-derived
    //  "did CTA ci get a unit" here with two 64-bit divisions per slice -- ncu: 18 us for the actor's reduce, all of it integer division)
    for (int ci = part; ci < nct; ci += WGR_LANES) {
      const float4 p = __ldg(reinterpret_cast<const float4*>(ws.PART + (int64_t)(c0 + ci) * TILE * 256) + cg * TILE + m);
      acc.x += p.x; acc.y += p.y; acc.z += p.z; acc.w += p.w;
    }
  }
#pragma unroll
  for (int o = 1; o < WGR_LANES; o <<= 1) {
    acc.x += __shfl_xor_sync(0xffffffffu, acc.x, o);
    acc.y += __shfl_xor_sync(0xffffffffu, acc.y, o);
    acc.z += __shfl_xor_sync(0xffffffffu, acc.z, o);
    acc.w += __shfl_xor_sync(0xffffffffu, acc.w, o);
  }
  if (!live || part != 0 || c >= J.N_real) return;
  float* o = J.out + (int64_t)m * J.ld + (int64_t)c * J.ldn;
  if (J.ldn == 1 && c + 3 < J.N_real && (reinterpret_cast<uintptr_t>(o) & 15) == 0) {      // one 16-byte read-modify-write
    float4 g = *reinterpret_cast<float4*>(o);
    g.x += acc.x; g.y += acc.y; g.z += acc.z; g.w += acc.w;
    *reinterpret_cast<float4*>(o) = g;
    return;
  }
  o[0] += acc.x;
  if (c + 1 < J.N_real) o[J.ldn] += acc.y;
  if (c + 2 < J.N_real) o[2 * J.ldn] += acc.z;
  if (c + 3 < J.N_real) o[3 * J.ldn] += acc.w;
}

// grad[map(i)] += sum_j part[r][j][i] for each region r in order (slices j in order, from 0.0f); the loss entry into loss[0]
__global__ void __launch_bounds__(256) k_tc_det_reduce(const float* __restrict__ part, int regions, int slices, int is_critic, int ns, int na,
                                                       float* __restrict__ grad, float* __restrict__ loss) {
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= TC_DET_SLICE) return;
  int64_t g = -1;
  if (is_critic) {
    const CriticLayout CL(ns);
    if (i < CWT) {
      const int l = i < kofs(1) ? 0 : (i < kofs(2) ? 1 : (i < kofs(3) ? 2 : 3));
      g = CL.b[l] + (i - kofs(l));
    } else if (i < CWT + CR_H4) {
      g = CL.W[4] + (i - CWT);
    } else if (i == CWT + CR_H4) {
      g = CL.b[4];
    }
  } else {
    const ActorLayout AL(ns, na);
    if (i < ACTOR_H) g = AL.b2 + i;
    else if (i < 2 * ACTOR_H) g = AL.b1 + (i - ACTOR_H);
    else if (i < 2 * ACTOR_H + na) g = AL.b3 + (i - 2 * ACTOR_H);
  }
  const bool is_loss = is_critic && i == TC_DET_LOSS && loss != nullptr;
  if (g < 0 && !is_loss) return;
  for (int r = 0; r < regions; ++r) {
    float s = 0.f;
    for (int j = 0; j < slices; ++j) s += part[((int64_t)r * slices + j) * TC_DET_SLICE + i];
    if (g >= 0) grad[g] += s;
    else loss[0] += s;
  }
}

// ================================================================================================== host side
static int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }
// every kernel of the update chain is launched with the programmatic-serialization attribute and calls pdl_wait() (common.cuh)
template <typename... P, typename... A>
static cudaError_t launch_tc(void (*kernel)(P...), dim3 grid, unsigned block, size_t smem, cudaStream_t st, A&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, P(args)...);
}

// carve the caller's workspace; returns the bytes used (base may be NULL to size it)
static int64_t tc_ws_layout(unsigned char* base, int64_t B, int ns, int na, TcWs* out) {
  const int64_t tiles = (B + TILE - 1) / TILE, rows = tiles * TILE;
  int64_t off = 0;
  TcWs w;
  memset(&w, 0, sizeof(w));
  auto take = [&](int64_t bytes) {
    unsigned char* p = base ? base + off : nullptr;
    off = align_up(off + bytes, 1024);
    return p;
  };
  auto f = [&](int64_t width) { return reinterpret_cast<float*>(take(rows * width * 4)); };
  w.XN = f(16); w.CS = f(CWT); w.SN = f(CWT); w.GG = f(256); w.DL = f(CWT); w.A0 = f(16); w.AA = f(256); w.EX = f(CWT); w.EE = f(CWT);
  w.VTN = f(1); w.VBAR = f(1); w.EXMAX = f(4); w.VB4 = f(4);
  w.XNA = f(16); w.H1 = f(ACTOR_H); w.H2 = f(ACTOR_H); w.CSP = f(CWT); w.D3 = f(16); w.E2 = f(ACTOR_H); w.E1 = f(ACTOR_H);
  w.ACT = f(na); w.SP = f(ns); w.FU = f((int64_t)ns * na); w.DRDA = f(na);
  w.PART = reinterpret_cast<float*>(take((int64_t)WG_MAX_CTAS * TILE * 256 * 4));
  const LayerSeq cf = seq_critic_fwd(), cb = seq_critic_bwd(4), af = seq_actor_fwd(), ab = seq_actor_bwd();
  w.S_tf = take(stream_bytes(cf)); w.S_cf = take(stream_bytes(cf)); w.S_cb = take(stream_bytes(cb));
  w.S_af = take(stream_bytes(af)); w.S_ab = take(stream_bytes(ab));
  w.US = reinterpret_cast<float*>(take(5 * 8 * 4));
  w.amax = reinterpret_cast<uint32_t*>(take(AM_COUNT * 4));
  w.tiles = tiles;
  if (out) *out = w;
  return off;
}

// image jobs of one network in one orientation, appended to T
static void prep_critic(PrepTable& T, const float* w, int ns, bool fwd, unsigned char* dst, float* us) {
  const CriticLayout L(ns);
  const LayerSeq S = fwd ? seq_critic_fwd() : seq_critic_bwd(4);
  for (int i = 0; i < 4; ++i) {
    const int l = fwd ? i : 3 - i;                 // critic layer whose kernel this image holds
    PrepJob& J = T.j[T.n++];
    J.W = w + L.W[l]; J.in = L.in[l]; J.out = L.out[l]; J.K = S.K[i]; J.N = S.N[i]; J.fwd = fwd ? 1 : 0; J.dst = dst; J.unscale = us + i;
    dst += (int64_t)S.K[i] * S.N[i] * 4;
  }
}
static void prep_actor(PrepTable& T, const float* w, int ns, int na, bool fwd, unsigned char* dst, float* us) {
  const ActorLayout L(ns, na);
  const int64_t Wo[3] = {L.W1, L.W2, L.W3};
  const int in[3] = {ns, ACTOR_H, ACTOR_H}, out[3] = {ACTOR_H, ACTOR_H, na};
  const LayerSeq S = fwd ? seq_actor_fwd() : seq_actor_bwd();
  for (int i = 0; i < S.n; ++i) {
    const int l = fwd ? i : 2 - i;
    PrepJob& J = T.j[T.n++];
    J.W = w + Wo[l]; J.in = in[l]; J.out = out[l]; J.K = S.K[i]; J.N = S.N[i]; J.fwd = fwd ? 1 : 0; J.dst = dst; J.unscale = us + i;
    dst += (int64_t)S.K[i] * S.N[i] * 4;
  }
}

template <typename K>
static int tc_smem_attr(K k, size_t bytes) {
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  return e == cudaSuccess ? 0 : (int)e;
}
static int num_sms() {
  int dev = 0, n = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  return n;
}
// Split `ctas` CTAs over the jobs so that the slowest CTA is as fast as possible.  A CTA takes whole units (64-sample half tiles);
// a unit of a job costs one stage per term, and a stage costs -- per-CTA global-timer stamps of a -DWG_CTA_TIMES build,
// B = 16 384 -- a latency-bound 1.15 us + 0.034 us per KB of the E operand (N / 4 KB) + next to nothing for the X operand:
// 1.7 us at N = 64, 2.3 us at N = 128, 3.3-3.4 us at N = 256, whatever M is.  (The first model, 0.8 us + bytes at 40 B / ns
// over whole tiles, gave the 7 x 64 job of the critic 22 CTAs that ran 43 us beside 32 us for the rest.)
static void wg_assign(WgTable& T, int ctas, int64_t tiles) {
  const int64_t units = tiles * (TILE / WG_KS);
  double unit_cost[8];
  for (int j = 0; j < T.njobs; ++j) unit_cost[j] = T.j[j].nterms * (1.15 + 0.034 * (T.j[j].N / 4) + 0.004 * ((T.j[j].M + 3) / 4));
  // smallest makespan for which the CTAs suffice: job j needs ceil(units / floor(makespan / unit_cost[j])) CTAs
  auto need = [&](double span) {
    int64_t total = 0;
    for (int j = 0; j < T.njobs; ++j) {
      const int64_t per = (int64_t)(span / unit_cost[j]);
      if (per < 1) return (int64_t)1 << 40;
      total += (units + per - 1) / per;
    }
    return total;
  };
  double lo = 0, hi = 0;
  for (int j = 0; j < T.njobs; ++j) hi = hi > unit_cost[j] * (double)(units + 1) ? hi : unit_cost[j] * (double)(units + 1);     // one CTA per job
  for (int it = 0; it < 48; ++it) {
    const double mid = 0.5 * (lo + hi);
    if (need(mid) <= ctas) hi = mid; else lo = mid;
  }
  T.cta0[0] = 0;
  for (int j = 0; j < T.njobs; ++j) {
    const int64_t per = (int64_t)(hi / unit_cost[j]);          // >= 1: a job never gets more CTAs than units, every CTA writes its block
    T.cta0[j + 1] = T.cta0[j] + (int)((units + per - 1) / per);
  }
}
static int launch_wgrad(WgTable& WT, const TcWs& ws, int sms, cudaStream_t st) {
  wg_assign(WT, sms < WG_MAX_CTAS - 8 ? sms : WG_MAX_CTAS - 8, ws.tiles);
  if (WT.cta0[WT.njobs] > WG_MAX_CTAS) return CACTO_E_SIZE;
  cudaError_t e = cudaFuncSetAttribute(k_tc_wgrad, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(WgSmem));
  if (e != cudaSuccess) return (int)e;
  if (cudaError_t le_ = launch_tc(k_tc_wgrad, dim3(WT.cta0[WT.njobs]), THREADS, sizeof(WgSmem), st, WT, ws)) return (int)le_;
  CACTO_LAUNCH_CHECK();
  int maxel = 0;
  for (int j = 0; j < WT.njobs; ++j) maxel = maxel > WT.j[j].M * (WT.j[j].N / 4) ? maxel : WT.j[j].M * (WT.j[j].N / 4);
  if (cudaError_t le_ = launch_tc(k_tc_wgrad_reduce, dim3((maxel + WGR_OUT - 1) / WGR_OUT, WT.njobs), 256, 0, st, WT, ws)) return (int)le_;
  CACTO_LAUNCH_CHECK();
  return 0;
}
// the deterministic variants have one partials slice per CTA: at most CACTO_DET_MAX_SLICES of them
template <bool DET>
static int det_grid(int grid) { return DET && grid > CACTO_DET_MAX_SLICES ? CACTO_DET_MAX_SLICES : grid; }
static WgOperand wg_op(const float* p, int W, int c0, int amax) { WgOperand o = {p, W, c0, amax}; return o; }

template <int SYS>
static int launch_actor_env(const cacto_sys_params& P, const float* state, const double* term, const TcWs& ws, int64_t B, cudaStream_t st) {
  if (cudaError_t le_ = launch_tc(k_tc_actor_env<SYS>, dim3((unsigned)((B + 127) / 128)), 128, 0, st, P, state, term, ws, B)) return (int)le_;
  return 0;
}

}  // namespace cacto

using namespace cacto;

#ifdef TCU_TRACE
extern "C" int cacto_debug_tcu_trace(long long* buf) { return (int)cudaMemcpyToSymbol(cacto::tcu::g_tcu_trace, &buf, sizeof(buf)); }
extern "C" int cacto_debug_tcu_trace_n(void) { return cacto::tcu::TCU_TRACE_N; }
#endif

extern "C" int64_t cacto_update_tc_workspace_bytes(int64_t B, int32_t ns, int32_t na) {
  if (B <= 0 || ns < 2 || ns > CACTO_MAX_NS || na < 1 || na > CACTO_MAX_NA) return 0;
  return tc_ws_layout(nullptr, B, ns, na, nullptr);
}

template <bool DET>
static int critic_grad_tc(const cacto_sys_params* p, const float* critic_params, const float* target_params, float w_S, int mc,
                                    const float* state, const float* state_next, const float* partial_rtg, const float* dVdx, const float* done,
                                    const float* weights, float inv_B, float* grad, float* rtg, float* V, float* V_target_s, float* loss, int64_t B,
                                    void* workspace, int64_t workspace_bytes, float* part, int64_t part_floats, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (B < 0) return CACTO_E_SIZE;
  if (B == 0) return 0;
  if (!critic_params || !target_params || !state || !partial_rtg || !weights || !grad || !rtg || !V || !V_target_s || !workspace) return CACTO_E_ARG;
  if (!mc && (!state_next || !done)) return CACTO_E_ARG;
  if (w_S != 0.f && !dVdx) return CACTO_E_ARG;
  if ((reinterpret_cast<uintptr_t>(workspace) & 255) || (reinterpret_cast<uintptr_t>(grad) & 15) || (reinterpret_cast<uintptr_t>(critic_params) & 15))
    return CACTO_E_ALIGN;
  if (DET) {
    if (!part) return CACTO_E_ARG;
    if (reinterpret_cast<uintptr_t>(part) & 15) return CACTO_E_ALIGN;
    const int64_t need = cacto_det_partials_floats(CACTO_DET_CRITIC_TC, B, p->ns, p->na, 0, 0);
    if (need < 0 || part_floats < need) return CACTO_E_SIZE;
  }
  TcWs ws;
  if (tc_ws_layout(static_cast<unsigned char*>(workspace), B, p->ns, p->na, &ws) > workspace_bytes) return CACTO_E_SIZE;
  cudaStream_t st = (cudaStream_t)stream;
  const bool sobolev = w_S != 0.f;
  const int ntiles = (int)ws.tiles, sms = num_sms();

  PrepTable PT;
  memset(&PT, 0, sizeof(PT));
  prep_critic(PT, target_params, p->ns, true, ws.S_tf, ws.US + 8 * ST_TF);
  prep_critic(PT, critic_params, p->ns, true, ws.S_cf, ws.US + 8 * ST_CF);
  prep_critic(PT, critic_params, p->ns, false, ws.S_cb, ws.US + 8 * ST_CB);
  PT.zero = ws.amax; PT.nzero = AM_COUNT;
  prep_finish(PT);
  if (cudaError_t le_ = launch_tc(k_tc_prepare, dim3(PT.cta0[PT.n]), 512, 0, st, PT)) return (int)le_;
  CACTO_LAUNCH_CHECK();

  if (int e = tc_smem_attr(k_tc_critic_fwd, sizeof(CriticSmemTc))) return e;
  FwdArgs FA;
  memset(&FA, 0, sizeof(FA));
  FA.nkinds = 0;
  if (!mc) FA.kind[FA.nkinds++] = FWD_TGT_NEXT;
  FA.kind[FA.nkinds++] = FWD_TGT_S;
  FA.kind[FA.nkinds++] = FWD_F;
  FA.critic = critic_params; FA.target = target_params; FA.state = state; FA.state_next = state_next; FA.V_out = V; FA.Vt_out = V_target_s; FA.B = B;
  const int fjobs = FA.nkinds * ntiles;
  if (cudaError_t le_ = launch_tc(k_tc_critic_fwd, dim3(fjobs < sms ? fjobs : sms), THREADS, sizeof(CriticSmemTc), st, *p, FA, ws, seq_critic_fwd(), fjobs)) return (int)le_;
  CACTO_LAUNCH_CHECK();

  BwdArgs BA;
  memset(&BA, 0, sizeof(BA));
  BA.critic = critic_params; BA.w_S = w_S; BA.sobolev = sobolev ? 1 : 0; BA.mc = mc; BA.prtg = partial_rtg; BA.dVdx = dVdx; BA.done = done; BA.weights = weights;
  BA.V = V; BA.inv_B = inv_B; BA.rtg_out = rtg; BA.loss_out = loss; BA.grad = grad; BA.B = B;
  const int grid = det_grid<DET>(ntiles < sms ? ntiles : sms);
  const size_t smem = sizeof(CriticSmemTc) + (DET ? TC_DET_SMEM : 0);
  // DET: one partials region of `grid` slices per colsum kernel, in launch order (G, adjoint, B)
  const int regions = sobolev ? 3 : 1;
  auto region = [&](int r) { return DET ? part + (int64_t)r * grid * TC_DET_SLICE : grad; };
  if (sobolev) {
    BA.grad = region(0);
    if (int e = tc_smem_attr(k_tc_critic_bwd<BWD_G, DET>, smem)) return e;
    if (cudaError_t le_ = launch_tc(k_tc_critic_bwd<BWD_G, DET>, dim3(grid), THREADS, smem, st, *p, BA, ws, seq_critic_bwd(4), ntiles)) return (int)le_;
    CACTO_LAUNCH_CHECK();
    if (int e = tc_smem_attr(k_tc_critic_adj<DET>, smem)) return e;
    if (cudaError_t le_ = launch_tc(k_tc_critic_adj<DET>, dim3(grid), THREADS, smem, st, *p, critic_params, region(1), ws, seq_critic_fwd(), ntiles, B)) return (int)le_;
    CACTO_LAUNCH_CHECK();
  }
  BA.grad = region(regions - 1);
  if (int e = tc_smem_attr(k_tc_critic_bwd<BWD_B, DET>, smem)) return e;
  if (cudaError_t le_ = launch_tc(k_tc_critic_bwd<BWD_B, DET>, dim3(grid), THREADS, smem, st, *p, BA, ws, seq_critic_bwd(3), ntiles)) return (int)le_;
  CACTO_LAUNCH_CHECK();

  const CriticLayout CL(p->ns);
  WgTable WT;
  memset(&WT, 0, sizeof(WT));
  WT.njobs = 5;
  {
    WgJob& J = WT.j[4];                       // d w5 (value part) = h_4^T vbar: 128 feature rows, one real output column
    J.nterms = 1; J.X[0] = wg_op(ws.SN, CWT, kofs(3), -1); J.E[0] = wg_op(ws.VB4, 4, 0, AM_VB);
    J.M = CR_H4; J.N = 16; J.N_real = 1; J.ld = 1; J.ldn = 1; J.out = grad + CL.W[4];
  }
  for (int l = 0; l < 4; ++l) {
    WgJob& J = WT.j[l];
    J.nterms = sobolev ? 2 : 1;
    J.X[0] = l == 0 ? wg_op(ws.XN, 16, 0, AM_XN) : wg_op(ws.SN, CWT, kofs(l - 1), -1);
    J.E[0] = wg_op(ws.EE, CWT, kofs(l), AM_EE);
    J.X[1] = l == 0 ? wg_op(ws.A0, 16, 0, AM_A0) : wg_op(ws.AA, 256, kofs(l - 1), AM_AA);
    J.E[1] = wg_op(ws.DL, CWT, kofs(l), AM_DL);
    J.M = CL.in[l]; J.N = CL.out[l]; J.N_real = CL.out[l]; J.ld = CL.out[l]; J.ldn = 1; J.out = grad + CL.W[l];
  }
  if (int e = launch_wgrad(WT, ws, sms, st)) return e;
  if (DET) {
    if (cudaError_t le_ = launch_tc(k_tc_det_reduce, dim3((TC_DET_SLICE + 255) / 256), 256, 0, st, (const float*)part, regions, grid, 1, (int)p->ns,
                                    (int)p->na, grad, loss)) return (int)le_;
    CACTO_LAUNCH_CHECK();
  }
  return 0;
}


template <bool DET>
static int actor_grad_tc(const cacto_sys_params* p, const float* actor_params, const float* critic_params, const float* state,
                                   const double* term, float inv_B, float* grad, float* actions, int64_t B, void* workspace, int64_t workspace_bytes,
                                   float* part, int64_t part_floats, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (B < 0) return CACTO_E_SIZE;
  if (B == 0) return 0;
  if (!actor_params || !critic_params || !state || !term || !grad || !workspace) return CACTO_E_ARG;
  if ((reinterpret_cast<uintptr_t>(workspace) & 255) || (reinterpret_cast<uintptr_t>(grad) & 15)) return CACTO_E_ALIGN;
  if (DET) {
    if (!part) return CACTO_E_ARG;
    if (reinterpret_cast<uintptr_t>(part) & 15) return CACTO_E_ALIGN;
    const int64_t need = cacto_det_partials_floats(CACTO_DET_ACTOR_TC, B, p->ns, p->na, 0, 0);
    if (need < 0 || part_floats < need) return CACTO_E_SIZE;
  }
  TcWs ws;
  if (tc_ws_layout(static_cast<unsigned char*>(workspace), B, p->ns, p->na, &ws) > workspace_bytes) return CACTO_E_SIZE;
  cudaStream_t st = (cudaStream_t)stream;
  const int ntiles = (int)ws.tiles, sms = num_sms(), grid = det_grid<DET>(ntiles < sms ? ntiles : sms);
  const size_t smem_c = sizeof(CriticSmemTc) + (DET ? TC_DET_SMEM : 0), smem_a = sizeof(ActorSmemTc) + (DET ? TC_DET_SMEM : 0);
  // DET: one partials region of `grid` slices per colsum kernel, in launch order (GP, actor backward)
  auto region = [&](int r) { return DET ? part + (int64_t)r * grid * TC_DET_SLICE : grad; };

  PrepTable PT;
  memset(&PT, 0, sizeof(PT));
  prep_critic(PT, critic_params, p->ns, true, ws.S_cf, ws.US + 8 * ST_CF);
  prep_critic(PT, critic_params, p->ns, false, ws.S_cb, ws.US + 8 * ST_CB);
  prep_actor(PT, actor_params, p->ns, p->na, true, ws.S_af, ws.US + 8 * ST_AF);
  prep_actor(PT, actor_params, p->ns, p->na, false, ws.S_ab, ws.US + 8 * ST_AB);
  PT.zero = ws.amax; PT.nzero = AM_COUNT;
  prep_finish(PT);
  if (cudaError_t le_ = launch_tc(k_tc_prepare, dim3(PT.cta0[PT.n]), 512, 0, st, PT)) return (int)le_;
  CACTO_LAUNCH_CHECK();

  if (int e = tc_smem_attr(k_tc_actor_fwd, sizeof(ActorSmemTc))) return e;
  if (cudaError_t le_ = launch_tc(k_tc_actor_fwd, dim3(grid), THREADS, sizeof(ActorSmemTc), st, *p, actor_params, state, actions, ws, seq_actor_fwd(), ntiles, B)) return (int)le_;
  CACTO_LAUNCH_CHECK();
  switch (p->system) {
    case CACTO_SINGLE_INTEGRATOR: if (int e = launch_actor_env<CACTO_SINGLE_INTEGRATOR>(*p, state, term, ws, B, st)) return e; break;
    case CACTO_DOUBLE_INTEGRATOR: if (int e = launch_actor_env<CACTO_DOUBLE_INTEGRATOR>(*p, state, term, ws, B, st)) return e; break;
    case CACTO_CAR: if (int e = launch_actor_env<CACTO_CAR>(*p, state, term, ws, B, st)) return e; break;
    case CACTO_CAR_PARK: if (int e = launch_actor_env<CACTO_CAR_PARK>(*p, state, term, ws, B, st)) return e; break;
    case CACTO_MANIPULATOR: if (int e = launch_actor_env<CACTO_MANIPULATOR>(*p, state, term, ws, B, st)) return e; break;
    case CACTO_UR5: if (int e = launch_actor_env<CACTO_UR5>(*p, state, term, ws, B, st)) return e; break;
    default: return CACTO_E_SYSTEM;
  }
  CACTO_LAUNCH_CHECK();

  if (int e = tc_smem_attr(k_tc_critic_fwd, sizeof(CriticSmemTc))) return e;
  FwdArgs FA;
  memset(&FA, 0, sizeof(FA));
  FA.nkinds = 1; FA.kind[0] = FWD_FP; FA.critic = critic_params; FA.target = critic_params; FA.state = state; FA.B = B;
  if (cudaError_t le_ = launch_tc(k_tc_critic_fwd, dim3(grid), THREADS, sizeof(CriticSmemTc), st, *p, FA, ws, seq_critic_fwd(), ntiles)) return (int)le_;
  CACTO_LAUNCH_CHECK();

  BwdArgs BA;
  memset(&BA, 0, sizeof(BA));
  BA.critic = critic_params; BA.inv_B = inv_B; BA.grad = region(0); BA.B = B;
  if (int e = tc_smem_attr(k_tc_critic_bwd<BWD_GP, DET>, smem_c)) return e;
  if (cudaError_t le_ = launch_tc(k_tc_critic_bwd<BWD_GP, DET>, dim3(grid), THREADS, smem_c, st, *p, BA, ws, seq_critic_bwd(4), ntiles)) return (int)le_;
  CACTO_LAUNCH_CHECK();

  if (int e = tc_smem_attr(k_tc_actor_bwd<DET>, smem_a)) return e;
  if (cudaError_t le_ = launch_tc(k_tc_actor_bwd<DET>, dim3(grid), THREADS, smem_a, st, *p, region(1), ws, seq_actor_bwd(), ntiles, B)) return (int)le_;
  CACTO_LAUNCH_CHECK();

  const ActorLayout AL(p->ns, p->na);
  WgTable WT;
  memset(&WT, 0, sizeof(WT));
  WT.njobs = 4;
  {
    WgJob& J = WT.j[0];                       // dW1 = xn^T e1
    J.nterms = 1; J.X[0] = wg_op(ws.XNA, 16, 0, AM_XNA); J.E[0] = wg_op(ws.E1, ACTOR_H, 0, AM_E1);
    J.M = p->ns; J.N = ACTOR_H; J.N_real = ACTOR_H; J.ld = ACTOR_H; J.ldn = 1; J.out = grad + AL.W1;
  }
  for (int h = 0; h < 2; ++h) {
    WgJob& J = WT.j[1 + h];                   // dW2 = h1^T e2, two blocks of 128 input features
    J.nterms = 1; J.X[0] = wg_op(ws.H1, ACTOR_H, 128 * h, AM_H1); J.E[0] = wg_op(ws.E2, ACTOR_H, 0, AM_E2);
    J.M = 128; J.N = ACTOR_H; J.N_real = ACTOR_H; J.ld = ACTOR_H; J.ldn = 1; J.out = grad + AL.W2 + (int64_t)128 * h * ACTOR_H;
  }
  {
    WgJob& J = WT.j[3];                       // dW3 = h2^T d3 as its transpose d3^T h2 (na feature rows, 256 outputs): out[j + k na]
    J.nterms = 1; J.X[0] = wg_op(ws.D3, 16, 0, AM_D3); J.E[0] = wg_op(ws.H2, ACTOR_H, 0, AM_H2);
    J.M = p->na; J.N = ACTOR_H; J.N_real = ACTOR_H; J.ld = 1; J.ldn = p->na; J.out = grad + AL.W3;
  }
  if (int e = launch_wgrad(WT, ws, sms, st)) return e;
  if (DET) {
    if (cudaError_t le_ = launch_tc(k_tc_det_reduce, dim3((TC_DET_SLICE + 255) / 256), 256, 0, st, (const float*)part, 2, grid, 0, (int)p->ns,
                                    (int)p->na, grad, (float*)nullptr)) return (int)le_;
    CACTO_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" int cacto_critic_grad_tc(const cacto_sys_params* p, const float* critic_params, const float* target_params, float w_S, int mc,
                                    const float* state, const float* state_next, const float* partial_rtg, const float* dVdx, const float* done,
                                    const float* weights, float inv_B, float* grad, float* rtg, float* V, float* V_target_s, float* loss, int64_t B,
                                    void* workspace, int64_t workspace_bytes, void* stream) {
  return critic_grad_tc<false>(p, critic_params, target_params, w_S, mc, state, state_next, partial_rtg, dVdx, done, weights, inv_B, grad, rtg, V,
                               V_target_s, loss, B, workspace, workspace_bytes, nullptr, 0, stream);
}

extern "C" int cacto_critic_grad_tc_det(const cacto_sys_params* p, const float* critic_params, const float* target_params, float w_S, int mc,
                                        const float* state, const float* state_next, const float* partial_rtg, const float* dVdx, const float* done,
                                        const float* weights, float inv_B, float* grad, float* rtg, float* V, float* V_target_s, float* loss, int64_t B,
                                        void* workspace, int64_t workspace_bytes, float* partials, int64_t partials_floats, void* stream) {
  return critic_grad_tc<true>(p, critic_params, target_params, w_S, mc, state, state_next, partial_rtg, dVdx, done, weights, inv_B, grad, rtg, V,
                              V_target_s, loss, B, workspace, workspace_bytes, partials, partials_floats, stream);
}

extern "C" int cacto_actor_grad_tc(const cacto_sys_params* p, const float* actor_params, const float* critic_params, const float* state,
                                   const double* term, float inv_B, float* grad, float* actions, int64_t B, void* workspace, int64_t workspace_bytes,
                                   void* stream) {
  return actor_grad_tc<false>(p, actor_params, critic_params, state, term, inv_B, grad, actions, B, workspace, workspace_bytes, nullptr, 0, stream);
}

extern "C" int cacto_actor_grad_tc_det(const cacto_sys_params* p, const float* actor_params, const float* critic_params, const float* state,
                                       const double* term, float inv_B, float* grad, float* actions, int64_t B, void* workspace, int64_t workspace_bytes,
                                       float* partials, int64_t partials_floats, void* stream) {
  return actor_grad_tc<true>(p, actor_params, critic_params, state, term, inv_B, grad, actions, B, workspace, workspace_bytes, partials, partials_floats,
                             stream);
}

