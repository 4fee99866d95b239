// mlp.cuh -- CTA-level building blocks of the actor / critic kernels (K1 rollout, K3 update).
//
// Data layout: a CTA owns a tile of S samples (rollouts or minibatch rows).  Activations of the tile
// live in shared memory, row-major [S][ld] with ld % 4 == 0; weights are streamed from global memory
// (they total < 400 KB for both networks and stay L2-resident) straight into registers as float4 --
// consecutive threads read consecutive 16-byte column groups of a weight row, so every weight load
// is fully coalesced and every activation load is a shared-memory broadcast.
//
//   tile_gemm      C[S x N]  = A[S x K] * W[K x N]        register tile TM x 4 per thread, fp32 FMA
//   tile_gemm_small C[S x N] = A[S x K] * W                N <= 16 (network heads), K split over lanes
//   tile_outer2    dW[K x N] += A1^T E1 (+ A2^T E2)        weight gradients, fp32 atomics to global
//   tile_colsum    db[N]    += sum_s E[s][n]
//
// fp32 CUDA-core FMA is used on purpose: the parity gate of this path is 1e-5 (rollout states) /
// 1e-4 (updated weights) against an fp32 reference, which bf16/tf32 tensor-core products do not
// meet (SURVEY.md section 7 "Tensor cores vs. parity").
#pragma once
#include <cuda_runtime.h>
#include "mlp_layout.cuh"

namespace cacto {

template <int S, int N, int NT>
struct GemmMap {
  static_assert(N % 4 == 0, "N must be a multiple of 4");
  static constexpr int CG = N / 4;                              // float4 column groups
  static_assert(CG <= NT && NT % CG == 0, "column groups must tile the CTA");
  static constexpr int RG = (NT / CG) < S ? (NT / CG) : S;      // row groups in use
  static_assert(S % RG == 0, "rows must split evenly");
  static constexpr int TM = S / RG;                             // rows per thread
};

__device__ __forceinline__ void fma4(float4& acc, float a, const float4& w) {
  acc.x = fmaf(a, w.x, acc.x);
  acc.y = fmaf(a, w.y, acc.y);
  acc.z = fmaf(a, w.z, acc.z);
  acc.w = fmaf(a, w.w, acc.w);
}

// C = A * W.  A: shared [S][lda]; W: global or shared, row k at W + k*ldw (ldw % 4 == 0, 16-byte aligned).
// epi(row, col, acc4) is called once per (row, 4-column group) owned by the thread.
// The caller synchronises (A must be complete before the call; the epilogue may overwrite A only
// after a __syncthreads() placed by the caller -- see the `sync_before_epilogue` flag).
template <int S, int N, int NT, bool SYNC_BEFORE_EPI, typename Epi>
__device__ __forceinline__ void tile_gemm(const float* __restrict__ A, int lda, int K, const float* __restrict__ W, int ldw,
                                          Epi&& epi) {
  typedef GemmMap<S, N, NT> M;
  constexpr int TM = M::TM;
  const int cg = threadIdx.x % M::CG, rg = threadIdx.x / M::CG;
  const bool active = rg < M::RG;
  float4 acc[TM];
#pragma unroll
  for (int r = 0; r < TM; ++r) acc[r] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (active) {
    const float* a0 = A + (size_t)(rg * TM) * lda;
    const float4* wp = reinterpret_cast<const float4*>(W) + cg;
    const int ldw4 = ldw >> 2;
    const int K4 = K & ~3;
    float4 w[4], wn[4];
    if (K4 > 0) {
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) w[kk] = wp[(size_t)kk * ldw4];
    }
    for (int k = 0; k < K4; k += 4) {
      if (k + 4 < K4) {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) wn[kk] = wp[(size_t)(k + 4 + kk) * ldw4];
      }
#pragma unroll
      for (int r = 0; r < TM; ++r) {
        const float4 a = *reinterpret_cast<const float4*>(a0 + r * lda + k);
        fma4(acc[r], a.x, w[0]);
        fma4(acc[r], a.y, w[1]);
        fma4(acc[r], a.z, w[2]);
        fma4(acc[r], a.w, w[3]);
      }
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) w[kk] = wn[kk];
    }
    for (int k = K4; k < K; ++k) {
      const float4 wk = wp[(size_t)k * ldw4];
#pragma unroll
      for (int r = 0; r < TM; ++r) fma4(acc[r], a0[r * lda + k], wk);
    }
  }
  if (SYNC_BEFORE_EPI) __syncthreads();
  if (active) {
#pragma unroll
    for (int r = 0; r < TM; ++r) epi(rg * TM + r, 4 * cg, acc[r]);
  }
}

// ------------------------------------------------------------------------------------------ weight pipeline
// Weights streamed into shared memory by the TMA engine: one elected thread issues a 1-D bulk copy
// (cp.async.bulk, SASS UBLKCP) of a contiguous chunk of <= W_CHUNK floats from global/L2 into one of two
// shared slots and an mbarrier counts the landed bytes; all threads then read the chunk with conflict-free
// LDS.128.  While a chunk is consumed the next one (of the same GEMM or the first chunk of the next GEMM)
// is already in flight, so the L2 latency of a weight fetch is paid once per kernel, not once per k-step
// (the latter made the B = 64 update latency-bound: profiles/README.md, "K3 at the reference's batch size").
constexpr int W_CHUNK = 8192;   // floats per slot (32 KB)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

struct WeightPipe {
  float* buf;          // 2 * W_CHUNK floats, 128-byte aligned
  uint64_t* bar;       // 2 mbarriers
  unsigned issued, consumed;

  __device__ __forceinline__ void init(float* b, uint64_t* br) {
    buf = b; bar = br; issued = 0; consumed = 0;
    if (threadIdx.x == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar[0])));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar[1])));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
  }
  // All threads call; thread 0 issues.  The target slot must no longer be read by any thread
  // (callers guarantee it with the __syncthreads() that ends the consumption of a chunk).
  __device__ __forceinline__ void issue(const float* __restrict__ g, int nfloats) {
    if (threadIdx.x == 0 && g != nullptr) {
      const unsigned slot = issued & 1u;
      const uint32_t bytes = (uint32_t)nfloats * 4u;
      const uint32_t mb = smem_u32(&bar[slot]);
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mb), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                       smem_u32(buf + slot * W_CHUNK)),
                   "l"(g), "r"(bytes), "r"(mb)
                   : "memory");
    }
    if (g != nullptr) ++issued;
  }
  __device__ __forceinline__ const float* wait() {
    const unsigned slot = consumed & 1u, parity = (consumed >> 1) & 1u;
    const uint32_t mb = smem_u32(&bar[slot]);
    uint32_t done = 0;
    unsigned spins = 0;
    while (!done) {
      if (++spins > (1u << 24)) __trap();      // a chunk that was never issued: fail loudly instead of hanging the GPU
      asm volatile(
          "{\n\t.reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t}"
          : "=r"(done)
          : "r"(mb), "r"(parity)
          : "memory");
    }
    ++consumed;
    return buf + slot * W_CHUNK;
  }
};

template <int N>
__host__ __device__ constexpr int chunk_rows(int K) { return (W_CHUNK / N) < K ? (W_CHUNK / N) : K; }

// Thread mapping of the streamed GEMMs for SMALL tiles (S <= 4, the reference's batch sizes): with one thread per (row group,
// column group) a 2-row tile keeps 1 (N = 64) to 4 (N = 256) of the 8 warps busy on a dependent chain of K / 4 steps while the
// rest wait at the barrier (ncu at B = 64: barrier = 36 % of the stall samples).  Here the reduction is split over the four
// quarter-warps (lane = 8 kg + c8: k-group kg takes k = 16 j + 4 kg .. + 3 of every block of 16; the 8 lanes of a quarter own 8
// adjacent float4 column groups: conflict-free 128-byte W reads, one broadcast float4 of A), rows over warps; the four partial
// sums meet in a two-step shuffle butterfly and lane group kg runs the epilogue of row kg.  K % 16 == 0.  (For 8- and 16-row
// tiles this mapping measured slower -- profiles/README.md -- the A broadcasts become the shared-memory bottleneck.)
template <int S, int N, int NT>
struct SplitKMap {
  static_assert(N % 32 == 0, "N must be a multiple of 32");
  static constexpr int CG = N / 4;              // float4 column groups
  static constexpr int WARPS = NT / 32;
  static constexpr int WC = CG / 8;             // warps across the columns
  static_assert(WC <= WARPS && WARPS % WC == 0, "column warps must tile the CTA");
  static constexpr int RG = (WARPS / WC) < S ? (WARPS / WC) : S;   // row groups in use (further warps idle)
  static_assert(S % RG == 0, "rows must split evenly");
  static constexpr int TM = S / RG;             // rows per thread
  static_assert(TM <= 4, "the epilogue hands row r to lane group r");
};

template <int S, int N, int NT, typename Epi>
__device__ __forceinline__ void gemm_streamed_splitk(WeightPipe& pipe, const float* __restrict__ A, int lda, int K,
                                                     const float* __restrict__ Wg, const float* __restrict__ next, int next_floats,
                                                     Epi&& epi) {
  typedef SplitKMap<S, N, NT> M;
  constexpr int TM = M::TM;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int kg = lane >> 3, cg = (warp % M::WC) * 8 + (lane & 7), rg = warp / M::WC;
  const bool active = rg < M::RG;
  float4 acc[TM];
#pragma unroll
  for (int r = 0; r < TM; ++r) acc[r] = make_float4(0.f, 0.f, 0.f, 0.f);
  const int rows_per_chunk = chunk_rows<N>(K);           // a multiple of 16 (8192 / N, or K)
  const int nchunks = (K + rows_per_chunk - 1) / rows_per_chunk;
  for (int c = 0; c < nchunks; ++c) {
    const int k0 = c * rows_per_chunk;
    const int kc = min(rows_per_chunk, K - k0);
    if (c + 1 < nchunks) {
      const int kn = min(rows_per_chunk, K - (k0 + rows_per_chunk));
      pipe.issue(Wg + (size_t)(k0 + rows_per_chunk) * N, kn * N);
    } else {
      pipe.issue(next, next_floats);
    }
    const float* w = pipe.wait();
    if (active) {
      const float* a0 = A + (size_t)(rg * TM) * lda + k0 + 4 * kg;
      const float4* wp = reinterpret_cast<const float4*>(w) + (size_t)(4 * kg) * (N / 4) + cg;
#pragma unroll 2
      for (int kb = 0; kb < kc; kb += 16) {
        const float4* wr = wp + (size_t)kb * (N / 4);
        const float4 w0 = wr[0], w1 = wr[N / 4], w2 = wr[2 * (N / 4)], w3 = wr[3 * (N / 4)];
#pragma unroll
        for (int r = 0; r < TM; ++r) {
          const float4 a = *reinterpret_cast<const float4*>(a0 + r * lda + kb);
          fma4(acc[r], a.x, w0);
          fma4(acc[r], a.y, w1);
          fma4(acc[r], a.z, w2);
          fma4(acc[r], a.w, w3);
        }
      }
    }
    __syncthreads();          // every thread is done with this slot before it is refilled
  }
  if (active) {               // warp-uniform: whole warps are active or idle
#pragma unroll
    for (int r = 0; r < TM; ++r) {
      float4 v = acc[r];
      v.x += __shfl_xor_sync(0xffffffffu, v.x, 8);
      v.y += __shfl_xor_sync(0xffffffffu, v.y, 8);
      v.z += __shfl_xor_sync(0xffffffffu, v.z, 8);
      v.w += __shfl_xor_sync(0xffffffffu, v.w, 8);
      v.x += __shfl_xor_sync(0xffffffffu, v.x, 16);
      v.y += __shfl_xor_sync(0xffffffffu, v.y, 16);
      v.z += __shfl_xor_sync(0xffffffffu, v.z, 16);
      v.w += __shfl_xor_sync(0xffffffffu, v.w, 16);
      if (r == kg) epi(rg * TM + r, 4 * cg, v);
    }
  }
}

// C = A * W with W [K x N] (row-major, ld = N, K % 4 == 0) streamed through the weight pipeline.
// Contract: the first chunk of W is already in flight; while the last chunk is being consumed the first
// chunk of `next` (next_floats floats, nullptr for none) is issued.  Ends WITHOUT a trailing barrier for
// the epilogue: the caller places the __syncthreads() that publishes C (as with tile_gemm).
template <int S, int N, int NT, typename Epi>
__device__ __forceinline__ void gemm_streamed(WeightPipe& pipe, const float* __restrict__ A, int lda, int K,
                                              const float* __restrict__ Wg, const float* __restrict__ next, int next_floats, Epi&& epi) {
  if constexpr (S <= 4) {
    gemm_streamed_splitk<S, N, NT>(pipe, A, lda, K, Wg, next, next_floats, epi);
    return;
  }
  typedef GemmMap<S, N, NT> M;
  constexpr int TM = M::TM;
  const int cg = threadIdx.x % M::CG, rg = threadIdx.x / M::CG;
  const bool active = rg < M::RG;
  float4 acc[TM];
#pragma unroll
  for (int r = 0; r < TM; ++r) acc[r] = make_float4(0.f, 0.f, 0.f, 0.f);
  const int rows_per_chunk = chunk_rows<N>(K);
  const int nchunks = (K + rows_per_chunk - 1) / rows_per_chunk;
  for (int c = 0; c < nchunks; ++c) {
    const int k0 = c * rows_per_chunk;
    const int kc = min(rows_per_chunk, K - k0);
    if (c + 1 < nchunks) {
      const int kn = min(rows_per_chunk, K - (k0 + rows_per_chunk));
      pipe.issue(Wg + (size_t)(k0 + rows_per_chunk) * N, kn * N);
    } else {
      pipe.issue(next, next_floats);
    }
    const float* w = pipe.wait();
    if (active) {
      const float* a0 = A + (size_t)(rg * TM) * lda + k0;
      const float4* wp = reinterpret_cast<const float4*>(w) + cg;
#pragma unroll 2
      for (int k = 0; k < kc; k += 4) {
        const float4 w0 = wp[(k + 0) * (N / 4)], w1 = wp[(k + 1) * (N / 4)], w2 = wp[(k + 2) * (N / 4)], w3 = wp[(k + 3) * (N / 4)];
#pragma unroll
        for (int r = 0; r < TM; ++r) {
          const float4 a = *reinterpret_cast<const float4*>(a0 + r * lda + k);
          fma4(acc[r], a.x, w0);
          fma4(acc[r], a.y, w1);
          fma4(acc[r], a.z, w2);
          fma4(acc[r], a.w, w3);
        }
      }
    }
    __syncthreads();          // every thread is done with this slot before it is refilled
  }
  if (active) {
#pragma unroll
    for (int r = 0; r < TM; ++r) epi(rg * TM + r, 4 * cg, acc[r]);
  }
}

// C[s][j] = sum_k A[s][k] * w(k, j) for tiny N.  W_KN: w(k, j) = W[k*N + j]; otherwise w(k, j) = W[j*ldw + k]
// (rows of a [N x K] matrix).  G lanes cooperate on one output.  epi(row, j, value).
template <int S, int NT, int G, bool W_KN, typename Epi>
__device__ __forceinline__ void tile_gemm_small(const float* __restrict__ A, int lda, int K, const float* __restrict__ W, int N,
                                                int ldw, Epi&& epi) {
  static_assert(G <= 32 && (G & (G - 1)) == 0, "G must be a power of two <= 32");
  const int sub = threadIdx.x % G, grp = threadIdx.x / G;
  constexpr int GROUPS = NT / G;
  const int total = S * N;
  for (int base = 0; base < total; base += GROUPS) {
    const int o = base + grp;
    const bool valid = o < total;
    const int s = valid ? o / N : 0, j = valid ? o - (o / N) * N : 0;
    float acc = 0.f;
    if (valid) {
      for (int k = sub; k < K; k += G) {
        const float w = W_KN ? W[(size_t)k * N + j] : W[(size_t)j * ldw + k];
        acc = fmaf(A[s * lda + k], w, acc);
      }
    }
#pragma unroll
    for (int off = G / 2; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (valid && sub == 0) epi(s, j, acc);
  }
}

// Adding a CTA's contribution into a gradient block.  DET = false: fp32 atomics into the shared accumulator (the order in which the
// CTAs land decides the low bits).  DET = true: the block is the CTA's own partials slice (csrc/det.cuh), which no other CTA
// touches, and each element is written by one thread of the CTA -- a plain read-modify-write in program order.
template <bool DET>
__device__ __forceinline__ void grad_add(float* p, float v) {
  if constexpr (DET) *p += v;
  else atomicAdd(p, v);
}
template <bool DET>
__device__ __forceinline__ void grad_add4(float* p, const float4& v) {
  if constexpr (DET) {
    float4 g = *reinterpret_cast<float4*>(p);
    g.x += v.x; g.y += v.y; g.z += v.z; g.w += v.w;
    *reinterpret_cast<float4*>(p) = g;
  } else {
    // one 16-byte vector reduction (red.global.add.v4.f32, sm_90+) instead of four scalar ones
    atomicAdd(reinterpret_cast<float4*>(p), v);
  }
}

// dW[k][n] += scale-free sum_s A1[s][k] E1[s][n] (+ A2[s][k] E2[s][n]); K x N outputs, atomics to global (grad_add).
// A*: shared [S][lda*] (k contiguous), E*: shared [S][lde*].  Rows k >= K are skipped.  KT = 4.  dW must be 16-byte aligned.
template <int S, int N, int NT, bool DET = false>
__device__ __forceinline__ void tile_outer2(const float* __restrict__ A1, int lda1, const float* __restrict__ E1, int lde1,
                                            const float* __restrict__ A2, int lda2, const float* __restrict__ E2, int lde2, int K,
                                            float* __restrict__ dW, int rows_valid) {
  static_assert(N % 4 == 0, "N % 4");
  constexpr int CG = N / 4;
  const int ktiles = (K + 3) >> 2;
  for (int t = threadIdx.x; t < ktiles * CG; t += NT) {
    const int cg = t % CG, k0 = (t / CG) << 2;
    float4 acc[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < rows_valid; ++s) {
      const float4 a = *reinterpret_cast<const float4*>(A1 + s * lda1 + k0);
      const float4 e = *reinterpret_cast<const float4*>(E1 + s * lde1 + 4 * cg);
      fma4(acc[0], a.x, e);
      fma4(acc[1], a.y, e);
      fma4(acc[2], a.z, e);
      fma4(acc[3], a.w, e);
    }
    if (A2 != nullptr) {
      for (int s = 0; s < rows_valid; ++s) {
        const float4 a = *reinterpret_cast<const float4*>(A2 + s * lda2 + k0);
        const float4 e = *reinterpret_cast<const float4*>(E2 + s * lde2 + 4 * cg);
        fma4(acc[0], a.x, e);
        fma4(acc[1], a.y, e);
        fma4(acc[2], a.z, e);
        fma4(acc[3], a.w, e);
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      // 16-byte accesses: the weight matrices start at multiples of 4 floats inside the 16-byte-aligned gradient block, N % 4 == 0
      if (k0 + i < K) grad_add4<DET>(dW + (size_t)(k0 + i) * N + 4 * cg, acc[i]);
    }
  }
}

// db[n] += sum_s E[s][n]
template <int NT, bool DET = false>
__device__ __forceinline__ void tile_colsum(const float* __restrict__ E, int lde, int N, int rows_valid, float* __restrict__ db) {
  for (int n = threadIdx.x; n < N; n += NT) {
    float acc = 0.f;
    for (int s = 0; s < rows_valid; ++s) acc += E[s * lde + n];
    grad_add<DET>(db + n, acc);
  }
}

// utils.py:17-24 -- x / norm for the state part, 2 t / T - 1 for the time (last) component.
__device__ __forceinline__ float normalize_component(const cacto_sys_params& P, int j, float x) {
  if (!P.normalize) return x;
  const float n = (float)P.state_norm[j];
  return (j == P.ns - 1) ? (x / n) * 2.f - 1.f : x / n;
}
// d normalised_j / d raw_j
__device__ __forceinline__ float normalize_scale(const cacto_sys_params& P, int j) {
  if (!P.normalize) return 1.f;
  const float n = (float)P.state_norm[j];
  return (j == P.ns - 1) ? 2.f / n : 1.f / n;
}

__device__ __forceinline__ float leaky(float z) { return z > 0.f ? z : LEAKY_ALPHA * z; }

}  // namespace cacto
