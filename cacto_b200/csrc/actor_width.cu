// actor_width.cu -- K1 (rollouts), NN.eval and K3 (actor gradient) for an actor of ANY hidden width:
//     ns -> NH1 -> NH2 -> na with LeakyReLU(0.3), 1 <= NH1, NH2 <= 512 (NeuralNetwork.py:51-63; conf.NH1 / conf.NH2).
// The fused kernels of rollout.cu / rollout_tc*.cu / update.cu are specialised for NH1 = NH2 = 256 (every reference conf); these
// take the widths at run time and read the Keras-layout parameter block as it is (no padded or transposed copy), so a policy
// update needs no preparation step and the actor gradient is one launch.
//
// Layer code shared by the three kernels (fp32 CUDA-core FMA, as the 256-wide FMA path and for the same parity reason):
//   wgemm      C[S x N] = A[S x K] W[K x N], N and the row stride of W at run time.  Warp-uniform work items of TM rows x 128
//              columns; lane l owns columns c0 + l + 32 q (q < 4), so every weight load of a warp is one coalesced 128-byte
//              segment of a weight row (any width, no alignment needed), and the activations are float4 shared-memory broadcasts.
//   wgemm_nt   C[S x M] = E[S x K] W^T for W [M x K] row-major (the actor backward without a transposed copy): one warp per
//              output unit, lanes stride the weight row (coalesced), per-sample partial sums meet in a shuffle butterfly.
//   wouter     dW[K x N] += A^T E over the CTA's tile of samples: ONE fp32 atomic per weight and tile (not per sample).
#include "common.cuh"
#include "det.cuh"
#include "mlp.cuh"
#include "systems.cuh"

namespace cacto {

constexpr int AW_NT = 256;            // threads per CTA
constexpr int AW_WARPS = AW_NT / 32;
constexpr int AW_NSP = 16;            // padded input width (>= CACTO_MAX_NS, multiple of 4)
constexpr int AW_NAP = 8;             // padded action width
constexpr int AW_RO_S = 32;           // rollouts per CTA (K1, NN.eval) ...
constexpr int AW_RO_S_WIDE = 16;      // ... and for K1 when 32 rollouts' hidden tiles would exceed AW_RO_WIDE_BYTES of shared memory
constexpr size_t AW_RO_WIDE_BYTES = 100 * 1024;   // (above it only one 8-warp CTA fits per SM; two 16-rollout CTAs do)
constexpr int AW_CW = CR_H1 + CR_H2 + CR_H3 + CR_H4;      // hidden units of the 'sine' critic
constexpr int AW_FUP = CACTO_MAX_NS * CACTO_MAX_NA + 2;   // ds'/da per sample

__host__ __device__ __forceinline__ int round4(int n) { return (n + 3) & ~3; }
__host__ __device__ __forceinline__ constexpr int aw_koff(int l) { return l == 0 ? 0 : (l == 1 ? CR_H1 : (l == 2 ? CR_H1 + CR_H2 : CR_H1 + CR_H2 + CR_H3)); }

template <int S, int TM, typename Epi>
__device__ __forceinline__ void wgemm(const float* A, int lda, int K, const float* __restrict__ W, int ldw, int N, Epi&& epi) {
  static_assert(S % TM == 0, "rows must split evenly");
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int ncb = (N + 127) >> 7, items = ncb * (S / TM);
  for (int it = warp; it < items; it += AW_WARPS) {
    const int c0 = (it % ncb) * 128 + lane, r0 = (it / ncb) * TM;
    const float* a0 = A + (size_t)r0 * lda;
    const float* w0 = W + c0;
    bool v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) v[q] = c0 + 32 * q < N;
    float acc[TM][4];
#pragma unroll
    for (int r = 0; r < TM; ++r)
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[r][q] = 0.f;
    const int K4 = K & ~3;
    for (int k = 0; k < K4; k += 4) {
      float w[4][4];
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
#pragma unroll
        for (int q = 0; q < 4; ++q) w[kk][q] = v[q] ? __ldg(w0 + (size_t)(k + kk) * ldw + 32 * q) : 0.f;
#pragma unroll
      for (int r = 0; r < TM; ++r) {
        const float4 a = *reinterpret_cast<const float4*>(a0 + r * lda + k);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          acc[r][q] = fmaf(a.x, w[0][q], acc[r][q]);
          acc[r][q] = fmaf(a.y, w[1][q], acc[r][q]);
          acc[r][q] = fmaf(a.z, w[2][q], acc[r][q]);
          acc[r][q] = fmaf(a.w, w[3][q], acc[r][q]);
        }
      }
    }
    for (int k = K4; k < K; ++k) {
      float w[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) w[q] = v[q] ? __ldg(w0 + (size_t)k * ldw + 32 * q) : 0.f;
#pragma unroll
      for (int r = 0; r < TM; ++r) {
        const float a = a0[r * lda + k];
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[r][q] = fmaf(a, w[q], acc[r][q]);
      }
    }
#pragma unroll
    for (int r = 0; r < TM; ++r)
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (v[q]) epi(r0 + r, c0 + 32 * q, acc[r][q]);
  }
}

// C[s][i] = sum_k E[s][k] W[i * ldw + k] for i < M (S <= 32).  epi(row, i, value).
template <int S, typename Epi>
__device__ __forceinline__ void wgemm_nt(const float* E, int lde, int K, const float* __restrict__ W, int ldw, int M, Epi&& epi) {
  static_assert(S <= 32, "lane s writes row s");
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = warp; i < M; i += AW_WARPS) {
    float acc[S];
#pragma unroll
    for (int s = 0; s < S; ++s) acc[s] = 0.f;
    const float* wr = W + (size_t)i * ldw;
    for (int k = lane; k < K; k += 32) {
      const float w = __ldg(wr + k);
#pragma unroll
      for (int s = 0; s < S; ++s) acc[s] = fmaf(E[s * lde + k], w, acc[s]);
    }
#pragma unroll
    for (int s = 0; s < S; ++s) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc[s] += __shfl_xor_sync(0xffffffffu, acc[s], o);
      if (lane == s) epi(s, i, acc[s]);
    }
  }
}

// dW[k][n] += sum_{s < rows} A[s][k] E[s][n], k < K, n < N (dW row stride N).  A: [S][lda], lda % 4 == 0, lda >= round4(K).
template <bool DET = false>
__device__ __forceinline__ void wouter(const float* A, int lda, const float* E, int lde, int K, int N, float* __restrict__ dW, int rows) {
  const int kq = (K + 3) >> 2;
  for (int t = threadIdx.x; t < kq * N; t += AW_NT) {
    const int n = t % N, k0 = (t / N) * 4;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int s = 0; s < rows; ++s) {
      const float e = E[s * lde + n];
      const float4 a = *reinterpret_cast<const float4*>(A + s * lda + k0);
      acc[0] = fmaf(a.x, e, acc[0]);
      acc[1] = fmaf(a.y, e, acc[1]);
      acc[2] = fmaf(a.z, e, acc[2]);
      acc[3] = fmaf(a.w, e, acc[3]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (k0 + i < K) grad_add<DET>(dW + (size_t)(k0 + i) * N + n, acc[i]);
  }
}

// Actor forward for a tile: X [S][AW_NSP] (normalised input) -> H1 [S][ld1], H2 [S][ld2] (LeakyReLU outputs), ACT [S][AW_NAP].
// Starts after a barrier that published X; ends synchronised.
template <int S, int TM>
__device__ __forceinline__ void actor_tile_forward(const float* __restrict__ aw, const ActorLayout& L, const float* X, float* H1, int ld1,
                                                   float* H2, int ld2, float* ACT) {
  wgemm<S, TM>(X, AW_NSP, L.ns, aw + L.W1, L.h1, L.h1, [&](int r, int c, float v) { H1[r * ld1 + c] = leaky(v + __ldg(aw + L.b1 + c)); });
  __syncthreads();
  wgemm<S, TM>(H1, ld1, L.h1, aw + L.W2, L.h2, L.h2, [&](int r, int c, float v) { H2[r * ld2 + c] = leaky(v + __ldg(aw + L.b2 + c)); });
  __syncthreads();
  tile_gemm_small<S, AW_NT, 8, true>(H2, ld2, L.h2, aw + L.W3, L.na, 0, [&](int s, int j, float v) { ACT[s * AW_NAP + j] = v + __ldg(aw + L.b3 + j); });
  __syncthreads();
}

__host__ __device__ __forceinline__ size_t ro_smem_bytes(int S, int h1, int h2) {
  return 4u * (size_t)S * (AW_NSP + AW_NAP + round4(h1) + round4(h2));
}

// ------------------------------------------------------------------------------------------ K1
// Same contract and structure as k_rollout (rollout.cu): a CTA owns S rollouts for their whole horizon, the hidden
// activations never leave shared memory (sized at launch from the widths), the dynamics run in fp64 on one thread per rollout.
template <int SYS, int S>
__global__ void __launch_bounds__(AW_NT, 2) k_rollout_width(const __grid_constant__ cacto_sys_params P, const float* __restrict__ actor,
                                                            int h1, int h2, const double* __restrict__ ics, const int32_t* __restrict__ horizon,
                                                            int T_max, double* __restrict__ states, double* __restrict__ controls,
                                                            int32_t* __restrict__ flags, double* __restrict__ rewards, int64_t B) {
  constexpr int NX = SysDims<SYS>::NX, NA = SysDims<SYS>::NA, NS = NX + 1;
  extern __shared__ __align__(16) float aw_smem[];
  __shared__ int tmax_s;
  const int ld1 = round4(h1), ld2 = round4(h2);
  float* X = aw_smem;
  float* ACT = X + S * AW_NSP;
  float* H1 = ACT + S * AW_NAP;
  float* H2 = H1 + S * ld1;
  const ActorLayout L(NS, NA, h1, h2);
  const int tid = threadIdx.x;
  const int64_t b = (int64_t)blockIdx.x * S + tid;
  const bool owner = tid < S && b < B;

  double x[NS];
  int h = 0, ok = 1;
  if (tid == 0) tmax_s = 0;
  __syncthreads();
  if (owner) {
#pragma unroll
    for (int j = 0; j < NS; ++j) {
      x[j] = ics[b * NS + j];
      states[(int64_t)j * B + b] = x[j];
    }
    h = min(max(horizon[b], 0), T_max);
    atomicMax(&tmax_s, h);
  }
  if (tid < S) {
#pragma unroll
    for (int j = 0; j < AW_NSP; ++j) X[tid * AW_NSP + j] = 0.f;
  }
  __syncthreads();
  const int tmax = tmax_s;

  for (int t = 0; t < tmax; ++t) {
    const bool live = owner && ok && t < h;
    if (tid < S) {
#pragma unroll
      for (int j = 0; j < NS; ++j) X[tid * AW_NSP + j] = live ? normalize_component(P, j, (float)x[j]) : 0.f;
    }
    __syncthreads();
    actor_tile_forward<S, S / 4>(actor, L, X, H1, ld1, H2, ld2, ACT);
    if (live) {
      double u[NA], xn[NS];
#pragma unroll
      for (int j = 0; j < NA; ++j) {
        u[j] = (double)ACT[tid * AW_NAP + j];
        controls[((int64_t)t * NA + j) * B + b] = u[j];
      }
      if (rewards != nullptr) rewards[(int64_t)t * B + b] = sys_reward<SYS, double>(P, P.w_running, x, u, false);
      sys_step<SYS, double>(P, x, u, xn);
      xn[NX] = x[NX] + P.dt;
      bool nan = false;
#pragma unroll
      for (int j = 0; j < NS; ++j) {
        x[j] = xn[j];
        nan |= (xn[j] != xn[j]);
        states[((int64_t)(t + 1) * NS + j) * B + b] = xn[j];
      }
      if (nan) ok = 0;                          // RL.py:229-231
      if (rewards != nullptr && t + 1 == h && !nan)
        rewards[(int64_t)(t + 1) * B + b] = sys_reward<SYS, double>(P, P.w_terminal, x, (const double*)nullptr, false);
    }
  }
  if (owner) flags[b] = ok;
}

// ------------------------------------------------------------------------------------------ NN.eval
__global__ void __launch_bounds__(AW_NT, 2) k_actor_forward_width(const __grid_constant__ cacto_sys_params P, const float* __restrict__ actor,
                                                                  int h1, int h2, const float* __restrict__ state, float* __restrict__ out,
                                                                  int64_t B) {
  constexpr int S = AW_RO_S;
  extern __shared__ __align__(16) float aw_smem[];
  const int ld1 = round4(h1), ld2 = round4(h2), ns = P.ns, na = P.na;
  float* X = aw_smem;
  float* ACT = X + S * AW_NSP;
  float* H1 = ACT + S * AW_NAP;
  float* H2 = H1 + S * ld1;
  const ActorLayout L(ns, na, h1, h2);
  const int64_t row0 = (int64_t)blockIdx.x * S;
  const int rows = (int)min((int64_t)S, B - row0);
  for (int i = threadIdx.x; i < S * AW_NSP; i += AW_NT) {
    const int s = i / AW_NSP, j = i - s * AW_NSP;
    X[i] = (s < rows && j < ns) ? normalize_component(P, j, state[(row0 + s) * ns + j]) : 0.f;
  }
  __syncthreads();
  actor_tile_forward<S, S / 4>(actor, L, X, H1, ld1, H2, ld2, ACT);
  for (int i = threadIdx.x; i < rows * na; i += AW_NT) {
    const int s = i / na, j = i - s * na;
    out[(row0 + s) * na + j] = ACT[s * AW_NAP + j];
  }
}

// ------------------------------------------------------------------------------------------ K3
// The analogue of k_actor_grad<SYS, S> (update.cu) for a run-time width: actor forward, s' / ds'/da / dr/da per sample
// (sys_step_Fu, sys_dr_da), 'sine' critic forward and input gradient at s' (with the critic's transposed copy), actor backward with
// the weight gradients reduced over the tile before one atomic per weight.
__host__ __device__ __forceinline__ size_t ag_smem_bytes(int S, int h1, int h2) {
  return 4u * (size_t)S * (3 * AW_NSP + 3 * AW_NAP + AW_FUP + AW_CW + 2 * CR_H4 + round4(h1) + max(round4(h1), round4(h2)) + round4(h2));
}

// DET: grad is the partials workspace (det.cuh); the CTA adds into its slice
template <int SYS, int S, bool DET = false>
__global__ void __launch_bounds__(AW_NT) k_actor_grad_width(const __grid_constant__ cacto_sys_params P, const float* __restrict__ aw, int h1, int h2,
                                                            const float* __restrict__ cw, const float* __restrict__ cwT,
                                                            const float* __restrict__ state, const double* __restrict__ term, float inv_B,
                                                            float* __restrict__ grad, float* __restrict__ actions_out, int64_t B) {
  pdl_wait();
  constexpr int NX = SysDims<SYS>::NX, NA = SysDims<SYS>::NA, NS = NX + 1, TM = S / 4;
  extern __shared__ __align__(16) float aw_smem[];
  const int ld1 = round4(h1), ld2 = round4(h2);
  float* XN = aw_smem;                  // [S][AW_NSP] normalised state
  float* XNP = XN + S * AW_NSP;         // [S][AW_NSP] normalised next state
  float* G0 = XNP + S * AW_NSP;         // [S][AW_NSP] dV/d(normalised s')
  float* ACT = G0 + S * AW_NSP;         // [S][AW_NAP]
  float* D3 = ACT + S * AW_NAP;
  float* DRDA = D3 + S * AW_NAP;
  float* FU = DRDA + S * AW_NAP;        // [S][AW_FUP]
  float* CS = FU + S * AW_FUP;          // [S][AW_CW] cos z of the critic's hidden layers
  float* C0 = CS + S * AW_CW;           // [S][CR_H4] x 2: critic activations, then its input-gradient sweep
  float* C1 = C0 + S * CR_H4;
  float* H1 = C1 + S * CR_H4;           // [S][ld1]
  float* H2 = H1 + S * ld1;             // [S][ld2]; later dL/dz1 [S][ld1]
  float* E = H2 + S * max(ld1, ld2);              // [S][ld2] dL/dz2
  const ActorLayout LA(NS, NA, h1, h2);
  const CriticLayout LC(NS);
  if constexpr (DET) grad += (size_t)blockIdx.x * det_stride(LA.total);
  const int tid = threadIdx.x;
  const int64_t row0 = (int64_t)blockIdx.x * S;
  const int rows = (int)min((int64_t)S, B - row0);

  for (int i = tid; i < S * AW_NSP; i += AW_NT) {
    const int s = i / AW_NSP, j = i - s * AW_NSP;
    XN[i] = (s < rows && j < NS) ? normalize_component(P, j, state[(row0 + s) * NS + j]) : 0.f;
  }
  __syncthreads();
  // ---- actor forward (NeuralNetwork.py:185)
  actor_tile_forward<S, TM>(aw, LA, XN, H1, ld1, H2, ld2, ACT);

  // ---- per sample: s' = f(s, a), ds'/da (normalised), dr/da  (NeuralNetwork.py:188,199-204)
  if (tid < S) {
    float xnp[AW_NSP];
#pragma unroll
    for (int j = 0; j < AW_NSP; ++j) xnp[j] = 0.f;
    if (tid < rows) {
      const int64_t b = row0 + tid;
      double x[NS], u[NA], xn[NS], Fu[NX * NA];
#pragma unroll
      for (int j = 0; j < NS; ++j) x[j] = (double)state[b * NS + j];
#pragma unroll
      for (int j = 0; j < NA; ++j) {
        u[j] = (double)ACT[tid * AW_NAP + j];
        if (actions_out != nullptr) actions_out[b * NA + j] = ACT[tid * AW_NAP + j];
      }
      sys_step_Fu<SYS, double>(P, x, u, xn, Fu);
      xn[NX] = x[NX] + P.dt;
#pragma unroll
      for (int i = 0; i < NX; ++i) {
        const double inv = P.normalize ? 1.0 / P.state_norm[i] : 1.0;
#pragma unroll
        for (int j = 0; j < NA; ++j) FU[tid * AW_FUP + i * NA + j] = (float)(Fu[i * NA + j] * inv);
      }
#pragma unroll
      for (int j = 0; j < NA; ++j) FU[tid * AW_FUP + NX * NA + j] = 0.f;
#pragma unroll
      for (int j = 0; j < NS; ++j) xnp[j] = normalize_component(P, j, (float)xn[j]);
      const double tm = term[b];
      const float w6 = (float)(tm * P.w_terminal[6] + (1.0 - tm) * P.w_running[6]);     // NeuralNetwork.py:201
      float uf[NA], g[NA];
#pragma unroll
      for (int j = 0; j < NA; ++j) uf[j] = ACT[tid * AW_NAP + j];
      sys_dr_da<SYS, float>(P, w6, uf, g);
#pragma unroll
      for (int j = 0; j < NA; ++j) DRDA[tid * AW_NAP + j] = g[j];
    }
#pragma unroll
    for (int j = 0; j < AW_NSP; ++j) XNP[tid * AW_NSP + j] = xnp[j];
  }
  __syncthreads();

  // ---- critic forward at s' keeping cos z_l, then the input-gradient sweep (NeuralNetwork.py:190-195)
  auto cf_epi = [&](int l, float* out) {
    return [&, l, out](int r, int c, float a) {
      float s, co;
      sincosf(a + __ldg(cw + LC.b[l] + c), &s, &co);
      out[r * CR_H4 + c] = s;
      CS[r * AW_CW + aw_koff(l) + c] = co;
    };
  };
  wgemm<S, TM>(XNP, AW_NSP, NS, cw + LC.W[0], CR_H1, CR_H1, cf_epi(0, C0));
  __syncthreads();
  wgemm<S, TM>(C0, CR_H4, CR_H1, cw + LC.W[1], CR_H2, CR_H2, cf_epi(1, C1));
  __syncthreads();
  wgemm<S, TM>(C1, CR_H4, CR_H2, cw + LC.W[2], CR_H3, CR_H3, cf_epi(2, C0));
  __syncthreads();
  wgemm<S, TM>(C0, CR_H4, CR_H3, cw + LC.W[3], CR_H4, CR_H4, cf_epi(3, C1));
  __syncthreads();
  for (int i = tid; i < S * CR_H4; i += AW_NT) {
    const int s = i / CR_H4, o = i - s * CR_H4;
    C0[i] = __ldg(cw + LC.W[4] + o) * CS[s * AW_CW + aw_koff(3) + o];
  }
  __syncthreads();
  // transposed block: W_l^T [out][in] at the same offsets, so the sweep is C = G W^T with W^T read row-major (ldw = in_l)
  auto cg_epi = [&](int l, float* out) {
    return [&, l, out](int r, int c, float a) { out[r * CR_H4 + c] = a * CS[r * AW_CW + aw_koff(l) + c]; };
  };
  wgemm<S, TM>(C0, CR_H4, CR_H4, cwT + LC.W[3], CR_H3, CR_H3, cg_epi(2, C1));
  __syncthreads();
  wgemm<S, TM>(C1, CR_H4, CR_H3, cwT + LC.W[2], CR_H2, CR_H2, cg_epi(1, C0));
  __syncthreads();
  wgemm<S, TM>(C0, CR_H4, CR_H2, cwT + LC.W[1], CR_H1, CR_H1, cg_epi(0, C1));
  __syncthreads();
  wgemm<S, TM>(C1, CR_H4, CR_H1, cwT + LC.W[0], NS, NS, [&](int r, int c, float a) { G0[r * AW_NSP + c] = a; });
  __syncthreads();

  // ---- dQ/da = dV/ds' . ds'/da + dr/da ; upstream gradient on the actor output = -dQ/da / B  (:206-228)
  for (int i = tid; i < S * AW_NAP; i += AW_NT) {
    const int s = i / AW_NAP, j = i - s * AW_NAP;
    float d3 = 0.f;
    if (s < rows && j < NA) {
      float q = DRDA[s * AW_NAP + j];
#pragma unroll
      for (int k = 0; k < NS; ++k) q = fmaf(normalize_scale(P, k) * G0[s * AW_NSP + k], FU[s * AW_FUP + k * NA + j], q);
      d3 = -q * inv_B;
    }
    D3[i] = d3;
  }
  __syncthreads();

  // ---- actor backward
  for (int i = tid; i < h2 * NA; i += AW_NT) {                 // dW3[k][j] += sum_s h2[s][k] d3[s][j]
    const int k = i / NA, j = i - k * NA;
    float acc = 0.f;
    for (int s = 0; s < rows; ++s) acc = fmaf(H2[s * ld2 + k], D3[s * AW_NAP + j], acc);
    grad_add<DET>(grad + LA.W3 + i, acc);
  }
  if (tid < NA) {
    float acc = 0.f;
    for (int s = 0; s < rows; ++s) acc += D3[s * AW_NAP + tid];
    grad_add<DET>(grad + LA.b3 + tid, acc);
  }
  for (int i = tid; i < S * h2; i += AW_NT) {                  // e2 = (d3 W3^T) * lrelu'(z2)
    const int s = i / h2, n = i - s * h2;
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < NA; ++j) acc = fmaf(D3[s * AW_NAP + j], __ldg(aw + LA.W3 + n * NA + j), acc);
    E[s * ld2 + n] = acc * (H2[s * ld2 + n] > 0.f ? 1.f : LEAKY_ALPHA);
  }
  __syncthreads();
  wouter<DET>(H1, ld1, E, ld2, h1, h2, grad + LA.W2, rows);
  tile_colsum<AW_NT, DET>(E, ld2, h2, rows, grad + LA.b2);
  // e1 = (e2 W2^T) * lrelu'(z1), re-strided to ld1, into the buffer of H2 (dead once e2 is formed; sized for either stride)
  float* E1 = H2;
  wgemm_nt<S>(E, ld2, h2, aw + LA.W2, h2, h1, [&](int s, int i, float v) { E1[s * ld1 + i] = v * (H1[s * ld1 + i] > 0.f ? 1.f : LEAKY_ALPHA); });
  __syncthreads();
  wouter<DET>(XN, AW_NSP, E1, ld1, NS, h1, grad + LA.W1, rows);
  tile_colsum<AW_NT, DET>(E1, ld1, h1, rows, grad + LA.b1);
}

template <typename K>
static int aw_smem_attr(K k, size_t bytes) {
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  return e == cudaSuccess ? 0 : (int)e;
}

template <int SYS, int S>
static int launch_rollout_width_s(const cacto_sys_params& P, const float* actor, int h1, int h2, const double* ics, const int32_t* horizon,
                                  int T_max, double* states, double* controls, int32_t* flags, double* rewards, int64_t B, cudaStream_t st) {
  auto k = k_rollout_width<SYS, S>;
  const size_t sm = ro_smem_bytes(S, h1, h2);
  if (int e = aw_smem_attr(k, sm)) return e;
  k<<<(unsigned)((B + S - 1) / S), AW_NT, sm, st>>>(P, actor, h1, h2, ics, horizon, T_max, states, controls, flags, rewards, B);
  CACTO_LAUNCH_CHECK();
  return 0;
}
template <int SYS>
static int launch_rollout_width(const cacto_sys_params& P, const float* actor, int h1, int h2, const double* ics, const int32_t* horizon,
                                int T_max, double* states, double* controls, int32_t* flags, double* rewards, int64_t B, cudaStream_t st) {
  if (ro_smem_bytes(AW_RO_S, h1, h2) > AW_RO_WIDE_BYTES)
    return launch_rollout_width_s<SYS, AW_RO_S_WIDE>(P, actor, h1, h2, ics, horizon, T_max, states, controls, flags, rewards, B, st);
  return launch_rollout_width_s<SYS, AW_RO_S>(P, actor, h1, h2, ics, horizon, T_max, states, controls, flags, rewards, B, st);
}

template <int SYS, int S>
static int launch_actor_grad_width_s(const cacto_sys_params& P, const float* aw, int h1, int h2, const float* cw, const float* cwT, const float* state,
                                     const double* term, float inv_B, float* grad, float* actions, int64_t B, cudaStream_t st) {
  auto k = k_actor_grad_width<SYS, S>;
  const size_t sm = ag_smem_bytes(S, h1, h2);
  if (int e = aw_smem_attr(k, sm)) return e;
  if (cudaError_t le = launch_pdl(k, (unsigned)((B + S - 1) / S), AW_NT, sm, st, P, aw, h1, h2, cw, cwT, state, term, inv_B, grad, actions, B))
    return (int)le;
  return 0;
}

template <int SYS>
static int launch_actor_grad_width(const cacto_sys_params& P, const float* aw, int h1, int h2, const float* cw, const float* cwT, const float* state,
                                   const double* term, float inv_B, float* grad, float* actions, int64_t B, cudaStream_t st) {
  if (actor_width_tile(B) == 4) return launch_actor_grad_width_s<SYS, 4>(P, aw, h1, h2, cw, cwT, state, term, inv_B, grad, actions, B, st);
  return launch_actor_grad_width_s<SYS, 16>(P, aw, h1, h2, cw, cwT, state, term, inv_B, grad, actions, B, st);
}

// deterministic variant: DET = true in waves of at most CACTO_DET_MAX_SLICES CTAs, then the fixed-order reduce (det.cuh)
template <int SYS, int S>
static int actor_grad_width_det_s(const cacto_sys_params& P, const float* aw, int h1, int h2, const float* cw, const float* cwT, const float* state,
                                  const double* term, float inv_B, float* grad, float* actions, int64_t B, float* part, cudaStream_t st) {
  auto k = k_actor_grad_width<SYS, S, true>;
  const size_t sm = ag_smem_bytes(S, h1, h2);
  if (int e = aw_smem_attr(k, sm)) return e;
  const int64_t n = ActorLayout(P.ns, P.na, h1, h2).total, tiles = (B + S - 1) / S, slices = det_slices(tiles), ns = P.ns, na = P.na;
  if (cudaError_t e = cudaMemsetAsync(part, 0, (size_t)(slices * det_stride(n)) * sizeof(float), st)) return (int)e;
  for (int64_t t0 = 0; t0 < tiles; t0 += slices) {
    const int64_t r0 = t0 * S, rows = B - r0 < slices * S ? B - r0 : slices * S;
    if (cudaError_t le = launch_pdl(k, (unsigned)((rows + S - 1) / S), AW_NT, sm, st, P, aw, h1, h2, cw, cwT, state + r0 * ns, term + r0, inv_B, part,
                                    actions ? actions + r0 * na : nullptr, rows))
      return (int)le;
    CACTO_LAUNCH_CHECK();
  }
  return det_reduce(part, slices, n, grad, nullptr, st);
}
template <int SYS>
static int actor_grad_width_det(const cacto_sys_params& P, const float* aw, int h1, int h2, const float* cw, const float* cwT, const float* state,
                                const double* term, float inv_B, float* grad, float* actions, int64_t B, float* part, cudaStream_t st) {
  if (actor_width_tile(B) == 4) return actor_grad_width_det_s<SYS, 4>(P, aw, h1, h2, cw, cwT, state, term, inv_B, grad, actions, B, part, st);
  return actor_grad_width_det_s<SYS, 16>(P, aw, h1, h2, cw, cwT, state, term, inv_B, grad, actions, B, part, st);
}

static bool aw_width_ok(int32_t h) { return h >= 1 && h <= CACTO_ACTOR_MAX_WIDTH; }
static bool aw_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace cacto

using namespace cacto;

extern "C" int64_t cacto_actor_width_param_count(int32_t ns, int32_t na, int32_t nh1, int32_t nh2) {
  if (ns < 1 || na < 1 || !aw_width_ok(nh1) || !aw_width_ok(nh2)) return CACTO_E_SIZE;
  return ActorLayout(ns, na, nh1, nh2).total;
}

#define AW_DISPATCH(FN, ...)                                                   \
  switch (p->system) {                                                         \
    case CACTO_SINGLE_INTEGRATOR: return FN<CACTO_SINGLE_INTEGRATOR>(__VA_ARGS__); \
    case CACTO_DOUBLE_INTEGRATOR: return FN<CACTO_DOUBLE_INTEGRATOR>(__VA_ARGS__); \
    case CACTO_CAR: return FN<CACTO_CAR>(__VA_ARGS__);                         \
    case CACTO_CAR_PARK: return FN<CACTO_CAR_PARK>(__VA_ARGS__);               \
    case CACTO_MANIPULATOR: return FN<CACTO_MANIPULATOR>(__VA_ARGS__);         \
    case CACTO_UR5: return FN<CACTO_UR5>(__VA_ARGS__);                         \
    default: return CACTO_E_SYSTEM;                                            \
  }

extern "C" int cacto_rollout_width(const cacto_sys_params* p, const float* actor_params, int32_t nh1, int32_t nh2, const double* ics,
                                   const int32_t* horizon, int32_t T_max, double* states, double* controls, int32_t* flags, double* rewards,
                                   int64_t B, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (!aw_width_ok(nh1) || !aw_width_ok(nh2) || B < 0 || T_max < 0) return CACTO_E_SIZE;
  if (!actor_params || !ics || !horizon || !states || !flags || (T_max > 0 && !controls)) return CACTO_E_ARG;
  if (!aw_aligned16(actor_params)) return CACTO_E_ALIGN;
  if (B == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  AW_DISPATCH(launch_rollout_width, *p, actor_params, nh1, nh2, ics, horizon, T_max, states, controls, flags, rewards, B, st)
}

extern "C" int cacto_actor_forward_width(const cacto_sys_params* p, const float* actor_params, int32_t nh1, int32_t nh2, const float* state,
                                         float* out, int64_t B, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (!aw_width_ok(nh1) || !aw_width_ok(nh2) || B < 0 || p->ns < 1 || p->ns > CACTO_MAX_NS || p->na < 1 || p->na > CACTO_MAX_NA)
    return CACTO_E_SIZE;
  if (!actor_params || !state || !out) return CACTO_E_ARG;
  if (!aw_aligned16(actor_params)) return CACTO_E_ALIGN;
  if (B == 0) return 0;
  const size_t sm = ro_smem_bytes(AW_RO_S, nh1, nh2);
  if (int e = aw_smem_attr(k_actor_forward_width, sm)) return e;
  k_actor_forward_width<<<(unsigned)((B + AW_RO_S - 1) / AW_RO_S), AW_NT, sm, (cudaStream_t)stream>>>(*p, actor_params, nh1, nh2, state, out, B);
  CACTO_LAUNCH_CHECK();
  return 0;
}

extern "C" int cacto_actor_grad_width(const cacto_sys_params* p, const float* actor_params, int32_t nh1, int32_t nh2, const float* critic_params,
                                      const float* critic_params_T, const float* state, const double* term, float inv_B, float* grad,
                                      float* actions, int64_t B, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (!aw_width_ok(nh1) || !aw_width_ok(nh2) || B < 0) return CACTO_E_SIZE;
  if (!actor_params || !critic_params || !critic_params_T || !state || !term || !grad) return CACTO_E_ARG;
  if (!aw_aligned16(actor_params) || !aw_aligned16(critic_params) || !aw_aligned16(critic_params_T) || !aw_aligned16(grad)) return CACTO_E_ALIGN;
  if (B == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  AW_DISPATCH(launch_actor_grad_width, *p, actor_params, nh1, nh2, critic_params, critic_params_T, state, term, inv_B, grad, actions, B, st)
}

extern "C" int cacto_actor_grad_width_det(const cacto_sys_params* p, const float* actor_params, int32_t nh1, int32_t nh2, const float* critic_params,
                                          const float* critic_params_T, const float* state, const double* term, float inv_B, float* grad,
                                          float* actions, int64_t B, float* partials, int64_t partials_floats, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (!aw_width_ok(nh1) || !aw_width_ok(nh2) || B < 0) return CACTO_E_SIZE;
  if (!actor_params || !critic_params || !critic_params_T || !state || !term || !grad || !partials) return CACTO_E_ARG;
  if (!aw_aligned16(actor_params) || !aw_aligned16(critic_params) || !aw_aligned16(critic_params_T) || !aw_aligned16(grad) || !aw_aligned16(partials))
    return CACTO_E_ALIGN;
  if (B == 0) return 0;
  const int64_t need = cacto_det_partials_floats(CACTO_DET_ACTOR_WIDTH, B, p->ns, p->na, nh1, nh2);
  if (need < 0 || partials_floats < need) return CACTO_E_SIZE;
  cudaStream_t st = (cudaStream_t)stream;
  AW_DISPATCH(actor_grad_width_det, *p, actor_params, nh1, nh2, critic_params, critic_params_T, state, term, inv_B, grad, actions, B, partials, st)
}
