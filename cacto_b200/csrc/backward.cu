// backward.cu -- K6: TO_Casadi.backward_pass (TO.py:119-202) for a batch of TO trajectories.
//
// The reference walks every trajectory backwards in Python: per knot it calls Env.augmented_derivative (K2), evaluates
// CasADi-differentiated cost gradients / Hessians (TO.py:147-164) and applies the DDP value recursion (TO.py:176-200);
// the result V_x is the dVdx column block of the replay buffer (main.py:237-240) that the Sobolev critic learns from.
// Here:
//   k_bp_knots    one thread per knot (all trajectories at once): A, B = sys_jac (the K2 arithmetic); l_x, l_xx of the
//                 reward (= -CAMS.cost, environment_TO.py cost_fun) by evaluating sys_reward on hyper-dual numbers
//                 (value, two first-order parts, one mixed second-order part: exact derivatives, no symbolic engine,
//                 everything in registers); l_u, l_uu of the separable control cost in closed form; l_xu = 0.  The per-knot
//                 code (bp_knot.cuh) is shared with the iLQR solver K7 (ddp.cu).
//   k_bp_riccati  one thread per trajectory: the recursion of TO.py:182-200 in fp64, with pinv(Q_uu + mu I) computed by
//                 a cyclic Jacobi eigen-decomposition (numpy.linalg.pinv semantics: |eigenvalue| <= 1e-15 max -> 0).
// Trajectories are ragged and concatenated (offsets[E+1], like cacto_rtg_window).  Workspace per knot:
// [l_x | l_xx | A | B | l_u | l_uu(diag)] doubles, caller-owned.
#include "bp_knot.cuh"

namespace cacto {

// ------------------------------------------------------------------------------------------ per-knot quantities
template <int SYS>
__global__ void __launch_bounds__(128) k_bp_knots(const __grid_constant__ cacto_sys_params P, const int64_t* __restrict__ offsets, int E,
                                                  const double* __restrict__ states, const double* __restrict__ controls,
                                                  double* __restrict__ ws, int64_t K) {
  constexpr int NX = SysDims<SYS>::NX, NA = SysDims<SYS>::NA, W = bp_stride(NX, NA);
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  const int e = knot_owner(offsets, E, k);
  const bool last = (k == offsets[e + 1] - 1);                    // terminal knot of its trajectory
  bp_knot_eval<SYS>(P, states + k * NX, controls + k * NA, last, ws + k * W);
}

// ------------------------------------------------------------------------------------------ pinv of a small symmetric matrix
// Cyclic Jacobi on shared-memory arrays A, V (M x M each), executed by ONE lane (the rotations are sequential); the caller
// synchronises the warp around it.  Same arithmetic and rotation order as the first version, which kept A and V in local memory.
template <int M>
__device__ void pinv_sym_lane(const double* Q, double* A, double* V) {
  for (int i = 0; i < M; ++i)
    for (int j = 0; j < M; ++j) {
      A[i * M + j] = 0.5 * (Q[i * M + j] + Q[j * M + i]);
      V[i * M + j] = (i == j) ? 1.0 : 0.0;
    }
  for (int sweep = 0; sweep < 40; ++sweep) {
    double off = 0.0, diag = 0.0;
    for (int i = 0; i < M; ++i)
      for (int j = 0; j < M; ++j) {
        if (i != j) off += A[i * M + j] * A[i * M + j]; else diag += A[i * M + j] * A[i * M + j];
      }
    // converged once the off-diagonal mass is at rounding level (sums of SQUARES: 1e-30 = (1e-15)^2).  The first version asked for
    // 1e-40, which rounding never reaches: all 40 sweeps ran at every knot -- 180 k warp instructions per knot for the UR5 (ncu).
    if (off <= 1e-30 * diag || off == 0.0) break;
    for (int p = 0; p < M - 1; ++p)
      for (int q = p + 1; q < M; ++q) {
        const double apq = A[p * M + q];
        if (apq == 0.0) continue;
        const double theta = (A[q * M + q] - A[p * M + p]) / (2.0 * apq);
        const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < M; ++k) {                      // A <- A J (columns p, q)
          const double akp = A[k * M + p], akq = A[k * M + q];
          A[k * M + p] = c * akp - s * akq;
          A[k * M + q] = s * akp + c * akq;
        }
        for (int k = 0; k < M; ++k) {                      // A <- J^T A (rows p, q)
          const double apk = A[p * M + k], aqk = A[q * M + k];
          A[p * M + k] = c * apk - s * aqk;
          A[q * M + k] = s * apk + c * aqk;
        }
        for (int k = 0; k < M; ++k) {
          const double vkp = V[k * M + p], vkq = V[k * M + q];
          V[k * M + p] = c * vkp - s * vkq;
          V[k * M + q] = s * vkp + c * vkq;
        }
      }
  }
}

// ------------------------------------------------------------------------------------------ value recursion
// One WARP per trajectory, all matrices in shared memory: every entry of V_xx A, V_xx B, the Q blocks, the gains and the new
// V_x / V_xx is a short dot product owned by one lane (entries are dealt round-robin), a __syncwarp() between the stages.
// (First version: one THREAD per trajectory with the same loops over local-memory arrays -- 0.58 ms per knot for the UR5's 12 x 12
// blocks, every operand an L1 round trip on a dependent chain; each entry is computed by the same expression as before.)
template <int SYS>
__global__ void __launch_bounds__(32) k_bp_riccati(const int64_t* __restrict__ offsets, int E, const double* __restrict__ ws, double mu,
                                                   double* __restrict__ Vx_out) {
  constexpr int NX = SysDims<SYS>::NX, NA = SysDims<SYS>::NA, W = bp_stride(NX, NA);
  __shared__ double Vx[NX], Vxx[NX * NX], VA[NX * NX], VB[NX * NA], Qx[NX], Qu[NA], Qxx[NX * NX], Quu[NA * NA], Qxu[NX * NA];
  __shared__ double Pi[NA * NA], PQu[NA], G[NX * NA], JA[NA * NA], JV[NA * NA], knot[W];
  const int e = blockIdx.x, lane = threadIdx.x;
  if (e >= E) return;
  const int64_t k0 = offsets[e], k1 = offsets[e + 1];
  if (k1 <= k0) return;
  {
    const double* o = ws + (k1 - 1) * W;                          // terminal knot: V = l (TO.py:172-174)
    for (int i = lane; i < NX; i += 32) { Vx[i] = o[i]; Vx_out[(k1 - 1) * (NX + 1) + i] = o[i]; }
    for (int i = lane; i < NX * NX; i += 32) Vxx[i] = o[NX + i];
    if (lane == 0) Vx_out[(k1 - 1) * (NX + 1) + NX] = 0.0;
  }
  __syncwarp();
  for (int64_t k = k1 - 2; k >= k0; --k) {
    for (int i = lane; i < W; i += 32) knot[i] = ws[k * W + i];
    __syncwarp();
    const double* lx = knot, *lxx = knot + NX, *A = lxx + NX * NX, *Bm = A + NX * NX, *lu = Bm + NX * NA, *luu = lu + NA;
    for (int idx = lane; idx < NX * (NX + NA); idx += 32) {       // V_xx A | V_xx B
      const int i = idx / (NX + NA), j = idx - i * (NX + NA);
      double s = 0.0;
      if (j < NX) {
        for (int c = 0; c < NX; ++c) s += Vxx[i * NX + c] * A[c * NX + j];
        VA[i * NX + j] = s;
      } else {
        for (int c = 0; c < NX; ++c) s += Vxx[i * NX + c] * Bm[c * NA + (j - NX)];
        VB[i * NA + (j - NX)] = s;
      }
    }
    __syncwarp();
    for (int idx = lane; idx < (NX + NA) * (1 + NX + NA); idx += 32) {   // Q_x | Q_xx | Q_xu ; Q_u | Q_uu (rows of [A B]^T)
      const int r = idx / (1 + NX + NA), cidx = idx - r * (1 + NX + NA);
      if (r < NX) {
        const int i = r;
        if (cidx == 0) {
          double s = lx[i];
          for (int c = 0; c < NX; ++c) s += A[c * NX + i] * Vx[c];
          Qx[i] = s;
        } else if (cidx <= NX) {
          const int j = cidx - 1;
          double t = lxx[i * NX + j];
          for (int c = 0; c < NX; ++c) t += A[c * NX + i] * VA[c * NX + j];
          Qxx[i * NX + j] = t;
        } else {
          const int j = cidx - 1 - NX;
          double t = 0.0;                                          // l_xu = 0: the cost is separable in x and u
          for (int c = 0; c < NX; ++c) t += A[c * NX + i] * VB[c * NA + j];
          Qxu[i * NA + j] = t;
        }
      } else {
        const int i = r - NX;
        if (cidx == 0) {
          double s = lu[i];
          for (int c = 0; c < NX; ++c) s += Bm[c * NA + i] * Vx[c];
          Qu[i] = s;
        } else if (cidx <= NA) {
          const int j = cidx - 1;
          double t = (i == j) ? luu[i] + mu : 0.0;                 // Qbar_uu = Q_uu + mu I (TO.py:192)
          for (int c = 0; c < NX; ++c) t += Bm[c * NA + i] * VB[c * NA + j];
          Quu[i * NA + j] = t;
        }
      }
    }
    __syncwarp();
    if (lane == 0) pinv_sym_lane<NA>(Quu, JA, JV);                 // eigen-decomposition of Qbar_uu
    __syncwarp();
    {
      double lmax = 0.0;
      for (int i = 0; i < NA; ++i) lmax = fmax(lmax, fabs(JA[i * NA + i]));
      const double cut = 1e-15 * lmax;
      for (int idx = lane; idx < NA * NA; idx += 32) {
        const int i = idx / NA, j = idx - i * NA;
        double acc = 0.0;
        for (int ev = 0; ev < NA; ++ev) {
          const double l = JA[ev * NA + ev];
          if (fabs(l) <= cut) continue;
          const double inv = 1.0 / l;
          acc += inv * JV[i * NA + ev] * JV[j * NA + ev];
        }
        Pi[idx] = acc;
      }
    }
    __syncwarp();
    for (int idx = lane; idx < NA + NX * NA; idx += 32) {          // pinv Q_u | Q_xu pinv
      if (idx < NA) {
        double s = 0.0;
        for (int j = 0; j < NA; ++j) s += Pi[idx * NA + j] * Qu[j];
        PQu[idx] = s;
      } else {
        const int i = (idx - NA) / NA, j = (idx - NA) - i * NA;
        double s = 0.0;
        for (int c = 0; c < NA; ++c) s += Qxu[i * NA + c] * Pi[c * NA + j];
        G[i * NA + j] = s;
      }
    }
    __syncwarp();
    for (int idx = lane; idx < NX * (1 + NX); idx += 32) {         // V_x | V_xx
      const int i = idx / (1 + NX), cidx = idx - i * (1 + NX);
      if (cidx == 0) {
        double s = Qx[i];
        for (int j = 0; j < NA; ++j) s -= Qxu[i * NA + j] * PQu[j];
        Vx[i] = s;
        Vx_out[k * (NX + 1) + i] = s;
      } else {
        const int j = cidx - 1;
        double t = Qxx[i * NX + j];
        for (int c = 0; c < NA; ++c) t -= G[i * NA + c] * Qxu[j * NA + c];
        Vxx[i * NX + j] = t;
      }
    }
    if (lane == 0) Vx_out[k * (NX + 1) + NX] = 0.0;
    __syncwarp();
  }
}

template <int SYS>
static int launch_backward(const cacto_sys_params& P, const int64_t* offsets, int E, const double* states, const double* controls, double mu,
                           double* ws, double* Vx, int64_t K, cudaStream_t st) {
  k_bp_knots<SYS><<<(unsigned)((K + 127) / 128), 128, 0, st>>>(P, offsets, E, states, controls, ws, K);
  CACTO_LAUNCH_CHECK();
  k_bp_riccati<SYS><<<(unsigned)E, 32, 0, st>>>(offsets, E, ws, mu, Vx);
  CACTO_LAUNCH_CHECK();
  return 0;
}

}  // namespace cacto

using namespace cacto;

extern "C" int64_t cacto_backward_pass_workspace_bytes(int32_t nx, int32_t na, int64_t n_knots) {
  if (nx < 1 || na < 1 || n_knots < 0) return CACTO_E_SIZE;
  return (int64_t)sizeof(double) * bp_stride(nx, na) * n_knots;
}

extern "C" int cacto_backward_pass(const cacto_sys_params* p, const int64_t* offsets, int32_t E, const double* states, const double* controls,
                                   int64_t n_knots, double mu, void* workspace, double* V_x, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (E < 0 || n_knots < 0) return CACTO_E_SIZE;
  if (E == 0 || n_knots == 0) return 0;
  if (!offsets || !states || !controls || !workspace || !V_x) return CACTO_E_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  double* ws = static_cast<double*>(workspace);
  switch (p->system) {
    case CACTO_SINGLE_INTEGRATOR: return launch_backward<CACTO_SINGLE_INTEGRATOR>(*p, offsets, E, states, controls, mu, ws, V_x, n_knots, st);
    case CACTO_DOUBLE_INTEGRATOR: return launch_backward<CACTO_DOUBLE_INTEGRATOR>(*p, offsets, E, states, controls, mu, ws, V_x, n_knots, st);
    case CACTO_CAR: return launch_backward<CACTO_CAR>(*p, offsets, E, states, controls, mu, ws, V_x, n_knots, st);
    case CACTO_CAR_PARK: return launch_backward<CACTO_CAR_PARK>(*p, offsets, E, states, controls, mu, ws, V_x, n_knots, st);
    case CACTO_MANIPULATOR: return launch_backward<CACTO_MANIPULATOR>(*p, offsets, E, states, controls, mu, ws, V_x, n_knots, st);
    case CACTO_UR5: return launch_backward<CACTO_UR5>(*p, offsets, E, states, controls, mu, ws, V_x, n_knots, st);
    default: return CACTO_E_SYSTEM;
  }
}
