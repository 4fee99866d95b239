// ddp.cu -- K7: the TO solve as batched iLQR (include/cacto_b200.h states the problem and the rule; oracle/ddp.py restates both).
//
//   k_ddp_knots     one thread per knot of the trajectories still running: K6's per-knot derivatives (bp_knot.cuh) at the iterate.
//   k_ddp_backward  one warp per trajectory, the structure of k_bp_riccati on the cost (the reward terms negated): Q blocks,
//                   Cholesky of Q_uu + mu I (lane 0), the NX + 1 triangular solves for k and K (one lane each), V_x / V_xx and the
//                   expected-change sums.  A non-positive pivot fails the pass.
//   k_ddp_probe     one thread per (trajectory, alpha): the closed-loop rollout, cost only.
//   k_ddp_commit    one thread per trajectory: the acceptance rule, the committed rollout (same function as the probe, so the cost
//                   written is the probed cost bit for bit), mu and status.
// The rollout is one __noinline__ function that the probe, the commit and the initial-cost kernel all call: one compiled body,
// one rounding of every operation.
#include "bp_knot.cuh"

namespace cacto {

__host__ __device__ constexpr int ddp_stride(int nx, int na) { return bp_stride(nx, na) + na + na * nx; }
enum { R_MU = 0, R_DV1 = 1, R_DV2 = 2, R_OK = 3, R_PROBE = 4, R_HIST = R_PROBE + CACTO_DDP_N_ALPHA };
static_assert(R_HIST + CACTO_DDP_HISTORY <= CACTO_DDP_TRAJ_DOUBLES, "trajectory record");

// J of the rollout from x_0 = states[k0] over knots k0 .. k1-1: u_k = u_bar_k (gains == nullptr) or
// u_bar_k + alpha k_k + K_k (x_k - x_bar_k).  write: the rollout replaces the iterate (x_bar_k is read before x_k overwrites it;
// the controls are written only with gains, the open-loop rollout leaves them as they are).
template <int SYS>
__device__ __noinline__ double ddp_rollout(const cacto_sys_params& P, int64_t k0, int64_t k1, const double* __restrict__ gains,
                                           double alpha, double* states, double* controls, bool write) {
  constexpr int NX = SysDims<SYS>::NX, NA = SysDims<SYS>::NA, WD = ddp_stride(NX, NA), W = bp_stride(NX, NA);
  double x[NX + 1], xn[NX + 1], u[NA];
  for (int i = 0; i < NX; ++i) x[i] = states[k0 * NX + i];
  x[NX] = 0.0;
  xn[NX] = 0.0;
  double J = 0.0;
  for (int64_t k = k0; k < k1 - 1; ++k) {
    if (gains != nullptr) {
      const double* kk = gains + k * WD + W, *KK = kk + NA;
      double dx[NX];
      for (int i = 0; i < NX; ++i) dx[i] = x[i] - states[k * NX + i];
      for (int a = 0; a < NA; ++a) {
        double s = controls[k * NA + a] + alpha * kk[a];
        for (int i = 0; i < NX; ++i) s += KK[a * NX + i] * dx[i];
        u[a] = s;
      }
    } else {
      for (int a = 0; a < NA; ++a) u[a] = controls[k * NA + a];
    }
    J -= sys_reward<SYS, double>(P, P.w_running, x, u, false);
    sys_step<SYS, double>(P, x, u, xn);
    if (write) {
      if (k > k0)
        for (int i = 0; i < NX; ++i) states[k * NX + i] = x[i];
      if (gains != nullptr)
        for (int a = 0; a < NA; ++a) controls[k * NA + a] = u[a];
    }
    for (int i = 0; i < NX; ++i) x[i] = xn[i];
  }
  J -= sys_reward<SYS, double>(P, P.w_terminal, x, (const double*)nullptr, false);
  if (write && k1 - 1 > k0)
    for (int i = 0; i < NX; ++i) states[(k1 - 1) * NX + i] = x[i];
  return J;
}

template <int SYS>
__global__ void __launch_bounds__(128) k_ddp_init(const __grid_constant__ cacto_sys_params P, const int64_t* __restrict__ offsets, int E,
                                                  double* states, double* controls, double* __restrict__ rec, double* __restrict__ cost,
                                                  int32_t* __restrict__ status, int32_t* __restrict__ iters) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E) return;
  double* r = rec + (int64_t)e * CACTO_DDP_TRAJ_DOUBLES;
  r[R_MU] = CACTO_DDP_MU_INIT;
  r[R_DV1] = r[R_DV2] = 0.0;
  r[R_OK] = 0.0;
  for (int j = 0; j < CACTO_DDP_N_ALPHA; ++j) r[R_PROBE + j] = 0.0;
  for (int j = 0; j < CACTO_DDP_HISTORY; ++j) r[R_HIST + j] = CACTO_DDP_H_NOT_RUN;
  iters[e] = 0;
  const int64_t k0 = offsets[e], k1 = offsets[e + 1];
  if (k1 <= k0) { cost[e] = 0.0; status[e] = CACTO_DDP_CONVERGED; return; }
  const double J = ddp_rollout<SYS>(P, k0, k1, nullptr, 0.0, states, controls, true);
  cost[e] = J;
  status[e] = !isfinite(J) ? CACTO_DDP_FAILED : (k1 - k0 == 1 ? CACTO_DDP_CONVERGED : CACTO_DDP_RUNNING);
}

template <int SYS>
__global__ void __launch_bounds__(128) k_ddp_knots(const __grid_constant__ cacto_sys_params P, const int64_t* __restrict__ offsets, int E,
                                                   const double* __restrict__ states, const double* __restrict__ controls,
                                                   const int32_t* __restrict__ status, double* __restrict__ ws, int64_t K) {
  constexpr int NX = SysDims<SYS>::NX, NA = SysDims<SYS>::NA, WD = ddp_stride(NX, NA);
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  const int e = knot_owner(offsets, E, k);
  if (status[e] != CACTO_DDP_RUNNING) return;
  bp_knot_eval<SYS>(P, states + k * NX, controls + k * NA, k == offsets[e + 1] - 1, ws + k * WD);
}

template <int SYS>
__global__ void __launch_bounds__(32) k_ddp_backward(const int64_t* __restrict__ offsets, int E, const int32_t* __restrict__ status,
                                                     double* __restrict__ ws, double* __restrict__ rec) {
  constexpr int NX = SysDims<SYS>::NX, NA = SysDims<SYS>::NA, W = bp_stride(NX, NA), WD = ddp_stride(NX, NA);
  __shared__ double Vx[NX], Vxx[NX * NX], VA[NX * NX], VB[NX * NA], Qx[NX], Qu[NA], Qxx[NX * NX], Quu[NA * NA], Qux[NA * NX];
  __shared__ double L[NA * NA], kk[NA], KK[NA * NX], Quuk[NA], QuuK[NA * NX], knot[W];
  __shared__ int fail;
  const int e = blockIdx.x, lane = threadIdx.x;
  if (e >= E || status[e] != CACTO_DDP_RUNNING) return;
  const int64_t k0 = offsets[e], k1 = offsets[e + 1];
  double* r = rec + (int64_t)e * CACTO_DDP_TRAJ_DOUBLES;
  const double mu = r[R_MU];
  {
    const double* o = ws + (k1 - 1) * WD;                         // terminal knot: V = c_term
    for (int i = lane; i < NX; i += 32) Vx[i] = -o[i];
    for (int i = lane; i < NX * NX; i += 32) Vxx[i] = -o[NX + i];
    if (lane == 0) fail = 0;
  }
  double dv1 = 0.0, dv2 = 0.0;                                     // lane 0's sums
  __syncwarp();
  for (int64_t k = k1 - 2; k >= k0; --k) {
    for (int i = lane; i < W; i += 32) knot[i] = ws[k * WD + i];
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
    for (int idx = lane; idx < (NX + NA) * (1 + NX); idx += 32) { // Q_x | Q_xx ; Q_u | Q_uu | Q_ux  (l_xu = 0)
      const int rr = idx / (1 + NX), c = idx - rr * (1 + NX);
      if (rr < NX) {
        const int i = rr;
        if (c == 0) {
          double s = -lx[i];
          for (int m = 0; m < NX; ++m) s += A[m * NX + i] * Vx[m];
          Qx[i] = s;
        } else {
          const int j = c - 1;
          double t = -lxx[i * NX + j];
          for (int m = 0; m < NX; ++m) t += A[m * NX + i] * VA[m * NX + j];
          Qxx[i * NX + j] = t;
        }
      } else {
        const int i = rr - NX;
        if (c == 0) {
          double s = -lu[i];
          for (int m = 0; m < NX; ++m) s += Bm[m * NA + i] * Vx[m];
          Qu[i] = s;
        } else {
          const int j = c - 1;
          double t = 0.0;
          for (int m = 0; m < NX; ++m) t += Bm[m * NA + i] * VA[m * NX + j];
          Qux[i * NX + j] = t;
          if (j < NA) {
            double q = (i == j) ? -luu[i] : 0.0;
            for (int m = 0; m < NX; ++m) q += Bm[m * NA + i] * VB[m * NA + j];
            Quu[i * NA + j] = q;
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0) {                                               // Cholesky of Quu + mu I
      for (int j = 0; j < NA; ++j) {
        double d = Quu[j * NA + j] + mu;
        for (int m = 0; m < j; ++m) d -= L[j * NA + m] * L[j * NA + m];
        if (!(d > 0.0) || !isfinite(d)) { fail = 1; break; }
        d = sqrt(d);
        L[j * NA + j] = d;
        for (int i = j + 1; i < NA; ++i) {
          double s = 0.5 * (Quu[i * NA + j] + Quu[j * NA + i]);
          for (int m = 0; m < j; ++m) s -= L[i * NA + m] * L[j * NA + m];
          L[i * NA + j] = s / d;
        }
      }
    }
    __syncwarp();
    if (fail) break;
    if (lane <= NX) {                                              // lane 0: k = -Quu~^-1 Q_u; lane 1 + i: column i of K
      double b[NA];
      for (int a = 0; a < NA; ++a) b[a] = lane == 0 ? -Qu[a] : -Qux[a * NX + lane - 1];
      for (int a = 0; a < NA; ++a) {
        double s = b[a];
        for (int m = 0; m < a; ++m) s -= L[a * NA + m] * b[m];
        b[a] = s / L[a * NA + a];
      }
      for (int a = NA - 1; a >= 0; --a) {
        double s = b[a];
        for (int m = a + 1; m < NA; ++m) s -= L[m * NA + a] * b[m];
        b[a] = s / L[a * NA + a];
      }
      for (int a = 0; a < NA; ++a) {
        if (lane == 0) kk[a] = b[a]; else KK[a * NX + lane - 1] = b[a];
      }
    }
    __syncwarp();
    double* g = ws + k * WD + W;                                   // [k | K] of this knot
    for (int idx = lane; idx < NA * (1 + NX); idx += 32) {         // Q_uu k | Q_uu K, and the gains to the workspace
      const int a = idx / (1 + NX), c = idx - a * (1 + NX);
      double s = 0.0;
      if (c == 0) {
        for (int m = 0; m < NA; ++m) s += Quu[a * NA + m] * kk[m];
        Quuk[a] = s;
        g[a] = kk[a];
      } else {
        for (int m = 0; m < NA; ++m) s += Quu[a * NA + m] * KK[m * NX + c - 1];
        QuuK[a * NX + c - 1] = s;
        g[NA + a * NX + c - 1] = KK[a * NX + c - 1];
      }
    }
    __syncwarp();
    if (lane == 0) {
      for (int a = 0; a < NA; ++a) {
        dv1 += kk[a] * Qu[a];
        dv2 += kk[a] * Quuk[a];
      }
    }
    for (int idx = lane; idx < NX * (1 + NX); idx += 32) {         // V_x | V_xx (unsymmetrised, into VA)
      const int i = idx / (1 + NX), c = idx - i * (1 + NX);
      if (c == 0) {
        double s = Qx[i];
        for (int a = 0; a < NA; ++a) s += KK[a * NX + i] * Quuk[a] + KK[a * NX + i] * Qu[a] + Qux[a * NX + i] * kk[a];
        Vx[i] = s;
      } else {
        const int j = c - 1;
        double t = Qxx[i * NX + j];
        for (int a = 0; a < NA; ++a) t += KK[a * NX + i] * QuuK[a * NX + j] + KK[a * NX + i] * Qux[a * NX + j] + Qux[a * NX + i] * KK[a * NX + j];
        VA[i * NX + j] = t;
      }
    }
    __syncwarp();
    for (int idx = lane; idx < NX * NX; idx += 32) {
      const int i = idx / NX, j = idx - i * NX;
      Vxx[idx] = 0.5 * (VA[i * NX + j] + VA[j * NX + i]);
    }
    __syncwarp();
  }
  if (lane == 0) {
    r[R_OK] = fail ? 0.0 : 1.0;
    r[R_DV1] = dv1;
    r[R_DV2] = dv2;
  }
}

__device__ __forceinline__ double ddp_alpha(int j) { return ldexp(1.0, -j); }

template <int SYS>
__global__ void __launch_bounds__(128) k_ddp_probe(const __grid_constant__ cacto_sys_params P, const int64_t* __restrict__ offsets, int E,
                                                   double* states, double* controls, const int32_t* __restrict__ status,
                                                   const double* __restrict__ ws, double* __restrict__ rec) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int e = t / CACTO_DDP_N_ALPHA, j = t - e * CACTO_DDP_N_ALPHA;
  if (e >= E || status[e] != CACTO_DDP_RUNNING) return;
  double* r = rec + (int64_t)e * CACTO_DDP_TRAJ_DOUBLES;
  if (r[R_OK] == 0.0) return;
  r[R_PROBE + j] = ddp_rollout<SYS>(P, offsets[e], offsets[e + 1], ws, ddp_alpha(j), states, controls, false);
}

template <int SYS>
__global__ void __launch_bounds__(128) k_ddp_commit(const __grid_constant__ cacto_sys_params P, const int64_t* __restrict__ offsets, int E,
                                                    double tol, double* states, double* controls, const double* __restrict__ ws,
                                                    double* __restrict__ rec, double* __restrict__ cost, int32_t* __restrict__ status,
                                                    int32_t* __restrict__ iters) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= E || status[e] != CACTO_DDP_RUNNING) return;
  double* r = rec + (int64_t)e * CACTO_DDP_TRAJ_DOUBLES;
  const int it = iters[e];
  iters[e] = it + 1;
  double mu = r[R_MU];
  const double J = cost[e];
  int outcome;
  if (r[R_OK] == 0.0) {
    outcome = CACTO_DDP_H_BACKWARD_FAILED;
  } else {
    const double dv1 = r[R_DV1], dv2 = r[R_DV2];
    if (fabs(dv1 + 0.5 * dv2) < tol * fabs(J)) {
      outcome = CACTO_DDP_H_CONVERGED;
    } else {
      outcome = CACTO_DDP_H_NO_STEP;
      for (int j = 0; j < CACTO_DDP_N_ALPHA; ++j) {
        const double a = ddp_alpha(j), Jp = r[R_PROBE + j];
        const double expected = -(a * dv1 + 0.5 * a * a * dv2);
        if (isfinite(Jp) && expected > 0.0 && J - Jp >= CACTO_DDP_C1 * expected) { outcome = j; break; }
      }
    }
  }
  if (it < CACTO_DDP_HISTORY) r[R_HIST + it] = outcome;
  if (outcome >= 0) {
    const double Jn = ddp_rollout<SYS>(P, offsets[e], offsets[e + 1], ws, ddp_alpha(outcome), states, controls, true);
    cost[e] = Jn;
    r[R_MU] = fmax(mu / CACTO_DDP_MU_FACTOR, CACTO_DDP_MU_MIN);
    if (J - Jn < tol * fabs(J)) status[e] = CACTO_DDP_CONVERGED;
  } else if (outcome == CACTO_DDP_H_CONVERGED) {
    status[e] = CACTO_DDP_CONVERGED;
  } else {
    mu *= CACTO_DDP_MU_FACTOR;
    r[R_MU] = mu;
    if (mu > CACTO_DDP_MU_MAX) status[e] = CACTO_DDP_FAILED;
  }
}

template <int SYS>
static int launch_ddp_init(const cacto_sys_params& P, const int64_t* offsets, int E, double* states, double* controls, double* rec,
                           double* cost, int32_t* status, int32_t* iters, cudaStream_t st) {
  k_ddp_init<SYS><<<(unsigned)((E + 127) / 128), 128, 0, st>>>(P, offsets, E, states, controls, rec, cost, status, iters);
  CACTO_LAUNCH_CHECK();
  return 0;
}

template <int SYS>
static int launch_ddp_iterate(const cacto_sys_params& P, const int64_t* offsets, int E, double* states, double* controls, int64_t K,
                              int n_iter, double tol, double* ws, double* rec, double* cost, int32_t* status, int32_t* iters,
                              cudaStream_t st) {
  const unsigned gk = (unsigned)((K + 127) / 128), gt = (unsigned)((E + 127) / 128);
  const unsigned gp = (unsigned)(((int64_t)E * CACTO_DDP_N_ALPHA + 127) / 128);
  for (int i = 0; i < n_iter; ++i) {
    k_ddp_knots<SYS><<<gk, 128, 0, st>>>(P, offsets, E, states, controls, status, ws, K);
    CACTO_LAUNCH_CHECK();
    k_ddp_backward<SYS><<<(unsigned)E, 32, 0, st>>>(offsets, E, status, ws, rec);
    CACTO_LAUNCH_CHECK();
    k_ddp_probe<SYS><<<gp, 128, 0, st>>>(P, offsets, E, states, controls, status, ws, rec);
    CACTO_LAUNCH_CHECK();
    k_ddp_commit<SYS><<<gt, 128, 0, st>>>(P, offsets, E, tol, states, controls, ws, rec, cost, status, iters);
    CACTO_LAUNCH_CHECK();
  }
  return 0;
}

static bool ddp_dims_ok(const cacto_sys_params* p) {
  switch (p->system) {
#define CACTO_DIMS(S) case S: return p->nx == SysDims<S>::NX && p->na == SysDims<S>::NA;
    CACTO_DIMS(CACTO_SINGLE_INTEGRATOR) CACTO_DIMS(CACTO_DOUBLE_INTEGRATOR) CACTO_DIMS(CACTO_CAR) CACTO_DIMS(CACTO_CAR_PARK)
    CACTO_DIMS(CACTO_MANIPULATOR) CACTO_DIMS(CACTO_UR5)
#undef CACTO_DIMS
    default: return false;
  }
}

}  // namespace cacto

using namespace cacto;

extern "C" int64_t cacto_ddp_workspace_bytes(int32_t nx, int32_t na, int64_t n_knots, int32_t E) {
  if (nx < 1 || na < 1 || n_knots < 0 || E < 0) return CACTO_E_SIZE;
  return (int64_t)sizeof(double) * ((int64_t)ddp_stride(nx, na) * n_knots + (int64_t)CACTO_DDP_TRAJ_DOUBLES * E);
}

#define CACTO_DDP_DISPATCH(call)                                                     \
  switch (p->system) {                                                               \
    case CACTO_SINGLE_INTEGRATOR: { constexpr int S = CACTO_SINGLE_INTEGRATOR; return call; } \
    case CACTO_DOUBLE_INTEGRATOR: { constexpr int S = CACTO_DOUBLE_INTEGRATOR; return call; } \
    case CACTO_CAR: { constexpr int S = CACTO_CAR; return call; }                    \
    case CACTO_CAR_PARK: { constexpr int S = CACTO_CAR_PARK; return call; }          \
    case CACTO_MANIPULATOR: { constexpr int S = CACTO_MANIPULATOR; return call; }    \
    case CACTO_UR5: { constexpr int S = CACTO_UR5; return call; }                    \
    default: return CACTO_E_SYSTEM;                                                  \
  }

// the per-trajectory records follow the per-knot blocks
static double* ddp_records(const cacto_sys_params* p, void* workspace, int64_t n_knots) {
  return static_cast<double*>(workspace) + (int64_t)ddp_stride(p->nx, p->na) * n_knots;
}

extern "C" int cacto_ddp_init(const cacto_sys_params* p, const int64_t* offsets, int32_t E, double* states, const double* controls,
                              int64_t n_knots, void* workspace, double* cost, int32_t* status, int32_t* iters, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (p->system < CACTO_SINGLE_INTEGRATOR || p->system > CACTO_UR5) return CACTO_E_SYSTEM;
  if (!ddp_dims_ok(p) || E < 0 || n_knots < 0) return CACTO_E_SIZE;
  if (E == 0) return 0;
  if (!offsets || !workspace || !cost || !status || !iters || (n_knots > 0 && (!states || !controls))) return CACTO_E_ARG;
  if ((reinterpret_cast<uintptr_t>(workspace) & 7) != 0) return CACTO_E_ALIGN;
  cudaStream_t st = (cudaStream_t)stream;
  double* rec = ddp_records(p, workspace, n_knots);
  double* ctl = const_cast<double*>(controls);                     // read only: the open-loop rollout writes states alone
  CACTO_DDP_DISPATCH((launch_ddp_init<S>(*p, offsets, E, states, ctl, rec, cost, status, iters, st)))
}

extern "C" int cacto_ddp_iterate(const cacto_sys_params* p, const int64_t* offsets, int32_t E, double* states, double* controls,
                                 int64_t n_knots, int32_t n_iter, double tol, void* workspace, double* cost, int32_t* status,
                                 int32_t* iters, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (p->system < CACTO_SINGLE_INTEGRATOR || p->system > CACTO_UR5) return CACTO_E_SYSTEM;
  if (!ddp_dims_ok(p) || E < 0 || n_knots < 0 || n_iter < 0) return CACTO_E_SIZE;
  if (E == 0 || n_knots == 0 || n_iter == 0) return 0;
  if (!offsets || !states || !controls || !workspace || !cost || !status || !iters) return CACTO_E_ARG;
  if ((reinterpret_cast<uintptr_t>(workspace) & 7) != 0) return CACTO_E_ALIGN;
  cudaStream_t st = (cudaStream_t)stream;
  double* ws = static_cast<double*>(workspace);
  double* rec = ddp_records(p, workspace, n_knots);
  CACTO_DDP_DISPATCH((launch_ddp_iterate<S>(*p, offsets, E, states, controls, n_knots, n_iter, tol, ws, rec, cost, status, iters, st)))
}
