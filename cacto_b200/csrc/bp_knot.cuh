// bp_knot.cuh -- the per-knot quantities of the TO backward pass (K6, backward.cu) shared with the iLQR solver (K7, ddp.cu):
// at one knot (x, u) of a trajectory, A, B = sys_jac and the gradient / Hessian of the reward (hyper-dual evaluation of sys_reward
// for the state part, closed form for the separable control part).  Layout of one knot's block (bp_stride(nx, na) doubles):
// [l_x | l_xx | A | B | l_u | l_uu(diag)]; at the terminal knot only l_x and l_xx are written.
#pragma once
#include "common.cuh"
#include "systems.cuh"

namespace cacto {

// ------------------------------------------------------------------------------------------ hyper-dual numbers
template <typename T>
struct HDual {
  T v, a, b, ab;
  __device__ __forceinline__ HDual() {}
  __device__ __forceinline__ HDual(T x) : v(x), a(T(0)), b(T(0)), ab(T(0)) {}
  __device__ __forceinline__ HDual(T x, T da, T db, T dab) : v(x), a(da), b(db), ab(dab) {}
};
template <typename T> struct scalar_of<HDual<T>> { typedef T type; };
template <typename T> __device__ __forceinline__ HDual<T> operator+(HDual<T> x, HDual<T> y) { return HDual<T>(x.v + y.v, x.a + y.a, x.b + y.b, x.ab + y.ab); }
template <typename T> __device__ __forceinline__ HDual<T> operator-(HDual<T> x, HDual<T> y) { return HDual<T>(x.v - y.v, x.a - y.a, x.b - y.b, x.ab - y.ab); }
template <typename T> __device__ __forceinline__ HDual<T> operator-(HDual<T> x) { return HDual<T>(-x.v, -x.a, -x.b, -x.ab); }
template <typename T> __device__ __forceinline__ HDual<T> operator*(HDual<T> x, HDual<T> y) {
  return HDual<T>(x.v * y.v, x.v * y.a + x.a * y.v, x.v * y.b + x.b * y.v, x.v * y.ab + x.a * y.b + x.b * y.a + x.ab * y.v);
}
template <typename T> __device__ __forceinline__ HDual<T>& operator+=(HDual<T>& x, HDual<T> y) { x = x + y; return x; }
// f(x) with f0 = f(x.v), f1 = f'(x.v), f2 = f''(x.v)
template <typename T> __device__ __forceinline__ HDual<T> hd_chain(HDual<T> x, T f0, T f1, T f2) {
  return HDual<T>(f0, f1 * x.a, f1 * x.b, f1 * x.ab + f2 * x.a * x.b);
}
template <typename T> __device__ __forceinline__ HDual<T> operator/(HDual<T> x, HDual<T> y) {
  const T r = T(1) / y.v;
  return x * hd_chain(y, r, -r * r, T(2) * r * r * r);
}
template <typename T> __device__ __forceinline__ bool operator>(HDual<T> x, HDual<T> y) { return x.v > y.v; }
template <typename T> __device__ __forceinline__ HDual<T> sqrt_(HDual<T> x) {
  const T s = sqrt_(x.v);
  return hd_chain(x, s, T(0.5) / s, T(-0.25) / (s * x.v));
}
template <typename T> __device__ __forceinline__ HDual<T> exp_(HDual<T> x) {
  const T e = exp_(x.v);
  return hd_chain(x, e, e, e);
}
template <typename T> __device__ __forceinline__ HDual<T> log_(HDual<T> x) {
  const T r = T(1) / x.v;
  return hd_chain(x, log_(x.v), r, -r * r);
}
template <typename T> __device__ __forceinline__ void sincos_from(HDual<T> x, T sv, T cv, HDual<T>& s, HDual<T>& c) {
  s = hd_chain(x, sv, cv, -sv);
  c = hd_chain(x, cv, -sv, -cv);
}
template <typename T> __device__ __forceinline__ void sincos_(HDual<T> x, HDual<T>& s, HDual<T>& c) {
  T sv, cv;
  sincos_(x.v, sv, cv);
  s = hd_chain(x, sv, cv, -sv);
  c = hd_chain(x, cv, -sv, -cv);
}

__host__ __device__ constexpr int bp_stride(int nx, int na) { return nx + 2 * nx * nx + nx * na + 2 * na; }

// ------------------------------------------------------------------------------------------ one knot
// x[NX] (no time column), u[NA] (ignored at the terminal knot, last = true) -> the knot's block o[bp_stride(NX, NA)].
template <int SYS>
__device__ __forceinline__ void bp_knot_eval(const cacto_sys_params& P, const double* __restrict__ xk, const double* __restrict__ uk, bool last,
                                             double* __restrict__ o) {
  constexpr int NX = SysDims<SYS>::NX, NA = SysDims<SYS>::NA;
  double x[NX + 1], u[NA];
#pragma unroll
  for (int i = 0; i < NX; ++i) x[i] = xk[i];
  x[NX] = 0.0;
#pragma unroll
  for (int i = 0; i < NA; ++i) u[i] = last ? 0.0 : uk[i];
  double* lx = o, *lxx = o + NX, *A = lxx + NX * NX, *Bm = A + NX * NX, *lu = Bm + NX * NA, *luu = lu + NA;
  const double* w = last ? P.w_terminal : P.w_running;
  // l_x, l_xx: one hyper-dual evaluation of the reward per pair (i <= j); the UR5's joint sin / cos once per knot, not per pair
  double sc_real[12];
  if constexpr (SYS == CACTO_UR5) ur5_sincos<double>(x, sc_real);
  for (int i = 0; i < NX; ++i) {
    for (int j = i; j < NX; ++j) {
      HDual<double> xs[NX + 1];
#pragma unroll
      for (int c = 0; c <= NX; ++c) xs[c] = HDual<double>(x[c], c == i ? 1.0 : 0.0, c == j ? 1.0 : 0.0, 0.0);
      const HDual<double> r = sys_reward<SYS, HDual<double>>(P, w, xs, (const HDual<double>*)nullptr, false, SYS == CACTO_UR5 ? sc_real : nullptr);
      lxx[i * NX + j] = r.ab;
      lxx[j * NX + i] = r.ab;
      if (j == i) lx[i] = r.a;
    }
  }
  if (!last) {
    double Fx[NX * NX], Fu[NX * NA];
    sys_jac<SYS, double>(P, x, u, Fx, Fu);
    for (int c = 0; c < NX * NX; ++c) A[c] = Fx[c];
    for (int c = 0; c < NX * NA; ++c) Bm[c] = Fu[c];
    // control part of the reward: -scale w6 sum(a^2 + w_b (a / u_max)^10)   (environment_TO.py bound_control_cost)
    for (int i = 0; i < NA; ++i) {
      const double um = P.u_max[i], r = u[i] / um;
      const double r2 = r * r, r4 = r2 * r2, r8 = r4 * r4;
      lu[i] = -P.scale * w[6] * (2.0 * u[i] + 10.0 * P.w_b * (r8 * r) / um);
      luu[i] = -P.scale * w[6] * (2.0 + 90.0 * P.w_b * r8 / (um * um));
    }
  }
}

// trajectory of knot k: binary search in offsets (E + 1 entries)
__device__ __forceinline__ int knot_owner(const int64_t* __restrict__ offsets, int E, int64_t k) {
  int lo = 0, hi = E;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (offsets[mid] <= k) lo = mid; else hi = mid;
  }
  return lo;
}

}  // namespace cacto
