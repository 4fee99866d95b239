// mlp_generic.cu -- NN.eval / compute_critic_grad / compute_actor_grad for critics of ANY of the reference's shapes.
//
// The fused update kernels of update.cu are specialised on the critic of every conf ('sine': ns-64-64-128-128-1, SIREN).
// NeuralNetwork.py also defines 'elu' (:65-78: ns-16-32-256-256-1, elu), 'sine-elu' (:80-93: 64 sin, 64 elu, 128 sin, 128 elu)
// and 'relu' (:110-128: 16-32-NH1-NH2-1, LeakyReLU 0.3).  These kernels cover them with a layer table instead of template
// shapes: ONE CTA PER SAMPLE, activations of all sweeps in shared memory, weights read straight from L2 (coalesced for
// h W products, warp-cooperative row dot products for W g products, so no transposed copy is needed), weight gradients
// accumulated with one fp32 atomic per weight and sample.  They are the latency-oriented / generic path; the tiled kernels
// remain the path of the default critic.
//
// Sobolev critic step per sample (SURVEY.md A.3; f_l activation of layer l, z_l pre-activations, h_l = f_l(z_l)):
//   F   z_l = h_{l-1} W_l + b_l,  V = z_L
//   G   g_L = 1,  q_{l-1} = W_l g_l,  g_{l-1} = q_{l-1} * f'_{l-1}(z_{l-1}),  dV/ds_j = scale_j q_0[j]
//   A   a_0 = scale * dL/d(dV/ds),  u_l = a_{l-1} W_l,  a_l = u_l * f'_l(z_l),  e_l = u_l * q_l * f''_l(z_l)
//   B   d_L = dL/dV,  d_{l-1} = (W_l d_l) * f'_{l-1}(z_{l-1}) + e_{l-1}
//   dW_l = h_{l-1} (x) d_l + a_{l-1} (x) g_l,  db_l = d_l
#include "common.cuh"
#include "mlp.cuh"
#include "systems.cuh"

namespace cacto {

constexpr int GEN_NT = 256;          // threads per CTA (= max layer width)
constexpr int GEN_MAXW = 256;        // max units per layer
constexpr int GEN_MAXL = CACTO_MLP_MAX_LAYERS;
constexpr int GEN_TOT = 1280;        // max total units of a network incl. its input (floats per activation array)
constexpr int GEN_MAXW_A = CACTO_ACTOR_MAX_WIDTH;              // max units per layer of the actor in the actor step
constexpr int GEN_TOT_A = CACTO_MAX_NS + 2 * GEN_MAXW_A + CACTO_MAX_NA;   // ... and its max total units

__device__ __forceinline__ float gen_slog(float x) { return x > 0.f ? logf(fmaxf(x, 1e-7f) + 1.f) : -logf(fmaxf(-x, 1e-7f) + 1.f); }
__device__ __forceinline__ float gen_slog_grad(float x) { return fabsf(x) >= 1e-7f ? 1.f / (fabsf(x) + 1.f) : 0.f; }

// activation codes of cacto_mlp_desc: value, first and second derivative at pre-activation z
__device__ __forceinline__ void gen_act(int code, float z, float& f, float& f1, float& f2) {
  if (code == CACTO_ACT_SIN) {
    float s, c;
    sincosf(z, &s, &c);
    f = s; f1 = c; f2 = -s;
  } else if (code == CACTO_ACT_ELU) {
    const float e = expf(z);
    f = z > 0.f ? z : e - 1.f; f1 = z > 0.f ? 1.f : e; f2 = z > 0.f ? 0.f : e;
  } else if (code == CACTO_ACT_LEAKY) {
    f = z > 0.f ? z : LEAKY_ALPHA * z; f1 = z > 0.f ? 1.f : LEAKY_ALPHA; f2 = 0.f;
  } else {
    f = z; f1 = 1.f; f2 = 0.f;
  }
}

struct GenNet {
  int L;                           // weight layers
  int dim[GEN_MAXL + 1];
  int act[GEN_MAXL];               // activation after layer l (0-based), last one linear
  int W[GEN_MAXL], b[GEN_MAXL];    // parameter offsets (Keras order)
  int off[GEN_MAXL + 1];           // offset of layer l's units inside the concatenated activation arrays (off[0] = input)
  int width;                       // total units incl. input
};
__device__ __forceinline__ GenNet gen_net(const cacto_mlp_desc& d) {
  GenNet n;
  n.L = d.n_layers;
  int o = 0, u = 0;
  for (int l = 0; l <= n.L; ++l) {
    n.dim[l] = d.dims[l];
    n.off[l] = u;
    u += d.dims[l];
  }
  n.width = u;
  for (int l = 0; l < n.L; ++l) {
    n.act[l] = d.act[l];
    n.W[l] = o; o += d.dims[l] * d.dims[l + 1];
    n.b[l] = o; o += d.dims[l + 1];
  }
  return n;
}

// out[j] = sum_i in[i] W[i][j] (+ bias[j]) for j < nout: thread per output unit, coalesced weight reads.
__device__ __forceinline__ void gen_fwd(const float* __restrict__ W, const float* __restrict__ bias, const float* in, int nin, int nout,
                                        float* out) {
  for (int j = threadIdx.x; j < nout; j += GEN_NT) {
    float acc = bias != nullptr ? bias[j] : 0.f;
    for (int i = 0; i < nin; ++i) acc = fmaf(in[i], W[(size_t)i * nout + j], acc);
    out[j] = acc;
  }
}
// out[i] = sum_j W[i][j] in[j] for i < nin: one warp per row, lanes stride the row (coalesced), shuffle reduction.
__device__ __forceinline__ void gen_bwd(const float* __restrict__ W, const float* in, int nin, int nout, float* out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = warp; i < nin; i += GEN_NT / 32) {
    float acc = 0.f;
    for (int j = lane; j < nout; j += 32) acc = fmaf(W[(size_t)i * nout + j], in[j], acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) out[i] = acc;
  }
}

// F sweep: Z (pre-activations), H (activations; H[off[0]..] = input), optionally F1 / F2 (f', f'').  Ends synchronised.
__device__ __forceinline__ void gen_forward(const GenNet& n, const float* __restrict__ p, float* Z, float* H, float* F1, float* F2) {
  for (int l = 0; l < n.L; ++l) {
    gen_fwd(p + n.W[l], p + n.b[l], H + n.off[l], n.dim[l], n.dim[l + 1], Z + n.off[l + 1]);
    __syncthreads();
    for (int j = threadIdx.x; j < n.dim[l + 1]; j += GEN_NT) {
      float f, f1, f2;
      gen_act(n.act[l], Z[n.off[l + 1] + j], f, f1, f2);
      H[n.off[l + 1] + j] = f;
      if (F1 != nullptr) F1[n.off[l + 1] + j] = f1;
      if (F2 != nullptr) F2[n.off[l + 1] + j] = f2;
    }
    __syncthreads();
  }
}
// G sweep from the scalar output (dim[L] == 1): Q[off[l]..] = dV/dh_l, G[off[l]..] = dV/dz_l.  Ends synchronised.
__device__ __forceinline__ void gen_input_grad(const GenNet& n, const float* __restrict__ p, const float* F1, float* Q, float* G) {
  if (threadIdx.x == 0) G[n.off[n.L]] = 1.f;
  __syncthreads();
  for (int l = n.L - 1; l >= 0; --l) {
    gen_bwd(p + n.W[l], G + n.off[l + 1], n.dim[l], n.dim[l + 1], Q + n.off[l]);
    __syncthreads();
    if (l > 0) {
      for (int j = threadIdx.x; j < n.dim[l]; j += GEN_NT) G[n.off[l] + j] = Q[n.off[l] + j] * F1[n.off[l] + j];
      __syncthreads();
    }
  }
}

// ------------------------------------------------------------------------------------------ NN.eval
struct GenEvalSmem {
  float Z[GEN_TOT], H[GEN_TOT], F1[GEN_TOT], Q[GEN_TOT], G[GEN_TOT];
};

__global__ void __launch_bounds__(GEN_NT) k_mlp_eval_gen(const __grid_constant__ cacto_sys_params P, const __grid_constant__ cacto_mlp_desc D,
                                                         const float* __restrict__ params, const float* __restrict__ state,
                                                         float* __restrict__ out, float* __restrict__ dout_ds, int64_t B) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GenEvalSmem& sm = *reinterpret_cast<GenEvalSmem*>(smem_raw);
  const GenNet n = gen_net(D);
  const int64_t b = blockIdx.x;
  const int ns = n.dim[0];
  for (int j = threadIdx.x; j < ns; j += GEN_NT) sm.H[j] = normalize_component(P, j, state[b * ns + j]);
  __syncthreads();
  gen_forward(n, params, sm.Z, sm.H, dout_ds != nullptr ? sm.F1 : nullptr, nullptr);
  const int no = n.dim[n.L];
  for (int j = threadIdx.x; j < no; j += GEN_NT) out[b * no + j] = sm.Z[n.off[n.L] + j];
  if (dout_ds != nullptr) {                        // dV/ds w.r.t. the RAW state (scalar output only)
    gen_input_grad(n, params, sm.F1, sm.Q, sm.G);
    for (int j = threadIdx.x; j < ns; j += GEN_NT) dout_ds[b * ns + j] = sm.Q[j] * normalize_scale(P, j);
  }
}

// ------------------------------------------------------------------------------------------ Sobolev critic step
struct GenCriticSmem {
  float Z[GEN_TOT], H[GEN_TOT], F1[GEN_TOT], F2[GEN_TOT];
  float Q[GEN_TOT], G[GEN_TOT], A[GEN_TOT], U[GEN_TOT];
  float E[GEN_TOT], DL[GEN_TOT], T[GEN_TOT];
  float red[GEN_NT / 32];
};

__global__ void __launch_bounds__(GEN_NT) k_critic_grad_gen(const __grid_constant__ cacto_sys_params P, const __grid_constant__ cacto_mlp_desc D,
                                                            const float* __restrict__ cw, const float* __restrict__ tw, float w_S, int mc,
                                                            const float* __restrict__ state, const float* __restrict__ state_next,
                                                            const float* __restrict__ prtg, const float* __restrict__ dVdx,
                                                            const float* __restrict__ done, const float* __restrict__ weights, float inv_B,
                                                            float* __restrict__ grad, float* __restrict__ rtg_out, float* __restrict__ V_out,
                                                            float* __restrict__ Vt_out, float* __restrict__ loss_out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  GenCriticSmem& sm = *reinterpret_cast<GenCriticSmem*>(smem_raw);
  const GenNet n = gen_net(D);
  const int64_t b = blockIdx.x;
  const int ns = n.dim[0], nx = ns - 1, tid = threadIdx.x;
  const bool sobolev = (w_S != 0.f);
  // ---- target critic: V_target(s_next) for the TD target (NeuralNetwork.py:154-159), V_target(s) for the caller (:177)
  float vt_next = 0.f;
  if (!mc) {
    for (int j = tid; j < ns; j += GEN_NT) sm.H[j] = normalize_component(P, j, state_next[b * ns + j]);
    __syncthreads();
    gen_forward(n, tw, sm.T, sm.H, nullptr, nullptr);
    vt_next = sm.T[n.off[n.L]];
    __syncthreads();
  }
  for (int j = tid; j < ns; j += GEN_NT) sm.H[j] = normalize_component(P, j, state[b * ns + j]);
  __syncthreads();
  gen_forward(n, tw, sm.T, sm.H, nullptr, nullptr);
  const float vt_s = sm.T[n.off[n.L]];
  __syncthreads();
  // ---- F (and G) of the critic
  gen_forward(n, cw, sm.Z, sm.H, sm.F1, sm.F2);
  const float V = sm.Z[n.off[n.L]];
  const float rtg = mc ? prtg[b] : prtg[b] + (1.f - done[b]) * vt_next;
  const float wi = weights[b];
  if (tid == 0) {
    rtg_out[b] = rtg;
    V_out[b] = V;
    Vt_out[b] = vt_s;
  }
  float loss = 0.f;
  for (int j = tid; j < n.width; j += GEN_NT) sm.E[j] = 0.f;
  if (sobolev) {
    gen_input_grad(n, cw, sm.F1, sm.Q, sm.G);
    // ---- loss seeds (NeuralNetwork.py:166-170): a_0 = scale * dL/d(dV/ds)
    for (int j = tid; j < ns; j += GEN_NT) {
      float a0 = 0.f;
      if (j < nx) {
        const float sc = normalize_scale(P, j);
        const float p = sm.Q[j] * sc;
        const float diff = gen_slog(p) - gen_slog(dVdx[b * ns + j]);
        loss += wi * diff * diff / (float)nx;
        a0 = sc * wi * inv_B * (2.f / (float)nx) * diff * gen_slog_grad(p);
      }
      sm.A[j] = a0;
    }
    __syncthreads();
    // ---- A sweep
    for (int l = 0; l < n.L; ++l) {
      gen_fwd(cw + n.W[l], nullptr, sm.A + n.off[l], n.dim[l], n.dim[l + 1], sm.U + n.off[l + 1]);
      __syncthreads();
      if (l + 1 < n.L) {
        for (int j = tid; j < n.dim[l + 1]; j += GEN_NT) {
          const int k = n.off[l + 1] + j;
          sm.A[k] = sm.U[k] * sm.F1[k];
          sm.E[k] = sm.U[k] * sm.Q[k] * sm.F2[k];
        }
        __syncthreads();
      }
    }
  }
  // ---- B sweep
  const float dv = V - rtg;
  const float seed = (sobolev ? w_S : 1.f) * wi * inv_B * 2.f * dv;
  if (tid == 0) {
    sm.DL[n.off[n.L]] = seed;
    loss += (sobolev ? w_S : 1.f) * wi * dv * dv;
  }
  __syncthreads();
  for (int l = n.L - 1; l >= 1; --l) {
    gen_bwd(cw + n.W[l], sm.DL + n.off[l + 1], n.dim[l], n.dim[l + 1], sm.T + n.off[l]);
    __syncthreads();
    for (int j = tid; j < n.dim[l]; j += GEN_NT) {
      const int k = n.off[l] + j;
      sm.DL[k] = sm.T[k] * sm.F1[k] + sm.E[k];
    }
    __syncthreads();
  }
  // ---- weight gradients: one atomic per weight
  for (int l = 0; l < n.L; ++l) {
    const int nin = n.dim[l], nout = n.dim[l + 1];
    const float* h = sm.H + n.off[l];
    const float* a = sm.A + n.off[l];
    const float* d = sm.DL + n.off[l + 1];
    const float* g = sm.G + n.off[l + 1];
    for (int e = tid; e < nin * nout; e += GEN_NT) {
      const int i = e / nout, j = e - i * nout;
      float v = h[i] * d[j];
      if (sobolev) v = fmaf(a[i], g[j], v);
      atomicAdd(grad + n.W[l] + e, v);
    }
    for (int j = tid; j < nout; j += GEN_NT) atomicAdd(grad + n.b[l] + j, d[j]);
  }
  // ---- loss (sum over the CTA, then one atomic)
  if (loss_out != nullptr) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) loss += __shfl_xor_sync(0xffffffffu, loss, o);
    if ((tid & 31) == 0) sm.red[tid >> 5] = loss;
    __syncthreads();
    if (tid == 0) {
      float s = 0.f;
      for (int w = 0; w < GEN_NT / 32; ++w) s += sm.red[w];
      atomicAdd(loss_out, s * inv_B);
    }
  }
}

// ------------------------------------------------------------------------------------------ actor step
// The per-sample environment terms (s' = Env.simulate_batch, Fu = Env.derivative_batch, dr/da) come from the batched kernels
// the reference-facing API already has (cacto_dyn_step / cacto_dyn_derivative / cacto_reward); this kernel does the network part.
// Shared memory: five activation arrays of the actor (tot_a floats each) and five of the critic (tot_c each), sized at launch
// from the two descriptors (gen_actor_smem_floats).
__host__ __device__ __forceinline__ int gen_units(const cacto_mlp_desc& d) {
  int u = 0;
  for (int l = 0; l <= d.n_layers; ++l) u += d.dims[l];
  return (u + 3) & ~3;
}
__host__ __device__ __forceinline__ int gen_actor_smem_floats(const cacto_mlp_desc& da, const cacto_mlp_desc& dc) {
  return 5 * gen_units(da) + 5 * gen_units(dc);
}

__global__ void __launch_bounds__(GEN_NT) k_actor_grad_gen(const __grid_constant__ cacto_sys_params P, const __grid_constant__ cacto_mlp_desc DA,
                                                           const float* __restrict__ aw, const __grid_constant__ cacto_mlp_desc DC,
                                                           const float* __restrict__ cw, const float* __restrict__ state,
                                                           const float* __restrict__ state_next, const float* __restrict__ Fu,
                                                           const float* __restrict__ dr_da, float inv_B, float* __restrict__ grad) {
  extern __shared__ __align__(16) float gen_smem[];
  struct {
    float *Za, *Ha, *F1a, *DLa, *Ta, *Z, *H, *F1, *Q, *G;
  } sm;
  {
    const int ta = gen_units(DA), tc = gen_units(DC);
    sm.Za = gen_smem; sm.Ha = sm.Za + ta; sm.F1a = sm.Ha + ta; sm.DLa = sm.F1a + ta; sm.Ta = sm.DLa + ta;
    sm.Z = sm.Ta + ta; sm.H = sm.Z + tc; sm.F1 = sm.H + tc; sm.Q = sm.F1 + tc; sm.G = sm.Q + tc;
  }
  const GenNet na_ = gen_net(DA), nc = gen_net(DC);
  const int64_t b = blockIdx.x;
  const int tid = threadIdx.x, ns = na_.dim[0], na = na_.dim[na_.L];
  // ---- actor forward (NeuralNetwork.py:185), critic forward + input gradient at s' (:190-195)
  for (int j = tid; j < ns; j += GEN_NT) {
    sm.Ha[j] = normalize_component(P, j, state[b * ns + j]);
    sm.H[j] = normalize_component(P, j, state_next[b * ns + j]);
  }
  __syncthreads();
  gen_forward(na_, aw, sm.Za, sm.Ha, sm.F1a, nullptr);
  gen_forward(nc, cw, sm.Z, sm.H, sm.F1, nullptr);
  gen_input_grad(nc, cw, sm.F1, sm.Q, sm.G);
  // ---- dQ/da = dV/ds' Fu + dr/da; upstream gradient of mean(-dQ/da . a)  (NeuralNetwork.py:206-231)
  if (tid < na) {
    float dq = dr_da[b * na + tid];
    for (int i = 0; i < ns; ++i) dq = fmaf(sm.Q[i] * normalize_scale(P, i), Fu[(b * ns + i) * na + tid], dq);
    sm.DLa[na_.off[na_.L] + tid] = -dq * inv_B;
  }
  __syncthreads();
  // ---- actor backward
  for (int l = na_.L - 1; l >= 1; --l) {
    gen_bwd(aw + na_.W[l], sm.DLa + na_.off[l + 1], na_.dim[l], na_.dim[l + 1], sm.Ta + na_.off[l]);
    __syncthreads();
    for (int j = tid; j < na_.dim[l]; j += GEN_NT) {
      const int k = na_.off[l] + j;
      sm.DLa[k] = sm.Ta[k] * sm.F1a[k];
    }
    __syncthreads();
  }
  for (int l = 0; l < na_.L; ++l) {
    const int nin = na_.dim[l], nout = na_.dim[l + 1];
    const float* h = sm.Ha + na_.off[l];
    const float* d = sm.DLa + na_.off[l + 1];
    for (int e = tid; e < nin * nout; e += GEN_NT) {
      const int i = e / nout, j = e - i * nout;
      atomicAdd(grad + na_.W[l] + e, h[i] * d[j]);
    }
    for (int j = tid; j < nout; j += GEN_NT) atomicAdd(grad + na_.b[l] + j, d[j]);
  }
}

static int gen_check_desc(const cacto_mlp_desc* d, int ns, int out_dim, int max_total = GEN_TOT, int max_width = GEN_MAXW) {
  if (!d) return CACTO_E_ARG;
  if (d->n_layers < 1 || d->n_layers > GEN_MAXL) return CACTO_E_SIZE;
  if (d->dims[0] != ns || (out_dim > 0 && d->dims[d->n_layers] != out_dim)) return CACTO_E_SIZE;
  int total = 0;
  for (int l = 0; l <= d->n_layers; ++l) {
    if (d->dims[l] < 1 || d->dims[l] > max_width) return CACTO_E_SIZE;
    total += d->dims[l];
  }
  if (total > max_total) return CACTO_E_SIZE;
  for (int l = 0; l < d->n_layers; ++l)
    if (d->act[l] < 0 || d->act[l] > CACTO_ACT_LEAKY) return CACTO_E_ARG;
  return 0;
}
template <typename K>
static int gen_smem(K k, size_t bytes) {
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  return e == cudaSuccess ? 0 : (int)e;
}

}  // namespace cacto

using namespace cacto;

extern "C" int cacto_mlp_forward_generic(const cacto_sys_params* p, const cacto_mlp_desc* d, const float* params, const float* state, float* out,
                                         float* dout_ds, int64_t B, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (int e = gen_check_desc(d, p->ns, 0)) return e;
  if (B < 0 || B > 0x7fffffff) return CACTO_E_SIZE;
  if (B == 0) return 0;
  if (!params || !state || !out) return CACTO_E_ARG;
  if (dout_ds != nullptr && d->dims[d->n_layers] != 1) return CACTO_E_SIZE;
  if (int e = gen_smem(k_mlp_eval_gen, sizeof(GenEvalSmem))) return e;
  k_mlp_eval_gen<<<(unsigned)B, GEN_NT, sizeof(GenEvalSmem), (cudaStream_t)stream>>>(*p, *d, params, state, out, dout_ds, B);
  CACTO_LAUNCH_CHECK();
  return 0;
}

extern "C" int cacto_critic_grad_generic(const cacto_sys_params* p, const cacto_mlp_desc* d, const float* critic_params, const float* target_params,
                                         float w_S, int mc, const float* state, const float* state_next, const float* partial_rtg,
                                         const float* dVdx, const float* done, const float* weights, float inv_B, float* grad, float* rtg,
                                         float* V, float* V_target_s, float* loss, int64_t B, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (int e = gen_check_desc(d, p->ns, 1)) return e;
  if (B < 0 || B > 0x7fffffff) return CACTO_E_SIZE;
  if (B == 0) return 0;
  if (!critic_params || !target_params || !state || !partial_rtg || !weights || !grad || !rtg || !V || !V_target_s) return CACTO_E_ARG;
  if (!mc && (!state_next || !done)) return CACTO_E_ARG;
  if (w_S != 0.f && !dVdx) return CACTO_E_ARG;
  if (int e = gen_smem(k_critic_grad_gen, sizeof(GenCriticSmem))) return e;
  k_critic_grad_gen<<<(unsigned)B, GEN_NT, sizeof(GenCriticSmem), (cudaStream_t)stream>>>(*p, *d, critic_params, target_params, w_S, mc, state,
                                                                                           state_next, partial_rtg, dVdx, done, weights, inv_B,
                                                                                           grad, rtg, V, V_target_s, loss);
  CACTO_LAUNCH_CHECK();
  return 0;
}

extern "C" int cacto_actor_grad_generic(const cacto_sys_params* p, const cacto_mlp_desc* d_actor, const float* actor_params,
                                        const cacto_mlp_desc* d_critic, const float* critic_params, const float* state,
                                        const float* state_next, const float* Fu, const float* dr_da, float inv_B, float* grad, int64_t B,
                                        void* stream) {
  if (!p) return CACTO_E_ARG;
  if (int e = gen_check_desc(d_actor, p->ns, p->na, GEN_TOT_A, GEN_MAXW_A)) return e;
  if (int e = gen_check_desc(d_critic, p->ns, 1)) return e;
  if (B < 0 || B > 0x7fffffff) return CACTO_E_SIZE;
  if (B == 0) return 0;
  if (!actor_params || !critic_params || !state || !state_next || !Fu || !dr_da || !grad) return CACTO_E_ARG;
  const size_t smem = 4u * (size_t)gen_actor_smem_floats(*d_actor, *d_critic);
  if (int e = gen_smem(k_actor_grad_gen, smem)) return e;
  k_actor_grad_gen<<<(unsigned)B, GEN_NT, smem, (cudaStream_t)stream>>>(*p, *d_actor, actor_params, *d_critic, critic_params, state,
                                                                                         state_next, Fu, dr_da, inv_B, grad);
  CACTO_LAUNCH_CHECK();
  return 0;
}
