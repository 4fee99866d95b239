// update.cu -- K3: the Sobolev critic / actor update of RL_AC.update (RL.py:101-118):
//   k_critic_grad   NN.compute_critic_grad (NeuralNetwork.py:150-178): TD(n) target from the target
//                   critic, forward F, input-gradient sweep G, Sobolev loss with the signed-log, adjoint
//                   sweep A through G (the second-order part) and backward sweep B, all for one tile of
//                   samples without leaving shared memory (SURVEY.md A.3);
//   k_actor_grad    NN.compute_actor_grad (NeuralNetwork.py:180-232): actor forward, Env.simulate_batch,
//                   Env.derivative_batch and d reward_batch/da per sample, critic F+G at s', dQ/da, actor
//                   backward (SURVEY.md A.4);
//   k_adam          tf.keras.optimizers.Adam step (TF 2.11: eps outside the bias correction) fused with the
//                   Polyak target update (RL.py:113-118), the refresh of the transposed weight copy used
//                   by the backward sweeps, and the zeroing of the gradient buffer;
//   k_*_forward     NN.eval for batches (NeuralNetwork.py:130-138).
// Weight gradients are accumulated with fp32 atomics into one buffer per network (what the NCCL
// all-reduce of the data-parallel path sums across GPUs).
#include "common.cuh"
#include "det.cuh"
#include "mlp.cuh"
#include "systems.cuh"

namespace cacto {

constexpr int UP_NT = 256;
constexpr int NSP = 16;   // padded state width in shared memory
constexpr int NAP = 8;    // padded action width
constexpr int CW = CR_H1 + CR_H2 + CR_H3 + CR_H4;   // 384 hidden units of the critic
// column offset of hidden layer l inside the [S][CW] activation arrays
__host__ __device__ __forceinline__ constexpr int koff(int l) { return l == 0 ? 0 : (l == 1 ? CR_H1 : (l == 2 ? CR_H1 + CR_H2 : CR_H1 + CR_H2 + CR_H3)); }

// custom_logarithm (NeuralNetwork.py:140-148) and its TensorFlow gradient (quirk Q10).
__device__ __forceinline__ float slog(float x) { return x > 0.f ? logf(fmaxf(x, 1e-7f) + 1.f) : -logf(fmaxf(-x, 1e-7f) + 1.f); }
__device__ __forceinline__ float slog_grad(float x) { return fabsf(x) >= 1e-7f ? 1.f / (fabsf(x) + 1.f) : 0.f; }

// sin / cos of the SIREN layers, deliberately NOT inlined: the accurate sinf / sincosf expand to ~40 instructions per call and
// sat in ~100 epilogue call sites -- a third of the 13 k instructions of k_critic_grad, whose small-batch runs are bound by
// instruction fetch (ncu: stall_no_inst 35 % of the samples at B = 64), every CTA walking the code once.
__device__ __noinline__ float sin_call(float x) { return sinf(x); }
__device__ __noinline__ float2 sincos_call(float x) {
  float2 r;
  sincosf(x, &r.x, &r.y);
  return r;
}
__device__ __forceinline__ float4 sin4(float4 a, float4 b) {
  return make_float4(sin_call(a.x + b.x), sin_call(a.y + b.y), sin_call(a.z + b.z), sin_call(a.w + b.w));
}
__device__ __forceinline__ void sincos4(float4 a, float4 b, float4& s, float4& c) {
  const float2 x = sincos_call(a.x + b.x), y = sincos_call(a.y + b.y), z = sincos_call(a.z + b.z), w = sincos_call(a.w + b.w);
  s = make_float4(x.x, y.x, z.x, w.x);
  c = make_float4(x.y, y.y, z.y, w.y);
}

// Order in which the streamed (K % 4 == 0) weight matrices are consumed by a kernel; built by every
// thread identically, read when a GEMM asks the pipeline to prefetch its successor.
struct WeightSeq {
  const float* ptr[24];
  int first[24];      // floats of the first chunk
  int n;
};
template <int N>
__device__ __forceinline__ void seq_push(WeightSeq& q, const float* p, int K) {
  q.ptr[q.n] = p;
  q.first[q.n] = chunk_rows<N>(K) * N;
  ++q.n;
}

// Load `rows` rows of a [B][ns] float state block, normalise (utils.py:17-24) and zero-pad to [S][NSP].
template <int S>
__device__ __forceinline__ void load_normalised(const cacto_sys_params& P, const float* __restrict__ g, int64_t row0, int rows,
                                                float (*X)[NSP]) {
  const int ns = P.ns;
  for (int i = threadIdx.x; i < S * NSP; i += UP_NT) {
    const int s = i / NSP, j = i - s * NSP;
    float v = 0.f;
    if (s < rows && j < ns) v = normalize_component(P, j, g[(row0 + s) * ns + j]);
    X[s][j] = v;
  }
}

// Streamed GEMM number `gi` of the kernel's weight sequence (prefetches the first chunk of number gi + 1).
template <int S, int N, typename SM, typename Epi>
__device__ __forceinline__ void streamed(WeightPipe& pipe, SM& sm, int& gi, const float* A, int lda, int K, Epi&& epi) {
  const bool more = gi + 1 < sm.seq.n;
  gemm_streamed<S, N, UP_NT>(pipe, A, lda, K, sm.seq.ptr[gi], more ? sm.seq.ptr[gi + 1] : nullptr, more ? sm.seq.first[gi + 1] : 0, epi);
  ++gi;
}
// the three streamed layers of a critic forward (weights w) / of a sweep with the transposed weights (wT)
__device__ __forceinline__ void seq_push_critic_fwd(WeightSeq& q, const CriticLayout& L, const float* w) {
  seq_push<CR_H2>(q, w + L.W[1], CR_H1);
  seq_push<CR_H3>(q, w + L.W[2], CR_H2);
  seq_push<CR_H4>(q, w + L.W[3], CR_H3);
}
__device__ __forceinline__ void seq_push_critic_bwd(WeightSeq& q, const CriticLayout& L, const float* wT) {
  seq_push<CR_H3>(q, wT + L.W[3], CR_H4);
  seq_push<CR_H2>(q, wT + L.W[2], CR_H3);
  seq_push<CR_H1>(q, wT + L.W[1], CR_H2);
}

// Small parameters of a critic (first layer, all biases, output weights) copied once per kernel into shared memory:
// they are touched by every phase of the sweeps, and an L2 round trip per phase is what a latency-bound kernel cannot hide.
struct CriticSmall {
  alignas(16) float W1[CACTO_MAX_NS * CR_H1];
  alignas(16) float b[CW + 4];          // hidden biases at koff(l), output bias at CW
  alignas(16) float w5[CR_H4];
};
struct CriticPtrs {
  const float* W0;
  const float* b[5];
  const float* W4;
};
// The small-parameter blocks are contiguous pieces of the flat parameter vector (16-byte aligned, sizes multiples of 16 bytes):
// thread 0 queues them as TMA bulk copies on one mbarrier -- one L2 round trip for the whole prologue instead of a chain of
// dependent LDG -> STS loops (ncu at B = 64: 19 % of the actor kernel's stall samples sat in its first 400 instructions).
__device__ __forceinline__ void bulk_g2s(void* sdst, const float* __restrict__ gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(sdst)), "l"(gsrc),
               "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void small_bar_init(uint64_t* bar) {          // thread 0, before WeightPipe::init (which fences and syncs)
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)));
}
__device__ __forceinline__ void small_bar_expect(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void small_bar_wait(uint64_t* bar) {           // all threads; the barrier completes exactly once per kernel
  const uint32_t mb = smem_u32(bar);
  uint32_t done = 0;
  unsigned spins = 0;
  while (!done) {
    if (++spins > (1u << 24)) __trap();
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(mb), "r"(0u)
        : "memory");
  }
}
__host__ __device__ __forceinline__ uint32_t critic_small_bytes(const CriticLayout& L) { return 4u * (uint32_t)(L.ns * CR_H1 + CW + CR_H4); }
// thread 0 only (after small_bar_expect)
__device__ __forceinline__ void load_critic_small(CriticSmall& d, const float* __restrict__ w, const CriticLayout& L, uint64_t* bar) {
  bulk_g2s(d.W1, w + L.W[0], 4u * (uint32_t)(L.ns * CR_H1), bar);
  bulk_g2s(d.b + koff(0), w + L.b[0], 4u * CR_H1, bar);
  bulk_g2s(d.b + koff(1), w + L.b[1], 4u * CR_H2, bar);
  bulk_g2s(d.b + koff(2), w + L.b[2], 4u * CR_H3, bar);
  bulk_g2s(d.b + koff(3), w + L.b[3], 4u * CR_H4, bar);
  bulk_g2s(d.w5, w + L.W[4], 4u * CR_H4, bar);
  d.b[CW] = w[L.b[4]];
}
__device__ __forceinline__ CriticPtrs critic_ptrs(const CriticSmall& d) {
  CriticPtrs p;
  p.W0 = d.W1;
  for (int l = 0; l < 4; ++l) p.b[l] = d.b + koff(l);
  p.b[4] = d.b + CW;
  p.W4 = d.w5;
  return p;
}
struct ActorSmall {
  alignas(16) float W1[CACTO_MAX_NS * ACTOR_H];
  alignas(16) float b1[ACTOR_H];
  alignas(16) float b2[ACTOR_H];
  alignas(16) float W3[ACTOR_H * CACTO_MAX_NA];
  float b3[8];
};
__host__ __device__ __forceinline__ uint32_t actor_small_bytes(const ActorLayout& L) {
  return 4u * (uint32_t)(L.ns * ACTOR_H + 2 * ACTOR_H + ACTOR_H * L.na);
}
// thread 0 only (after small_bar_expect)
__device__ __forceinline__ void load_actor_small(ActorSmall& d, const float* __restrict__ w, const ActorLayout& L, uint64_t* bar) {
  bulk_g2s(d.W1, w + L.W1, 4u * (uint32_t)(L.ns * ACTOR_H), bar);
  bulk_g2s(d.b1, w + L.b1, 4u * ACTOR_H, bar);
  bulk_g2s(d.b2, w + L.b2, 4u * ACTOR_H, bar);
  bulk_g2s(d.W3, w + L.W3, 4u * (uint32_t)(ACTOR_H * L.na), bar);
  for (int j = 0; j < L.na; ++j) d.b3[j] = w[L.b3 + j];
}

// Forward pass of the sine critic for a tile, activations ping-ponging between two [S][ld] scratch
// buffers (>= 128 columns used).  V[s] receives the value.  Ends with a __syncthreads().
template <int S, typename SM>
__device__ __forceinline__ void critic_forward_tile(WeightPipe& pipe, SM& sm, int& gi, const CriticPtrs& cp, const CriticLayout& L,
                                                    const float (*XN)[NSP], float* bufA, float* bufB, int ld, float* V) {
  tile_gemm<S, CR_H1, UP_NT, false>(&XN[0][0], NSP, L.ns, cp.W0, CR_H1, [&](int r, int c, const float4& a) {
    const float4 b = *reinterpret_cast<const float4*>(cp.b[0] + c);
    *reinterpret_cast<float4*>(bufA + r * ld + c) = sin4(a, b);
  });
  __syncthreads();
  streamed<S, CR_H2>(pipe, sm, gi, bufA, ld, CR_H1, [&](int r, int c, const float4& a) {
    const float4 b = *reinterpret_cast<const float4*>(cp.b[1] + c);
    *reinterpret_cast<float4*>(bufB + r * ld + c) = sin4(a, b);
  });
  __syncthreads();
  streamed<S, CR_H3>(pipe, sm, gi, bufB, ld, CR_H2, [&](int r, int c, const float4& a) {
    const float4 b = *reinterpret_cast<const float4*>(cp.b[2] + c);
    *reinterpret_cast<float4*>(bufA + r * ld + c) = sin4(a, b);
  });
  __syncthreads();
  streamed<S, CR_H4>(pipe, sm, gi, bufA, ld, CR_H3, [&](int r, int c, const float4& a) {
    const float4 b = *reinterpret_cast<const float4*>(cp.b[3] + c);
    *reinterpret_cast<float4*>(bufB + r * ld + c) = sin4(a, b);
  });
  __syncthreads();
  tile_gemm_small<S, UP_NT, 8, true>(bufB, ld, CR_H4, cp.W4, 1, 0, [&](int s, int, float v) { V[s] = v + cp.b[4][0]; });
  __syncthreads();
}

// ------------------------------------------------------------------------------------------ critic
template <int S>
struct CriticSmem {
  alignas(128) float WB[2 * W_CHUNK];
  uint64_t bar[2], bar_small;
  WeightSeq seq;
  CriticSmall sc, st;                       // critic / target critic small parameters
  alignas(16) float X2[2 * S][NSP];         // rows [0, S): normalised state, rows [S, 2S): normalised next state
  float A0[S][NSP], G0[S][NSP];
  float SN[S][CW], CS[S][CW], G[S][CW], DL[S][CW], A[S][CW];
  float V[S], VT2[2 * S], Y[S], VBAR[S], WGT[S];
  float loss;
};

// DET: grad is the partials workspace (det.cuh); the CTA adds into its slice, the loss partial included.
template <int S, bool DET = false>
__global__ void __launch_bounds__(UP_NT) k_critic_grad(const __grid_constant__ cacto_sys_params P, const float* __restrict__ cw,
                                                       const float* __restrict__ cwT, const float* __restrict__ tw, float w_S, int mc,
                                                       const float* __restrict__ state, const float* __restrict__ state_next,
                                                       const float* __restrict__ prtg, const float* __restrict__ dVdx,
                                                       const float* __restrict__ done, const float* __restrict__ weights, float inv_B,
                                                       float* __restrict__ grad, float* __restrict__ rtg_out, float* __restrict__ V_out,
                                                       float* __restrict__ Vt_out, float* __restrict__ loss_out, int64_t B) {
  pdl_wait();
  extern __shared__ __align__(128) unsigned char smem_raw[];
  CriticSmem<S>& sm = *reinterpret_cast<CriticSmem<S>*>(smem_raw);
  const CriticLayout L(P.ns);
  if constexpr (DET) grad += (size_t)blockIdx.x * det_stride(L.total);
  const int ns = P.ns, nx = P.nx, tid = threadIdx.x;
  const int64_t row0 = (int64_t)blockIdx.x * S;
  const int rows = (int)min((int64_t)S, B - row0);
  const bool sobolev = (w_S != 0.f);

  WeightPipe pipe;
  int gi = 0;
  if (tid == 0) {
    sm.seq.n = 0;
    seq_push_critic_fwd(sm.seq, L, tw);      // one target pass over [s; s_next] (2S rows)
    seq_push_critic_fwd(sm.seq, L, cw);
    if (sobolev) {
      seq_push_critic_bwd(sm.seq, L, cwT);
      seq_push_critic_fwd(sm.seq, L, cw);
    }
    seq_push_critic_bwd(sm.seq, L, cwT);
    sm.loss = 0.f;
    small_bar_init(&sm.bar_small);
  }
  pipe.init(sm.WB, sm.bar);
  pipe.issue(sm.seq.ptr[0], sm.seq.first[0]);
  if (tid == 0) {
    small_bar_expect(&sm.bar_small, 2u * critic_small_bytes(L));
    load_critic_small(sm.sc, cw, L, &sm.bar_small);
    load_critic_small(sm.st, tw, L, &sm.bar_small);
  }
  float (*XN)[NSP] = sm.X2;
  load_normalised<S>(P, state, row0, rows, XN);
  if (!mc) load_normalised<S>(P, state_next, row0, rows, sm.X2 + S);
  const CriticPtrs cp = critic_ptrs(sm.sc), tp = critic_ptrs(sm.st);
  small_bar_wait(&sm.bar_small);
  __syncthreads();

  // ---- target critic: V_t(s_next) for the TD(n) tail (NeuralNetwork.py:157-158) and V_t(s) (:178)
  // (A and DL, unused until the sweeps, serve as [2S][128] scratch)
  if (!mc) critic_forward_tile<2 * S>(pipe, sm, gi, tp, L, sm.X2, &sm.A[0][0], &sm.DL[0][0], CR_H4, sm.VT2);
  else critic_forward_tile<S>(pipe, sm, gi, tp, L, sm.X2, &sm.A[0][0], &sm.DL[0][0], CR_H4, sm.VT2);
  if (tid < S) {
    float y = 0.f, w = 0.f;
    if (tid < rows) {
      const int64_t b = row0 + tid;
      y = mc ? prtg[b] : prtg[b] + (1.f - done[b]) * sm.VT2[S + tid];
      w = weights[b];
      rtg_out[b] = y;
      Vt_out[b] = sm.VT2[tid];
    }
    sm.Y[tid] = y;
    sm.WGT[tid] = w;
  }

  // ---- F: forward, keeping sin z_l and cos z_l of every hidden layer
  auto f_epi = [&](int l) {
    return [&, l](int r, int c, const float4& a) {
      const float4 b = *reinterpret_cast<const float4*>(cp.b[l] + c);
      float4 s, co;
      sincos4(a, b, s, co);
      *reinterpret_cast<float4*>(&sm.SN[r][koff(l) + c]) = s;
      *reinterpret_cast<float4*>(&sm.CS[r][koff(l) + c]) = co;
    };
  };
  tile_gemm<S, CR_H1, UP_NT, false>(&XN[0][0], NSP, ns, cp.W0, CR_H1, f_epi(0));
  __syncthreads();
  streamed<S, CR_H2>(pipe, sm, gi, &sm.SN[0][koff(0)], CW, CR_H1, f_epi(1));
  __syncthreads();
  streamed<S, CR_H3>(pipe, sm, gi, &sm.SN[0][koff(1)], CW, CR_H2, f_epi(2));
  __syncthreads();
  streamed<S, CR_H4>(pipe, sm, gi, &sm.SN[0][koff(2)], CW, CR_H3, f_epi(3));
  __syncthreads();
  tile_gemm_small<S, UP_NT, 8, true>(&sm.SN[0][koff(3)], CW, CR_H4, cp.W4, 1, 0,
                                     [&](int s, int, float v) { sm.V[s] = v + cp.b[4][0]; });
  __syncthreads();
  if (tid < rows) V_out[row0 + tid] = sm.V[tid];

  if (sobolev) {
    // ---- G: dV/dx through the network (tape2 of NeuralNetwork.py:162-165)
    for (int i = tid; i < S * CR_H4; i += UP_NT) {
      const int s = i / CR_H4, o = i - s * CR_H4;
      const float w5 = cp.W4[o];
      sm.G[s][koff(3) + o] = w5;
      sm.DL[s][koff(3) + o] = w5 * sm.CS[s][koff(3) + o];
    }
    __syncthreads();
    auto g_epi = [&](int l) {
      return [&, l](int r, int c, const float4& a) {
        const float4 co = *reinterpret_cast<const float4*>(&sm.CS[r][koff(l) + c]);
        *reinterpret_cast<float4*>(&sm.G[r][koff(l) + c]) = a;
        *reinterpret_cast<float4*>(&sm.DL[r][koff(l) + c]) = make_float4(a.x * co.x, a.y * co.y, a.z * co.z, a.w * co.w);
      };
    };
    streamed<S, CR_H3>(pipe, sm, gi, &sm.DL[0][koff(3)], CW, CR_H4, g_epi(2));
    __syncthreads();
    streamed<S, CR_H2>(pipe, sm, gi, &sm.DL[0][koff(2)], CW, CR_H3, g_epi(1));
    __syncthreads();
    streamed<S, CR_H1>(pipe, sm, gi, &sm.DL[0][koff(1)], CW, CR_H2, g_epi(0));
    __syncthreads();
    tile_gemm_small<S, UP_NT, 8, false>(&sm.DL[0][koff(0)], CW, CR_H1, cp.W0, ns, CR_H1,
                                        [&](int s, int j, float v) { sm.G0[s][j] = v; });
    __syncthreads();
  }

  // ---- loss and its seeds (NeuralNetwork.py:167-173; SURVEY.md A.3 step 3)
  {
    float lsum = 0.f;
    if (sobolev) {
      for (int i = tid; i < S * NSP; i += UP_NT) {
        const int s = i / NSP, j = i - s * NSP;
        float a0 = 0.f;
        if (s < rows && j < nx) {
          const float D = normalize_scale(P, j);
          const float gs = D * sm.G0[s][j];
          const float diff = slog(dVdx[(row0 + s) * ns + j]) - slog(gs);
          const float wn = sm.WGT[s] * inv_B / (float)nx;
          a0 = D * (-2.f * wn * diff * slog_grad(gs));
          lsum += wn * diff * diff;
        }
        sm.A0[s][j] = a0;
      }
    }
    if (tid < S) {
      float vbar = 0.f;
      if (tid < rows) {
        const float e = sm.Y[tid] - sm.V[tid];
        const float k = sobolev ? w_S : 1.f;
        vbar = -2.f * sm.WGT[tid] * k * inv_B * e;
        lsum += sm.WGT[tid] * k * inv_B * e * e;
      }
      sm.VBAR[tid] = vbar;
    }
    for (int off = 16; off > 0; off >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, off);
    if constexpr (DET) {
      // per-warp partials behind CriticSmem (launched with UP_NT / 32 more floats), summed in warp order
      if ((tid & 31) == 0) reinterpret_cast<float*>(smem_raw + sizeof(CriticSmem<S>))[tid >> 5] = lsum;
    } else {
      if ((tid & 31) == 0 && lsum != 0.f) atomicAdd(&sm.loss, lsum);
    }
  }
  __syncthreads();
  if constexpr (DET) {
    if (tid == 0) {
      const float* lw = reinterpret_cast<const float*>(smem_raw + sizeof(CriticSmem<S>));
      float l = 0.f;
      for (int w = 0; w < UP_NT / 32; ++w) l += lw[w];
      grad[L.total] += l;
    }
  } else {
    if (tid == 0 && loss_out != nullptr) atomicAdd(loss_out, sm.loss);
  }

  if (sobolev) {
    // ---- A: adjoint sweep through G (second-order terms); extra_l overwrites g_l, a_l kept for the outer products
    auto a_epi = [&](int l) {
      return [&, l](int r, int c, const float4& t) {
        const float4 co = *reinterpret_cast<const float4*>(&sm.CS[r][koff(l) + c]);
        const float4 si = *reinterpret_cast<const float4*>(&sm.SN[r][koff(l) + c]);
        const float4 g = *reinterpret_cast<const float4*>(&sm.G[r][koff(l) + c]);
        *reinterpret_cast<float4*>(&sm.A[r][koff(l) + c]) = make_float4(t.x * co.x, t.y * co.y, t.z * co.z, t.w * co.w);
        *reinterpret_cast<float4*>(&sm.G[r][koff(l) + c]) =
            make_float4(-t.x * g.x * si.x, -t.y * g.y * si.y, -t.z * g.z * si.z, -t.w * g.w * si.w);
      };
    };
    tile_gemm<S, CR_H1, UP_NT, false>(&sm.A0[0][0], NSP, ns, cp.W0, CR_H1, a_epi(0));
    __syncthreads();
    streamed<S, CR_H2>(pipe, sm, gi, &sm.A[0][koff(0)], CW, CR_H1, a_epi(1));
    __syncthreads();
    streamed<S, CR_H3>(pipe, sm, gi, &sm.A[0][koff(1)], CW, CR_H2, a_epi(2));
    __syncthreads();
    streamed<S, CR_H4>(pipe, sm, gi, &sm.A[0][koff(2)], CW, CR_H3, a_epi(3));
    __syncthreads();
    tile_colsum<UP_NT, DET>(&sm.A[0][koff(3)], CW, CR_H4, rows, grad + L.W[4]);       // d w5 += sum_s a_4
  } else {
    for (int i = tid; i < S * CW; i += UP_NT) sm.G[i / CW][i % CW] = 0.f;
    __syncthreads();
  }

  // ---- B: ordinary backward through F with the injected second-order terms
  for (int i = tid; i < S * CR_H4; i += UP_NT) {
    const int s = i / CR_H4, o = i - s * CR_H4;
    sm.G[s][koff(3) + o] += sm.VBAR[s] * cp.W4[o] * sm.CS[s][koff(3) + o];      // e_4
  }
  for (int o = tid; o < CR_H4; o += UP_NT) {                                                   // d w5 += sum_s vbar h_4
    float acc = 0.f;
    for (int s = 0; s < rows; ++s) acc += sm.VBAR[s] * sm.SN[s][koff(3) + o];
    grad_add<DET>(grad + L.W[4] + o, acc);
  }
  if (tid == 0) {
    float acc = 0.f;
    for (int s = 0; s < rows; ++s) acc += sm.VBAR[s];
    grad_add<DET>(grad + L.b[4], acc);
  }
  __syncthreads();
  auto b_epi = [&](int l) {   // e_l = (e_{l+1} W_{l+1}^T) * cos z_l + extra_l
    return [&, l](int r, int c, const float4& hb) {
      const float4 co = *reinterpret_cast<const float4*>(&sm.CS[r][koff(l) + c]);
      float4 g = *reinterpret_cast<const float4*>(&sm.G[r][koff(l) + c]);
      g.x += hb.x * co.x; g.y += hb.y * co.y; g.z += hb.z * co.z; g.w += hb.w * co.w;
      *reinterpret_cast<float4*>(&sm.G[r][koff(l) + c]) = g;
    };
  };
  const float* A2 = sobolev ? &sm.A[0][0] : nullptr;
  // layer 4
  tile_outer2<S, CR_H4, UP_NT, DET>(&sm.SN[0][koff(2)], CW, &sm.G[0][koff(3)], CW, A2 ? A2 + koff(2) : nullptr, CW, &sm.DL[0][koff(3)], CW,
                               CR_H3, grad + L.W[3], rows);
  tile_colsum<UP_NT, DET>(&sm.G[0][koff(3)], CW, CR_H4, rows, grad + L.b[3]);
  streamed<S, CR_H3>(pipe, sm, gi, &sm.G[0][koff(3)], CW, CR_H4, b_epi(2));
  __syncthreads();
  // layer 3
  tile_outer2<S, CR_H3, UP_NT, DET>(&sm.SN[0][koff(1)], CW, &sm.G[0][koff(2)], CW, A2 ? A2 + koff(1) : nullptr, CW, &sm.DL[0][koff(2)], CW,
                               CR_H2, grad + L.W[2], rows);
  tile_colsum<UP_NT, DET>(&sm.G[0][koff(2)], CW, CR_H3, rows, grad + L.b[2]);
  streamed<S, CR_H2>(pipe, sm, gi, &sm.G[0][koff(2)], CW, CR_H3, b_epi(1));
  __syncthreads();
  // layer 2
  tile_outer2<S, CR_H2, UP_NT, DET>(&sm.SN[0][koff(0)], CW, &sm.G[0][koff(1)], CW, A2 ? A2 + koff(0) : nullptr, CW, &sm.DL[0][koff(1)], CW,
                               CR_H1, grad + L.W[1], rows);
  tile_colsum<UP_NT, DET>(&sm.G[0][koff(1)], CW, CR_H2, rows, grad + L.b[1]);
  streamed<S, CR_H1>(pipe, sm, gi, &sm.G[0][koff(1)], CW, CR_H2, b_epi(0));
  __syncthreads();
  // layer 1
  tile_outer2<S, CR_H1, UP_NT, DET>(&XN[0][0], NSP, &sm.G[0][koff(0)], CW, sobolev ? &sm.A0[0][0] : nullptr, NSP, &sm.DL[0][koff(0)], CW, ns,
                               grad + L.W[0], rows);
  tile_colsum<UP_NT, DET>(&sm.G[0][koff(0)], CW, CR_H1, rows, grad + L.b[0]);
}

// ------------------------------------------------------------------------------------------ actor
template <int S>
struct ActorSmem {
  alignas(128) float WB[2 * W_CHUNK];
  uint64_t bar[2], bar_small;
  WeightSeq seq;
  ActorSmall sa;
  CriticSmall sc;
  alignas(16) float XN[S][NSP];
  float XNP[S][NSP], G0[S][NSP];
  float H1[S][ACTOR_H], H2[S][ACTOR_H], E[S][ACTOR_H];
  float CS[S][CW];
  float CH[2][S][CR_H4];
  float DLp[2][S][CR_H4];
  float FU[S][CACTO_MAX_NS * CACTO_MAX_NA + 2];
  float ACT[S][NAP], D3[S][NAP], DRDA[S][NAP];
};

template <int SYS, int S, bool DET = false>
__global__ void __launch_bounds__(UP_NT) k_actor_grad(const __grid_constant__ cacto_sys_params P, const float* __restrict__ aw,
                                                      const float* __restrict__ awT, const float* __restrict__ cw,
                                                      const float* __restrict__ cwT, const float* __restrict__ state,
                                                      const double* __restrict__ term, float inv_B, float* __restrict__ grad,
                                                      float* __restrict__ actions_out, int64_t B) {
  pdl_wait();
  constexpr int NX = SysDims<SYS>::NX, NA = SysDims<SYS>::NA, NS = NX + 1;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  ActorSmem<S>& sm = *reinterpret_cast<ActorSmem<S>*>(smem_raw);
  const ActorLayout LA(NS, NA);
  const CriticLayout LC(NS);
  if constexpr (DET) grad += (size_t)blockIdx.x * det_stride(LA.total);
  const int tid = threadIdx.x;
  const int64_t row0 = (int64_t)blockIdx.x * S;
  const int rows = (int)min((int64_t)S, B - row0);

  WeightPipe pipe;
  int gi = 0;
  if (tid == 0) {
    sm.seq.n = 0;
    seq_push<ACTOR_H>(sm.seq, aw + LA.W2, ACTOR_H);
    seq_push_critic_fwd(sm.seq, LC, cw);
    seq_push_critic_bwd(sm.seq, LC, cwT);
    seq_push<ACTOR_H>(sm.seq, awT + LA.W2, ACTOR_H);
    small_bar_init(&sm.bar_small);
  }
  pipe.init(sm.WB, sm.bar);
  pipe.issue(sm.seq.ptr[0], sm.seq.first[0]);
  if (tid == 0) {
    small_bar_expect(&sm.bar_small, actor_small_bytes(LA) + critic_small_bytes(LC));
    load_actor_small(sm.sa, aw, LA, &sm.bar_small);
    load_critic_small(sm.sc, cw, LC, &sm.bar_small);
  }
  load_normalised<S>(P, state, row0, rows, sm.XN);
  const CriticPtrs cp = critic_ptrs(sm.sc);
  small_bar_wait(&sm.bar_small);
  __syncthreads();
  // ---- actor forward (NeuralNetwork.py:185)
  tile_gemm<S, ACTOR_H, UP_NT, false>(&sm.XN[0][0], NSP, NS, sm.sa.W1, ACTOR_H, [&](int r, int c, const float4& a) {
    const float4 b = *reinterpret_cast<const float4*>(sm.sa.b1 + c);
    *reinterpret_cast<float4*>(&sm.H1[r][c]) = make_float4(leaky(a.x + b.x), leaky(a.y + b.y), leaky(a.z + b.z), leaky(a.w + b.w));
  });
  __syncthreads();
  streamed<S, ACTOR_H>(pipe, sm, gi, &sm.H1[0][0], ACTOR_H, ACTOR_H, [&](int r, int c, const float4& a) {
    const float4 b = *reinterpret_cast<const float4*>(sm.sa.b2 + c);
    *reinterpret_cast<float4*>(&sm.H2[r][c]) = make_float4(leaky(a.x + b.x), leaky(a.y + b.y), leaky(a.z + b.z), leaky(a.w + b.w));
  });
  __syncthreads();
  tile_gemm_small<S, UP_NT, 8, true>(&sm.H2[0][0], ACTOR_H, ACTOR_H, sm.sa.W3, NA, 0,
                                     [&](int s, int j, float v) { sm.ACT[s][j] = v + sm.sa.b3[j]; });
  __syncthreads();

  // ---- per sample: s' = f(s, a), ds'/da (normalised), dr/da  (NeuralNetwork.py:188,199-204)
  if (tid < S) {
    float xnp[NSP];
#pragma unroll
    for (int j = 0; j < NSP; ++j) xnp[j] = 0.f;
    if (tid < rows) {
      const int64_t b = row0 + tid;
      double x[NS], u[NA], xn[NS], Fu[NX * NA];
#pragma unroll
      for (int j = 0; j < NS; ++j) x[j] = (double)state[b * NS + j];
#pragma unroll
      for (int j = 0; j < NA; ++j) {
        u[j] = (double)sm.ACT[tid][j];
        if (actions_out != nullptr) actions_out[b * NA + j] = sm.ACT[tid][j];
      }
      sys_step_Fu<SYS, double>(P, x, u, xn, Fu);
      xn[NX] = x[NX] + P.dt;
#pragma unroll
      for (int i = 0; i < NX; ++i) {
        const double inv = P.normalize ? 1.0 / P.state_norm[i] : 1.0;
#pragma unroll
        for (int j = 0; j < NA; ++j) sm.FU[tid][i * NA + j] = (float)(Fu[i * NA + j] * inv);
      }
#pragma unroll
      for (int j = 0; j < NA; ++j) sm.FU[tid][NX * NA + j] = 0.f;
#pragma unroll
      for (int j = 0; j < NS; ++j) xnp[j] = normalize_component(P, j, (float)xn[j]);
      const double tm = term[b];
      const float w6 = (float)(tm * P.w_terminal[6] + (1.0 - tm) * P.w_running[6]);     // NeuralNetwork.py:201
      float uf[NA], g[NA];
#pragma unroll
      for (int j = 0; j < NA; ++j) uf[j] = sm.ACT[tid][j];
      sys_dr_da<SYS, float>(P, w6, uf, g);
#pragma unroll
      for (int j = 0; j < NA; ++j) sm.DRDA[tid][j] = g[j];
    }
#pragma unroll
    for (int j = 0; j < NSP; ++j) sm.XNP[tid][j] = xnp[j];
  }
  __syncthreads();

  // ---- critic forward at s' keeping cos z_l, then the input-gradient sweep (NeuralNetwork.py:190-195)
  auto cf_epi = [&](int l, float* out) {
    return [&, l, out](int r, int c, const float4& a) {
      const float4 b = *reinterpret_cast<const float4*>(cp.b[l] + c);
      float4 s, co;
      sincos4(a, b, s, co);
      *reinterpret_cast<float4*>(out + r * CR_H4 + c) = s;
      *reinterpret_cast<float4*>(&sm.CS[r][koff(l) + c]) = co;
    };
  };
  float* ch0 = &sm.CH[0][0][0];
  float* ch1 = &sm.CH[1][0][0];
  tile_gemm<S, CR_H1, UP_NT, false>(&sm.XNP[0][0], NSP, NS, cp.W0, CR_H1, cf_epi(0, ch0));
  __syncthreads();
  streamed<S, CR_H2>(pipe, sm, gi, ch0, CR_H4, CR_H1, cf_epi(1, ch1));
  __syncthreads();
  streamed<S, CR_H3>(pipe, sm, gi, ch1, CR_H4, CR_H2, cf_epi(2, ch0));
  __syncthreads();
  streamed<S, CR_H4>(pipe, sm, gi, ch0, CR_H4, CR_H3, cf_epi(3, ch1));
  __syncthreads();
  float* dl0 = &sm.DLp[0][0][0];
  float* dl1 = &sm.DLp[1][0][0];
  for (int i = tid; i < S * CR_H4; i += UP_NT) {
    const int s = i / CR_H4, o = i - s * CR_H4;
    dl0[s * CR_H4 + o] = cp.W4[o] * sm.CS[s][koff(3) + o];
  }
  __syncthreads();
  auto cg_epi = [&](int l, float* out) {
    return [&, l, out](int r, int c, const float4& a) {
      const float4 co = *reinterpret_cast<const float4*>(&sm.CS[r][koff(l) + c]);
      *reinterpret_cast<float4*>(out + r * CR_H4 + c) = make_float4(a.x * co.x, a.y * co.y, a.z * co.z, a.w * co.w);
    };
  };
  streamed<S, CR_H3>(pipe, sm, gi, dl0, CR_H4, CR_H4, cg_epi(2, dl1));
  __syncthreads();
  streamed<S, CR_H2>(pipe, sm, gi, dl1, CR_H4, CR_H3, cg_epi(1, dl0));
  __syncthreads();
  streamed<S, CR_H1>(pipe, sm, gi, dl0, CR_H4, CR_H2, cg_epi(0, dl1));
  __syncthreads();
  tile_gemm_small<S, UP_NT, 8, false>(dl1, CR_H4, CR_H1, cp.W0, NS, CR_H1, [&](int s, int j, float v) { sm.G0[s][j] = v; });
  __syncthreads();

  // ---- dQ/da = dV/ds' . ds'/da + dr/da ; upstream gradient on the actor output = -dQ/da / B  (:206-228)
  for (int i = tid; i < S * NAP; i += UP_NT) {
    const int s = i / NAP, j = i - s * NAP;
    float d3 = 0.f;
    if (s < rows && j < NA) {
      float q = sm.DRDA[s][j];
#pragma unroll
      for (int k = 0; k < NS; ++k) q = fmaf(normalize_scale(P, k) * sm.G0[s][k], sm.FU[s][k * NA + j], q);
      d3 = -q * inv_B;
    }
    sm.D3[s][j] = d3;
  }
  __syncthreads();

  // ---- actor backward
  for (int i = tid; i < ACTOR_H * NA; i += UP_NT) {            // dW3[k][j] += sum_s h2[s][k] d3[s][j]
    const int k = i / NA, j = i - k * NA;
    float acc = 0.f;
    for (int s = 0; s < rows; ++s) acc = fmaf(sm.H2[s][k], sm.D3[s][j], acc);
    grad_add<DET>(grad + LA.W3 + i, acc);
  }
  if (tid < NA) {
    float acc = 0.f;
    for (int s = 0; s < rows; ++s) acc += sm.D3[s][tid];
    grad_add<DET>(grad + LA.b3 + tid, acc);
  }
  for (int i = tid; i < S * ACTOR_H; i += UP_NT) {             // e2 = (d3 W3^T) * lrelu'(z2)
    const int s = i / ACTOR_H, n = i - s * ACTOR_H;
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < NA; ++j) acc = fmaf(sm.D3[s][j], sm.sa.W3[n * NA + j], acc);
    sm.E[s][n] = acc * (sm.H2[s][n] > 0.f ? 1.f : LEAKY_ALPHA);
  }
  __syncthreads();
  tile_outer2<S, ACTOR_H, UP_NT, DET>(&sm.H1[0][0], ACTOR_H, &sm.E[0][0], ACTOR_H, nullptr, 0, nullptr, 0, ACTOR_H, grad + LA.W2, rows);
  tile_colsum<UP_NT, DET>(&sm.E[0][0], ACTOR_H, ACTOR_H, rows, grad + LA.b2);
  streamed<S, ACTOR_H>(pipe, sm, gi, &sm.E[0][0], ACTOR_H, ACTOR_H, [&](int r, int c, const float4& a) {
    const float4 h = *reinterpret_cast<const float4*>(&sm.H1[r][c]);
    *reinterpret_cast<float4*>(&sm.H2[r][c]) =
        make_float4(a.x * (h.x > 0.f ? 1.f : LEAKY_ALPHA), a.y * (h.y > 0.f ? 1.f : LEAKY_ALPHA), a.z * (h.z > 0.f ? 1.f : LEAKY_ALPHA),
                    a.w * (h.w > 0.f ? 1.f : LEAKY_ALPHA));
  });
  __syncthreads();
  tile_outer2<S, ACTOR_H, UP_NT, DET>(&sm.XN[0][0], NSP, &sm.H2[0][0], ACTOR_H, nullptr, 0, nullptr, 0, NS, grad + LA.W1, rows);
  tile_colsum<UP_NT, DET>(&sm.H2[0][0], ACTOR_H, ACTOR_H, rows, grad + LA.b1);
}

// ------------------------------------------------------------------------------------------ forward-only kernels
template <int S>
struct EvalSmem {
  alignas(128) float WB[2 * W_CHUNK];
  uint64_t bar[2];
  WeightSeq seq;
  alignas(16) float XN[S][NSP];
  float A[S][ACTOR_H], Bf[S][ACTOR_H];
  float CS[S][CW];
  float V[S], G0[S][NSP];
  float ACT[S][NAP];
};

template <int S>
__global__ void __launch_bounds__(UP_NT) k_actor_forward(const __grid_constant__ cacto_sys_params P, const float* __restrict__ aw,
                                                         const float* __restrict__ state, float* __restrict__ out, int64_t B) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  EvalSmem<S>& sm = *reinterpret_cast<EvalSmem<S>*>(smem_raw);
  const int ns = P.ns, na = P.na;
  const ActorLayout LA(ns, na);
  const int64_t row0 = (int64_t)blockIdx.x * S;
  const int rows = (int)min((int64_t)S, B - row0);
  WeightPipe pipe;
  int gi = 0;
  if (threadIdx.x == 0) {
    sm.seq.n = 0;
    seq_push<ACTOR_H>(sm.seq, aw + LA.W2, ACTOR_H);
  }
  pipe.init(sm.WB, sm.bar);
  pipe.issue(sm.seq.ptr[0], sm.seq.first[0]);
  load_normalised<S>(P, state, row0, rows, sm.XN);
  __syncthreads();
  tile_gemm<S, ACTOR_H, UP_NT, false>(&sm.XN[0][0], NSP, ns, aw + LA.W1, ACTOR_H, [&](int r, int c, const float4& a) {
    const float4 b = __ldg(reinterpret_cast<const float4*>(aw + LA.b1 + c));
    *reinterpret_cast<float4*>(&sm.A[r][c]) = make_float4(leaky(a.x + b.x), leaky(a.y + b.y), leaky(a.z + b.z), leaky(a.w + b.w));
  });
  __syncthreads();
  streamed<S, ACTOR_H>(pipe, sm, gi, &sm.A[0][0], ACTOR_H, ACTOR_H, [&](int r, int c, const float4& a) {
    const float4 b = __ldg(reinterpret_cast<const float4*>(aw + LA.b2 + c));
    *reinterpret_cast<float4*>(&sm.Bf[r][c]) = make_float4(leaky(a.x + b.x), leaky(a.y + b.y), leaky(a.z + b.z), leaky(a.w + b.w));
  });
  __syncthreads();
  tile_gemm_small<S, UP_NT, 8, true>(&sm.Bf[0][0], ACTOR_H, ACTOR_H, aw + LA.W3, na, 0, [&](int s, int j, float v) {
    if (s < rows) out[(row0 + s) * na + j] = v + __ldg(aw + LA.b3 + j);
  });
}

template <int S>
__global__ void __launch_bounds__(UP_NT) k_critic_forward(const __grid_constant__ cacto_sys_params P, const float* __restrict__ cw,
                                                          const float* __restrict__ state, float* __restrict__ value,
                                                          float* __restrict__ dV_ds, int64_t B) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  EvalSmem<S>& sm = *reinterpret_cast<EvalSmem<S>*>(smem_raw);
  const int ns = P.ns, tid = threadIdx.x;
  const CriticLayout L(ns);
  const int64_t row0 = (int64_t)blockIdx.x * S;
  const int rows = (int)min((int64_t)S, B - row0);
  WeightPipe pipe;
  int gi = 0;
  if (tid == 0) {
    sm.seq.n = 0;
    seq_push_critic_fwd(sm.seq, L, cw);
  }
  pipe.init(sm.WB, sm.bar);
  pipe.issue(sm.seq.ptr[0], sm.seq.first[0]);
  load_normalised<S>(P, state, row0, rows, sm.XN);
  __syncthreads();
  float* bufA = &sm.A[0][0];
  float* bufB = &sm.Bf[0][0];
  auto f_epi = [&](int l, float* out) {
    return [&, l, out](int r, int c, const float4& a) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(cw + L.b[l] + c));
      float4 s, co;
      sincos4(a, b, s, co);
      *reinterpret_cast<float4*>(out + r * ACTOR_H + c) = s;
      *reinterpret_cast<float4*>(&sm.CS[r][koff(l) + c]) = co;
    };
  };
  tile_gemm<S, CR_H1, UP_NT, false>(&sm.XN[0][0], NSP, ns, cw + L.W[0], CR_H1, f_epi(0, bufA));
  __syncthreads();
  streamed<S, CR_H2>(pipe, sm, gi, bufA, ACTOR_H, CR_H1, f_epi(1, bufB));
  __syncthreads();
  streamed<S, CR_H3>(pipe, sm, gi, bufB, ACTOR_H, CR_H2, f_epi(2, bufA));
  __syncthreads();
  streamed<S, CR_H4>(pipe, sm, gi, bufA, ACTOR_H, CR_H3, f_epi(3, bufB));
  __syncthreads();
  tile_gemm_small<S, UP_NT, 8, true>(bufB, ACTOR_H, CR_H4, cw + L.W[4], 1, 0, [&](int s, int, float v) {
    if (s < rows) value[row0 + s] = v + __ldg(cw + L.b[4]);
  });
  if (dV_ds == nullptr) return;
  __syncthreads();
  // input gradient with the un-transposed weights (forward-only callers have no transposed copy):
  // g_{l-1}[s][i] = sum_o delta_l[s][o] W_l[i][o]  -> G lanes per output over contiguous W rows
  for (int i = tid; i < S * CR_H4; i += UP_NT) {
    const int s = i / CR_H4, o = i - s * CR_H4;
    bufA[s * ACTOR_H + o] = __ldg(cw + L.W[4] + o) * sm.CS[s][koff(3) + o];
  }
  __syncthreads();
  tile_gemm_small<S, UP_NT, 8, false>(bufA, ACTOR_H, CR_H4, cw + L.W[3], CR_H3, CR_H4,
                                      [&](int s, int j, float v) { bufB[s * ACTOR_H + j] = v * sm.CS[s][koff(2) + j]; });
  __syncthreads();
  tile_gemm_small<S, UP_NT, 8, false>(bufB, ACTOR_H, CR_H3, cw + L.W[2], CR_H2, CR_H3,
                                      [&](int s, int j, float v) { bufA[s * ACTOR_H + j] = v * sm.CS[s][koff(1) + j]; });
  __syncthreads();
  tile_gemm_small<S, UP_NT, 8, false>(bufA, ACTOR_H, CR_H2, cw + L.W[1], CR_H1, CR_H2,
                                      [&](int s, int j, float v) { bufB[s * ACTOR_H + j] = v * sm.CS[s][koff(0) + j]; });
  __syncthreads();
  tile_gemm_small<S, UP_NT, 8, false>(bufB, ACTOR_H, CR_H1, cw + L.W[0], ns, CR_H1, [&](int s, int j, float v) {
    if (s < rows) dV_ds[(row0 + s) * ns + j] = normalize_scale(P, j) * v;
  });
}

// ------------------------------------------------------------------------------------------ optimiser
struct LayerTable {
  int n;
  int64_t W[5];
  int in[5], out[5];
};

// index of parameter i inside the per-layer transposed copy (weights [in][out] -> [out][in], biases unchanged)
__device__ __forceinline__ int64_t transposed_index(const LayerTable& T, int64_t i) {
  for (int l = 0; l < T.n; ++l) {
    const int64_t sz = (int64_t)T.in[l] * T.out[l];
    if (i >= T.W[l] && i < T.W[l] + sz) {
      const int64_t e = i - T.W[l];
      const int r = (int)(e / T.out[l]), c = (int)(e - (int64_t)r * T.out[l]);
      return T.W[l] + (int64_t)c * T.in[l] + r;
    }
  }
  return i;
}

// 1 - h for a hyperparameter h that arrived as a float: TF 2.11's optimizer (and RL.py:116-118's Polyak step) form 1 - beta / 1 - tau in
// Python double precision from the decimal literal and only then round to fp32, which is not 1.f - (float)h (for beta2 = 0.999 the two
// differ by 1.3e-5 relative).  The float encodes at most 7 significant decimals of the literal: recover them, subtract in double.
static inline float one_minus(float h) {
  if (!(h > 0.f && h < 1.f)) return 1.f - h;
  double scale = 1e7;
  for (double a = h; a < 0.1; a *= 10.0) scale *= 10.0;      // keep 7 significant digits for small h (tau = 0.001)
  return (float)(1.0 - nearbyint((double)h * scale) / scale);
}

// p -= alpha * m / (sqrt(v) + eps) with m += (g - m)(1 - b1), v += (g^2 - v)(1 - b2)   (SURVEY.md A.5), the Polyak target
// update (RL.py:116-118) and the refresh of the transposed copy, for parameter i with gradient gi
__device__ __forceinline__ void adam_element(int64_t i, float gi, float* __restrict__ p, float* __restrict__ m, float* __restrict__ v, float alpha,
                                             float omb1, float omb2, float eps, float* __restrict__ target, float2 tt, float* __restrict__ pT,
                                             const LayerTable& T) {
  float mi = m[i], vi = v[i];
  mi += (gi - mi) * omb1;
  vi += (gi * gi - vi) * omb2;
  m[i] = mi;
  v[i] = vi;
  const float pi = p[i] - (mi * alpha) / (sqrtf(vi) + eps);
  p[i] = pi;
  if (target != nullptr) target[i] = pi * tt.x + target[i] * tt.y;
  if (pT != nullptr) pT[transposed_index(T, i)] = pi;
}

__global__ void __launch_bounds__(256) k_adam(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                              float alpha, const float* __restrict__ alpha_dev, float omb1, float omb2, float eps,
                                              float* __restrict__ target, float2 tt,
                                              float* __restrict__ pT, LayerTable T, int64_t n) {
  pdl_wait();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gi = g[i];
  g[i] = 0.f;
  if (alpha_dev != nullptr) alpha = __ldg(alpha_dev);     // device-side schedule (CUDA-graph replays)
  adam_element(i, gi, p, m, v, alpha, omb1, omb2, eps, target, tt, pT, T);
}

// ---- data-parallel update: the gradient all-reduce fused into the Adam step over NVLink peer memory (SURVEY.md 8e).
// Every rank keeps its gradient sums in a CUDA-IPC region mapped by all ranks of the box.  The kernel (i) announces "my
// gradients of launch number `epoch` are complete" with one system-scope release store into the flag word [rank] of every peer,
// (ii) waits until the flag words of all peers in its own region have reached `epoch`, (iii) sums the W gradient blocks in
// rank order 0..W-1 with peer loads through NVSwitch -- the same order on every rank, so the replicas stay bit-identical --
// and applies Adam / Polyak / the transposed refresh.  The rank's own gradient block cannot be cleared here (peers may
// still be reading it); instead the kernel clears `zero_other`, the gradient block of the OTHER network: every peer has
// finished reading that block before it announced the step this kernel has just waited for (critic and actor steps
// alternate, RL.py:104-109).  Replaces two NCCL all-reduce launches per update by two flag round trips.
struct PeerTable {
  const float* grad[CACTO_MAX_PEERS];   // gradient block of every rank (own block included), peer-mapped
  unsigned* flags[CACTO_MAX_PEERS];     // flag words [CACTO_MAX_PEERS] of every rank
  int world, rank;
};

__global__ void __launch_bounds__(256) k_adam_peer(float* __restrict__ p, PeerTable R, float* __restrict__ zero_other, int64_t n_other,
                                                   float* __restrict__ m, float* __restrict__ v, const float* __restrict__ alpha_dev, float omb1,
                                                   float omb2, float eps, float* __restrict__ target, float2 tt, float* __restrict__ pT,
                                                   LayerTable T, int64_t n) {
  pdl_wait();
  // words [0, CACTO_MAX_PEERS) of a rank's flag row: arrival epochs written by the peers; [CACTO_MAX_PEERS]: number of steps this
  // rank has completed (the epoch base, never rewound -- unlike the Adam step counter, which graph capture restores);
  // [CACTO_MAX_PEERS + 1]: CTA ticket of the running launch
  unsigned* mine = R.flags[R.rank];
  const unsigned epoch = *reinterpret_cast<volatile unsigned*>(mine + CACTO_MAX_PEERS) + 1u;
  if (blockIdx.x == 0 && threadIdx.x < R.world) {          // the preceding gradient kernel has completed (stream order)
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(R.flags[threadIdx.x] + R.rank), "r"(epoch) : "memory");
  }
  if (threadIdx.x < R.world) {
    const unsigned* f = mine + threadIdx.x;
    unsigned seen = 0, spins = 0;
    unsigned long long t0 = 0;
    while (true) {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(f) : "memory");
      if ((int)(seen - epoch) >= 0) break;
      if ((++spins & 255u) == 0) {                         // a peer that never arrives: fail loudly after 20 s instead of hanging
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        if (t0 == 0) t0 = now;
        else if (now - t0 > 20000000000ull) __trap();
      }
    }
  }
  __syncthreads();
  const int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t j = i0; j < n_other; j += stride) zero_other[j] = 0.f;
  const float alpha = __ldg(alpha_dev);
  for (int64_t i = i0; i < n; i += stride) {
    float x[CACTO_MAX_PEERS];
#pragma unroll
    for (int r = 0; r < CACTO_MAX_PEERS; ++r) {            // all peer loads in flight together (one NVLink round trip), ...
      x[r] = 0.f;
      if (r < R.world) asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(x[r]) : "l"(R.grad[r] + i) : "memory");
    }
    float gi = x[0];
#pragma unroll
    for (int r = 1; r < CACTO_MAX_PEERS; ++r)              // ... summed in rank order
      if (r < R.world) gi += x[r];
    adam_element(i, gi, p, m, v, alpha, omb1, omb2, eps, target, tt, pT, T);
  }
  __syncthreads();
  if (threadIdx.x == 0) {                                  // the last CTA to finish advances the epoch base for the next launch
    const unsigned ticket = atomicAdd(mine + CACTO_MAX_PEERS + 1, 1u);
    if (ticket == gridDim.x - 1) {
      mine[CACTO_MAX_PEERS + 1] = 0u;
      *reinterpret_cast<volatile unsigned*>(mine + CACTO_MAX_PEERS) = epoch;
    }
  }
}

__global__ void __launch_bounds__(256) k_transpose(const float* __restrict__ p, float* __restrict__ pT, LayerTable T, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  pT[transposed_index(T, i)] = p[i];
}

static LayerTable make_table(int is_critic, int ns, int na, int64_t* total) {
  LayerTable T;
  if (is_critic) {
    CriticLayout L(ns);
    T.n = 5;
    for (int l = 0; l < 5; ++l) { T.W[l] = L.W[l]; T.in[l] = L.in[l]; T.out[l] = L.out[l]; }
    *total = L.total;
  } else {
    ActorLayout L(ns, na);
    T.n = 3;
    T.W[0] = L.W1; T.in[0] = ns; T.out[0] = ACTOR_H;
    T.W[1] = L.W2; T.in[1] = ACTOR_H; T.out[1] = ACTOR_H;
    T.W[2] = L.W3; T.in[2] = ACTOR_H; T.out[2] = na;
    for (int l = 3; l < 5; ++l) { T.W[l] = 0; T.in[l] = 0; T.out[l] = 0; }
    *total = L.total;
  }
  return T;
}

template <typename K>
static int smem_attr(K k, size_t bytes) {
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  return e == cudaSuccess ? 0 : (int)e;
}

// Samples per CTA.  A CTA walks a latency chain of ~25 dependent phases whose length grows with its rows, and one CTA fits an SM
// (200 KB of shared memory): the smallest tile that still covers the batch in ONE wave of 148 CTAs wins -- 2 rows up to B = 296
// (the reference's 64 / 128: 103.7 / 109.4 us per update as a CUDA graph vs 127 us with 8-row tiles), 4 up to 592, 8 below the
// size where 16-row tiles fill the GPU, 16 (best FMA : LDS ratio) beyond.
static int pick_tile(int64_t B) { return B >= 16 * 148 ? 16 : (B <= 2 * 148 ? 2 : (B <= 4 * 148 ? 4 : 8)); }

template <int SYS>
static int launch_actor_grad(const cacto_sys_params& P, const float* aw, const float* awT, const float* cw, const float* cwT,
                             const float* state, const double* term, float inv_B, float* grad, float* actions, int64_t B,
                             cudaStream_t st) {
  if (pick_tile(B) == 16) {
    auto k = k_actor_grad<SYS, 16>;
    if (int e = smem_attr(k, sizeof(ActorSmem<16>))) return e;
    if (cudaError_t le = launch_pdl(k, (unsigned)((B + 15) / 16), UP_NT, sizeof(ActorSmem<16>), st, P, aw, awT, cw, cwT, state, term, inv_B, grad, actions, B)) return (int)le;
  } else if (pick_tile(B) == 8) {
    auto k = k_actor_grad<SYS, 8>;
    if (int e = smem_attr(k, sizeof(ActorSmem<8>))) return e;
    if (cudaError_t le = launch_pdl(k, (unsigned)((B + 7) / 8), UP_NT, sizeof(ActorSmem<8>), st, P, aw, awT, cw, cwT, state, term, inv_B, grad, actions, B)) return (int)le;
  } else if (pick_tile(B) == 4) {
    auto k = k_actor_grad<SYS, 4>;
    if (int e = smem_attr(k, sizeof(ActorSmem<4>))) return e;
    if (cudaError_t le = launch_pdl(k, (unsigned)((B + 3) / 4), UP_NT, sizeof(ActorSmem<4>), st, P, aw, awT, cw, cwT, state, term, inv_B, grad, actions, B)) return (int)le;
  } else {
    auto k = k_actor_grad<SYS, 2>;
    if (int e = smem_attr(k, sizeof(ActorSmem<2>))) return e;
    if (cudaError_t le = launch_pdl(k, (unsigned)((B + 1) / 2), UP_NT, sizeof(ActorSmem<2>), st, P, aw, awT, cw, cwT, state, term, inv_B, grad, actions, B)) return (int)le;
  }
  CACTO_LAUNCH_CHECK();
  return 0;
}

}  // namespace cacto

using namespace cacto;

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

extern "C" int cacto_critic_grad(const cacto_sys_params* p, const float* critic_params, const float* critic_params_T,
                                 const float* target_params, float w_S, int mc, const float* state, const float* state_next,
                                 const float* partial_rtg, const float* dVdx, const float* done, const float* weights, float inv_B,
                                 float* grad, float* rtg, float* V, float* V_target_s, float* loss, int64_t B, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (B < 0) return CACTO_E_SIZE;
  if (B == 0) return 0;
  if (!critic_params || !critic_params_T || !target_params || !state || !partial_rtg || !weights || !grad || !rtg || !V || !V_target_s)
    return CACTO_E_ARG;
  if (!mc && (!state_next || !done)) return CACTO_E_ARG;
  if (w_S != 0.f && !dVdx) return CACTO_E_ARG;
  if (!aligned16(critic_params) || !aligned16(critic_params_T) || !aligned16(target_params) || !aligned16(grad)) return CACTO_E_ALIGN;
  cudaStream_t st = (cudaStream_t)stream;
  if (pick_tile(B) == 16) {
    auto k = k_critic_grad<16>;
    if (int e = smem_attr(k, sizeof(CriticSmem<16>))) return e;
    if (cudaError_t le = launch_pdl(k, (unsigned)((B + 15) / 16), UP_NT, sizeof(CriticSmem<16>), st, *p, critic_params, critic_params_T, target_params, w_S, mc, state,
                                                                        state_next, partial_rtg, dVdx, done, weights, inv_B, grad, rtg, V,
                                                                        V_target_s, loss, B)) return (int)le;
  } else if (pick_tile(B) == 8) {
    auto k = k_critic_grad<8>;
    if (int e = smem_attr(k, sizeof(CriticSmem<8>))) return e;
    if (cudaError_t le = launch_pdl(k, (unsigned)((B + 7) / 8), UP_NT, sizeof(CriticSmem<8>), st, *p, critic_params, critic_params_T, target_params, w_S, mc, state,
                                                                     state_next, partial_rtg, dVdx, done, weights, inv_B, grad, rtg, V,
                                                                     V_target_s, loss, B)) return (int)le;
  } else if (pick_tile(B) == 4) {
    auto k = k_critic_grad<4>;
    if (int e = smem_attr(k, sizeof(CriticSmem<4>))) return e;
    if (cudaError_t le = launch_pdl(k, (unsigned)((B + 3) / 4), UP_NT, sizeof(CriticSmem<4>), st, *p, critic_params, critic_params_T, target_params, w_S, mc, state,
                                                                     state_next, partial_rtg, dVdx, done, weights, inv_B, grad, rtg, V,
                                                                     V_target_s, loss, B)) return (int)le;
  } else {
    auto k = k_critic_grad<2>;
    if (int e = smem_attr(k, sizeof(CriticSmem<2>))) return e;
    if (cudaError_t le = launch_pdl(k, (unsigned)((B + 1) / 2), UP_NT, sizeof(CriticSmem<2>), st, *p, critic_params, critic_params_T, target_params, w_S, mc, state,
                                                                     state_next, partial_rtg, dVdx, done, weights, inv_B, grad, rtg, V,
                                                                     V_target_s, loss, B)) return (int)le;
  }
  CACTO_LAUNCH_CHECK();
  return 0;
}

extern "C" int cacto_actor_grad(const cacto_sys_params* p, const float* actor_params, const float* actor_params_T,
                                const float* critic_params, const float* critic_params_T, const float* state, const double* term,
                                float inv_B, float* grad, float* actions, int64_t B, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (B < 0) return CACTO_E_SIZE;
  if (B == 0) return 0;
  if (!actor_params || !actor_params_T || !critic_params || !critic_params_T || !state || !term || !grad) return CACTO_E_ARG;
  if (!aligned16(actor_params) || !aligned16(actor_params_T) || !aligned16(critic_params) || !aligned16(critic_params_T) || !aligned16(grad))
    return CACTO_E_ALIGN;
  cudaStream_t st = (cudaStream_t)stream;
  switch (p->system) {
    case CACTO_SINGLE_INTEGRATOR: return launch_actor_grad<CACTO_SINGLE_INTEGRATOR>(*p, actor_params, actor_params_T, critic_params, critic_params_T, state, term, inv_B, grad, actions, B, st);
    case CACTO_DOUBLE_INTEGRATOR: return launch_actor_grad<CACTO_DOUBLE_INTEGRATOR>(*p, actor_params, actor_params_T, critic_params, critic_params_T, state, term, inv_B, grad, actions, B, st);
    case CACTO_CAR: return launch_actor_grad<CACTO_CAR>(*p, actor_params, actor_params_T, critic_params, critic_params_T, state, term, inv_B, grad, actions, B, st);
    case CACTO_CAR_PARK: return launch_actor_grad<CACTO_CAR_PARK>(*p, actor_params, actor_params_T, critic_params, critic_params_T, state, term, inv_B, grad, actions, B, st);
    case CACTO_MANIPULATOR: return launch_actor_grad<CACTO_MANIPULATOR>(*p, actor_params, actor_params_T, critic_params, critic_params_T, state, term, inv_B, grad, actions, B, st);
    case CACTO_UR5: return launch_actor_grad<CACTO_UR5>(*p, actor_params, actor_params_T, critic_params, critic_params_T, state, term, inv_B, grad, actions, B, st);
    default: return CACTO_E_SYSTEM;
  }
}

// ---- deterministic variants (det.cuh): the same kernels with DET = true, in waves of at most CACTO_DET_MAX_SLICES CTAs
namespace cacto {

__global__ void __launch_bounds__(256) k_det_reduce(const float* __restrict__ part, int64_t slices, int64_t stride, int64_t n,
                                                    float* __restrict__ grad, float* __restrict__ loss) {
  pdl_wait();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n || (i == n && loss == nullptr)) return;
  float s = 0.f;
  for (int64_t j = 0; j < slices; ++j) s += part[j * stride + i];
  if (i < n) grad[i] += s;
  else loss[0] += s;
}

int det_reduce(const float* part, int64_t slices, int64_t n, float* grad, float* loss, cudaStream_t st) {
  if (cudaError_t le = launch_pdl(k_det_reduce, (unsigned)((n + 1 + 255) / 256), 256, 0, st, part, slices, det_stride(n), n, grad, loss)) return (int)le;
  CACTO_LAUNCH_CHECK();
  return 0;
}

static bool partials_ok(int64_t have, int64_t need) { return need >= 0 && have >= need; }

template <int S>
static int critic_grad_det_s(const cacto_sys_params& P, const float* cw, const float* cwT, const float* tw, float w_S, int mc, const float* state,
                             const float* state_next, const float* prtg, const float* dVdx, const float* done, const float* weights, float inv_B,
                             float* grad, float* rtg, float* V, float* Vt, float* loss, int64_t B, float* part, cudaStream_t st) {
  auto k = k_critic_grad<S, true>;
  const size_t smem = sizeof(CriticSmem<S>) + (UP_NT / 32) * sizeof(float);
  if (int e = smem_attr(k, smem)) return e;
  const int64_t n = CriticLayout(P.ns).total, tiles = (B + S - 1) / S, slices = det_slices(tiles), ns = P.ns;
  if (cudaError_t e = cudaMemsetAsync(part, 0, (size_t)(slices * det_stride(n)) * sizeof(float), st)) return (int)e;
  for (int64_t t0 = 0; t0 < tiles; t0 += slices) {
    const int64_t r0 = t0 * S, rows = min(B - r0, slices * S);
    if (cudaError_t le = launch_pdl(k, (unsigned)((rows + S - 1) / S), UP_NT, smem, st, P, cw, cwT, tw, w_S, mc, state + r0 * ns,
                                    state_next ? state_next + r0 * ns : nullptr, prtg + r0, dVdx ? dVdx + r0 * ns : nullptr, done ? done + r0 : nullptr,
                                    weights + r0, inv_B, part, rtg + r0, V + r0, Vt + r0, loss, rows))
      return (int)le;
    CACTO_LAUNCH_CHECK();
  }
  return det_reduce(part, slices, n, grad, loss, st);
}

template <int SYS, int S>
static int actor_grad_det_s(const cacto_sys_params& P, const float* aw, const float* awT, const float* cw, const float* cwT, const float* state,
                            const double* term, float inv_B, float* grad, float* actions, int64_t B, float* part, cudaStream_t st) {
  auto k = k_actor_grad<SYS, S, true>;
  if (int e = smem_attr(k, sizeof(ActorSmem<S>))) return e;
  const int64_t n = ActorLayout(P.ns, P.na).total, tiles = (B + S - 1) / S, slices = det_slices(tiles), ns = P.ns, na = P.na;
  if (cudaError_t e = cudaMemsetAsync(part, 0, (size_t)(slices * det_stride(n)) * sizeof(float), st)) return (int)e;
  for (int64_t t0 = 0; t0 < tiles; t0 += slices) {
    const int64_t r0 = t0 * S, rows = min(B - r0, slices * S);
    if (cudaError_t le = launch_pdl(k, (unsigned)((rows + S - 1) / S), UP_NT, sizeof(ActorSmem<S>), st, P, aw, awT, cw, cwT, state + r0 * ns, term + r0,
                                    inv_B, part, actions ? actions + r0 * na : nullptr, rows))
      return (int)le;
    CACTO_LAUNCH_CHECK();
  }
  return det_reduce(part, slices, n, grad, nullptr, st);
}

template <int SYS>
static int actor_grad_det(const cacto_sys_params& P, const float* aw, const float* awT, const float* cw, const float* cwT, const float* state,
                          const double* term, float inv_B, float* grad, float* actions, int64_t B, float* part, cudaStream_t st) {
  switch (pick_tile(B)) {
    case 16: return actor_grad_det_s<SYS, 16>(P, aw, awT, cw, cwT, state, term, inv_B, grad, actions, B, part, st);
    case 8: return actor_grad_det_s<SYS, 8>(P, aw, awT, cw, cwT, state, term, inv_B, grad, actions, B, part, st);
    case 4: return actor_grad_det_s<SYS, 4>(P, aw, awT, cw, cwT, state, term, inv_B, grad, actions, B, part, st);
    default: return actor_grad_det_s<SYS, 2>(P, aw, awT, cw, cwT, state, term, inv_B, grad, actions, B, part, st);
  }
}

}  // namespace cacto

extern "C" int64_t cacto_det_partials_floats(int32_t net, int64_t B, int32_t ns, int32_t na, int32_t nh1, int32_t nh2) {
  if (B < 0 || ns < 2 || ns > CACTO_MAX_NS || na < 1 || na > CACTO_MAX_NA) return CACTO_E_SIZE;
  int64_t n, tile;
  switch (net) {
    case CACTO_DET_CRITIC: n = CriticLayout(ns).total; tile = pick_tile(B); break;
    case CACTO_DET_ACTOR: n = ActorLayout(ns, na).total; tile = pick_tile(B); break;
    case CACTO_DET_ACTOR_WIDTH:
      if (nh1 < 1 || nh1 > CACTO_ACTOR_MAX_WIDTH || nh2 < 1 || nh2 > CACTO_ACTOR_MAX_WIDTH) return CACTO_E_SIZE;
      n = ActorLayout(ns, na, nh1, nh2).total; tile = actor_width_tile(B); break;
    case CACTO_DET_CRITIC_TC:      // tcgen05 engine: 3 / 2 regions of fixed-size slices, one per CTA of a <= 296-CTA grid over 128-sample tiles
    case CACTO_DET_ACTOR_TC: return (net == CACTO_DET_CRITIC_TC ? 3 : 2) * det_slices((B + 127) / 128) * det_tc_slice;
    default: return CACTO_E_SIZE;
  }
  return det_slices((B + tile - 1) / tile) * det_stride(n);
}

extern "C" int cacto_critic_grad_det(const cacto_sys_params* p, const float* critic_params, const float* critic_params_T,
                                     const float* target_params, float w_S, int mc, const float* state, const float* state_next,
                                     const float* partial_rtg, const float* dVdx, const float* done, const float* weights, float inv_B,
                                     float* grad, float* rtg, float* V, float* V_target_s, float* loss, int64_t B, float* partials,
                                     int64_t partials_floats, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (B < 0) return CACTO_E_SIZE;
  if (B == 0) return 0;
  if (!critic_params || !critic_params_T || !target_params || !state || !partial_rtg || !weights || !grad || !rtg || !V || !V_target_s || !partials)
    return CACTO_E_ARG;
  if (!mc && (!state_next || !done)) return CACTO_E_ARG;
  if (w_S != 0.f && !dVdx) return CACTO_E_ARG;
  if (!aligned16(critic_params) || !aligned16(critic_params_T) || !aligned16(target_params) || !aligned16(grad) || !aligned16(partials))
    return CACTO_E_ALIGN;
  if (!partials_ok(partials_floats, cacto_det_partials_floats(CACTO_DET_CRITIC, B, p->ns, p->na, 0, 0))) return CACTO_E_SIZE;
  cudaStream_t st = (cudaStream_t)stream;
  switch (pick_tile(B)) {
    case 16: return critic_grad_det_s<16>(*p, critic_params, critic_params_T, target_params, w_S, mc, state, state_next, partial_rtg, dVdx, done, weights,
                                          inv_B, grad, rtg, V, V_target_s, loss, B, partials, st);
    case 8: return critic_grad_det_s<8>(*p, critic_params, critic_params_T, target_params, w_S, mc, state, state_next, partial_rtg, dVdx, done, weights,
                                        inv_B, grad, rtg, V, V_target_s, loss, B, partials, st);
    case 4: return critic_grad_det_s<4>(*p, critic_params, critic_params_T, target_params, w_S, mc, state, state_next, partial_rtg, dVdx, done, weights,
                                        inv_B, grad, rtg, V, V_target_s, loss, B, partials, st);
    default: return critic_grad_det_s<2>(*p, critic_params, critic_params_T, target_params, w_S, mc, state, state_next, partial_rtg, dVdx, done, weights,
                                         inv_B, grad, rtg, V, V_target_s, loss, B, partials, st);
  }
}

extern "C" int cacto_actor_grad_det(const cacto_sys_params* p, const float* actor_params, const float* actor_params_T,
                                    const float* critic_params, const float* critic_params_T, const float* state, const double* term,
                                    float inv_B, float* grad, float* actions, int64_t B, float* partials, int64_t partials_floats, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (B < 0) return CACTO_E_SIZE;
  if (B == 0) return 0;
  if (!actor_params || !actor_params_T || !critic_params || !critic_params_T || !state || !term || !grad || !partials) return CACTO_E_ARG;
  if (!aligned16(actor_params) || !aligned16(actor_params_T) || !aligned16(critic_params) || !aligned16(critic_params_T) || !aligned16(grad) ||
      !aligned16(partials))
    return CACTO_E_ALIGN;
  if (!partials_ok(partials_floats, cacto_det_partials_floats(CACTO_DET_ACTOR, B, p->ns, p->na, 0, 0))) return CACTO_E_SIZE;
  cudaStream_t st = (cudaStream_t)stream;
  switch (p->system) {
    case CACTO_SINGLE_INTEGRATOR: return actor_grad_det<CACTO_SINGLE_INTEGRATOR>(*p, actor_params, actor_params_T, critic_params, critic_params_T, state, term, inv_B, grad, actions, B, partials, st);
    case CACTO_DOUBLE_INTEGRATOR: return actor_grad_det<CACTO_DOUBLE_INTEGRATOR>(*p, actor_params, actor_params_T, critic_params, critic_params_T, state, term, inv_B, grad, actions, B, partials, st);
    case CACTO_CAR: return actor_grad_det<CACTO_CAR>(*p, actor_params, actor_params_T, critic_params, critic_params_T, state, term, inv_B, grad, actions, B, partials, st);
    case CACTO_CAR_PARK: return actor_grad_det<CACTO_CAR_PARK>(*p, actor_params, actor_params_T, critic_params, critic_params_T, state, term, inv_B, grad, actions, B, partials, st);
    case CACTO_MANIPULATOR: return actor_grad_det<CACTO_MANIPULATOR>(*p, actor_params, actor_params_T, critic_params, critic_params_T, state, term, inv_B, grad, actions, B, partials, st);
    case CACTO_UR5: return actor_grad_det<CACTO_UR5>(*p, actor_params, actor_params_T, critic_params, critic_params_T, state, term, inv_B, grad, actions, B, partials, st);
    default: return CACTO_E_SYSTEM;
  }
}

extern "C" int cacto_actor_forward(const cacto_sys_params* p, const float* actor_params, const float* state, float* out, int64_t B,
                                   void* stream) {
  if (!p) return CACTO_E_ARG;
  if (B < 0) return CACTO_E_SIZE;
  if (B == 0) return 0;
  if (!actor_params || !state || !out) return CACTO_E_ARG;
  if (!aligned16(actor_params)) return CACTO_E_ALIGN;
  auto k = k_actor_forward<16>;
  if (int e = smem_attr(k, sizeof(EvalSmem<16>))) return e;
  k<<<(unsigned)((B + 15) / 16), UP_NT, sizeof(EvalSmem<16>), (cudaStream_t)stream>>>(*p, actor_params, state, out, B);
  CACTO_LAUNCH_CHECK();
  return 0;
}

extern "C" int cacto_critic_forward(const cacto_sys_params* p, const float* critic_params, const float* state, float* value,
                                    float* dV_ds, int64_t B, void* stream) {
  if (!p) return CACTO_E_ARG;
  if (B < 0) return CACTO_E_SIZE;
  if (B == 0) return 0;
  if (!critic_params || !state || !value) return CACTO_E_ARG;
  if (!aligned16(critic_params)) return CACTO_E_ALIGN;
  auto k = k_critic_forward<16>;
  if (int e = smem_attr(k, sizeof(EvalSmem<16>))) return e;
  k<<<(unsigned)((B + 15) / 16), UP_NT, sizeof(EvalSmem<16>), (cudaStream_t)stream>>>(*p, critic_params, state, value, dV_ds, B);
  CACTO_LAUNCH_CHECK();
  return 0;
}

// alpha_t = lr(step) sqrt(1 - b2^t) / (1 - b1^t), t = step + 1, evaluated on the device so that a captured
// CUDA graph of the update can be replayed without host-side scalars.  Also clears `zero_me` (loss accumulator).
__global__ void k_adam_schedule(long long* __restrict__ step, const float* __restrict__ boundaries, const float* __restrict__ values,
                                int nb, float beta1, float beta2, float* __restrict__ alpha_out, float* __restrict__ zero_me) {
  pdl_wait();
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const long long it = step[0];
  int k = 0;
  for (int i = 0; i < nb; ++i) k += (boundaries[i] < (float)it) ? 1 : 0;        // PiecewiseConstantDecay: values[#{b < step}]
  const float lr = values[k];
  const float t = (float)(it + 1);
  alpha_out[0] = lr * sqrtf(1.f - powf(beta2, t)) / (1.f - powf(beta1, t));
  step[0] = it + 1;
  if (zero_me != nullptr) zero_me[0] = 0.f;
}

// the schedules of the two optimizers of an update in ONE launch (a one-thread kernel costs a launch slot of ~2.7 us on the
// update's critical path, whatever it computes): lane 0 of warp 0 serves the first optimizer, lane 0 of warp 1 the second
struct AdamSched { long long* step; const float* boundaries; const float* values; int nb; float beta1, beta2; float* alpha_out; };
__global__ void k_adam_schedule2(AdamSched a, AdamSched b, float* __restrict__ zero_me) {
  pdl_wait();
  if (blockIdx.x != 0 || (threadIdx.x & 31) != 0 || threadIdx.x >= 64) return;
  const AdamSched& S = threadIdx.x == 0 ? a : b;
  const long long it = S.step[0];
  int k = 0;
  for (int i = 0; i < S.nb; ++i) k += (S.boundaries[i] < (float)it) ? 1 : 0;
  const float t = (float)(it + 1);
  S.alpha_out[0] = S.values[k] * sqrtf(1.f - powf(S.beta2, t)) / (1.f - powf(S.beta1, t));
  S.step[0] = it + 1;
  if (threadIdx.x == 0 && zero_me != nullptr) zero_me[0] = 0.f;
}

extern "C" int cacto_adam_schedule2(int64_t* step_a, const float* boundaries_a, const float* values_a, int32_t nb_a, float beta1_a, float beta2_a,
                                    float* alpha_a, int64_t* step_b, const float* boundaries_b, const float* values_b, int32_t nb_b, float beta1_b,
                                    float beta2_b, float* alpha_b, float* zero_or_null, void* stream) {
  if (!step_a || !values_a || !alpha_a || (nb_a > 0 && !boundaries_a) || nb_a < 0) return CACTO_E_ARG;
  if (!step_b || !values_b || !alpha_b || (nb_b > 0 && !boundaries_b) || nb_b < 0) return CACTO_E_ARG;
  if (step_a == step_b || alpha_a == alpha_b) return CACTO_E_ARG;
  AdamSched A = {reinterpret_cast<long long*>(step_a), boundaries_a, values_a, nb_a, beta1_a, beta2_a, alpha_a};
  AdamSched Bs = {reinterpret_cast<long long*>(step_b), boundaries_b, values_b, nb_b, beta1_b, beta2_b, alpha_b};
  if (cudaError_t le = launch_pdl(k_adam_schedule2, 1, 64, 0, (cudaStream_t)stream, A, Bs, zero_or_null)) return (int)le;
  CACTO_LAUNCH_CHECK();
  return 0;
}

extern "C" int cacto_adam_schedule(int64_t* step, const float* boundaries, const float* values, int32_t nb, float beta1, float beta2,
                                   float* alpha_out, float* zero_or_null, void* stream) {
  if (!step || !values || !alpha_out || (nb > 0 && !boundaries) || nb < 0) return CACTO_E_ARG;
  if (cudaError_t le = launch_pdl(k_adam_schedule, 1, 32, 0, (cudaStream_t)stream, reinterpret_cast<long long*>(step), boundaries, values, nb,
                                  beta1, beta2, alpha_out, zero_or_null))
    return (int)le;
  CACTO_LAUNCH_CHECK();
  return 0;
}

extern "C" int cacto_adam_step(float* params, float* grad, float* m, float* v, float alpha_t, const float* alpha_dev_or_null, float beta1, float beta2, float eps,
                               float* target_or_null, float tau, float* params_T_or_null, int32_t is_critic, int32_t ns, int32_t na,
                               int64_t n, void* stream) {
  if (!params || !grad || !m || !v) return CACTO_E_ARG;
  int64_t total = 0;
  LayerTable T = make_table(is_critic, ns, na, &total);
  if (params_T_or_null == nullptr) {          // no transposed copy to refresh (generic networks): any flat block of n parameters
    if (n < 0) return CACTO_E_SIZE;
    if (n == 0) return 0;
    T.n = 0;
  } else if (n != total) {
    return CACTO_E_SIZE;
  }
  if (cudaError_t le = launch_pdl(k_adam, (unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream, params, grad, m, v, alpha_t, alpha_dev_or_null,
                                  one_minus(beta1), one_minus(beta2), eps, target_or_null, make_float2(tau, one_minus(tau)), params_T_or_null, T, n))
    return (int)le;
  CACTO_LAUNCH_CHECK();
  return 0;
}

extern "C" int cacto_adam_step_peer(float* params, const float* const* peer_grads, uint32_t* const* peer_flags, int32_t world, int32_t rank,
                                    float* zero_other_or_null, int64_t n_other, float* m, float* v,
                                    const float* alpha_dev, float beta1, float beta2, float eps, float* target_or_null, float tau,
                                    float* params_T_or_null, int32_t is_critic, int32_t ns, int32_t na, int64_t n, int32_t max_ctas,
                                    void* stream) {
  if (max_ctas < 0) return CACTO_E_ARG;
  if (!params || !peer_grads || !peer_flags || !m || !v || !alpha_dev) return CACTO_E_ARG;
  if (world < 1 || world > CACTO_MAX_PEERS || rank < 0 || rank >= world || n_other < 0 || (n_other > 0 && !zero_other_or_null)) return CACTO_E_ARG;
  int64_t total = 0;
  LayerTable T = make_table(is_critic, ns, na, &total);
  if (params_T_or_null == nullptr) {
    if (n <= 0) return CACTO_E_SIZE;
    T.n = 0;
  } else if (n != total) {
    return CACTO_E_SIZE;
  }
  PeerTable R;
  R.world = world;
  R.rank = rank;
  for (int r = 0; r < CACTO_MAX_PEERS; ++r) {
    R.grad[r] = r < world ? peer_grads[r] : nullptr;
    R.flags[r] = r < world ? reinterpret_cast<unsigned*>(peer_flags[r]) : nullptr;
    if (r < world && (!R.grad[r] || !R.flags[r])) return CACTO_E_ARG;
  }
  int64_t ctas = (n + 255) / 256;
  if (max_ctas > 0 && ctas > max_ctas) ctas = max_ctas;
  if (cudaError_t le = launch_pdl(k_adam_peer, (unsigned)ctas, 256, 0, (cudaStream_t)stream, params, R, zero_other_or_null, n_other, m, v, alpha_dev,
                                  one_minus(beta1), one_minus(beta2), eps, target_or_null, make_float2(tau, one_minus(tau)), params_T_or_null, T, n))
    return (int)le;
  CACTO_LAUNCH_CHECK();
  return 0;
}

extern "C" int cacto_transpose_params(const float* params, float* params_T, int32_t is_critic, int32_t ns, int32_t na, void* stream) {
  if (!params || !params_T) return CACTO_E_ARG;
  int64_t total = 0;
  LayerTable T = make_table(is_critic, ns, na, &total);
  k_transpose<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(params, params_T, T, total);
  CACTO_LAUNCH_CHECK();
  return 0;
}
