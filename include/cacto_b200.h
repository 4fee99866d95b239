/* cacto_b200.h -- C ABI of libcacto_b200.so: the B200 (sm_100a) implementation of CACTO's
 * data-parallel learning hot path.
 *
 * The reference (nadimkanazi/cacto) is pure Python with no FFI of its own; its drop-in boundary is
 * the module API wired in main.py:145-151.  Every entry point below names the reference method(s)
 * whose arithmetic it replaces; the Python host in cacto_b200/ keeps those methods' names and
 * signatures and calls these symbols through ctypes (see INTEGRATION.md).
 *
 * Conventions (all entry points):
 *   - device pointers only, caller owns every buffer, nothing is allocated or freed here;
 *   - asynchronous on `stream` (a cudaStream_t passed as void*), no hidden synchronisation;
 *   - returns 0 on success, a negative CACTO_E_* on bad arguments, a positive cudaError_t on
 *     launch failure; never throws, never prints;
 *   - no global mutable state: system constants travel in the POD cacto_sys_params.
 *   - dtype: 0 = float32, 1 = float64.  layout: 0 = rows [B][width] (the reference's batch API),
 *     1 = structure-of-arrays [width][B] (coalesced; used by the rollout trajectories).
 */
#ifndef CACTO_B200_H
#define CACTO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CACTO_ABI_VERSION 1

enum { CACTO_E_ARG = -1, CACTO_E_SYSTEM = -2, CACTO_E_DTYPE = -3, CACTO_E_SIZE = -4, CACTO_E_ALIGN = -5 };

enum cacto_system {
  CACTO_SINGLE_INTEGRATOR = 0, /* environment.py:165 */
  CACTO_DOUBLE_INTEGRATOR = 1, /* environment.py:288 + urdf/double_integrator.urdf */
  CACTO_CAR = 2,               /* environment.py:364 */
  CACTO_CAR_PARK = 3,          /* environment.py:493 */
  CACTO_MANIPULATOR = 4,       /* environment.py:654 + urdf/planar_manipulator_3dof.urdf */
  CACTO_UR5 = 5                /* environment.py:736 + urdf/ur5_robot.urdf */
};

#define CACTO_MAX_NS 13
#define CACTO_MAX_NA 6
#define CACTO_MAX_JOINTS 6
#define CACTO_MAX_PEERS 8          /* GPUs of one box that share gradient blocks over NVLink peer memory */
#define CACTO_IPC_HANDLE_BYTES 64  /* sizeof(cudaIpcMemHandle_t) */

/* Serial chain extracted from the URDF (what Pinocchio builds in conf_*.py: RobotWrapper.BuildFromURDF). */
typedef struct {
  int32_t n;                            /* joints */
  int32_t jtype[CACTO_MAX_JOINTS];      /* 0 revolute, 1 prismatic */
  int32_t axis[CACTO_MAX_JOINTS];       /* 0 x, 1 y, 2 z */
  double p[CACTO_MAX_JOINTS][3];        /* joint origin in the parent frame */
  double R[CACTO_MAX_JOINTS][9];        /* fixed rotation parent->joint frame, row-major (rpy) */
  double mass[CACTO_MAX_JOINTS];
  double com[CACTO_MAX_JOINTS][3];
  double inertia[CACTO_MAX_JOINTS][6];  /* ixx iyy izz ixy ixz iyz about the COM */
  double ee_p[3];                       /* EE frame on the last link */
  double gravity;                       /* 9.81 */
} cacto_chain;

/* Everything the kernels read from conf_<system>.py. */
typedef struct {
  int32_t system;      /* enum cacto_system */
  int32_t nx, ns, na;  /* ns = nx + 1 (time is the last state) */
  int32_t normalize;   /* conf.NORMALIZE_INPUTS */
  int32_t pad_;
  double dt;
  double state_norm[CACTO_MAX_NS + 3];  /* conf.state_norm_arr (ns entries) */
  double u_max[CACTO_MAX_NA + 2];
  /* cost function (environment.py reward(), Appendix A.1 of SURVEY.md) */
  double scale, offset, alpha, alpha2, w_b;
  double target[3];
  double obs[18];            /* conf.obs_param */
  double L_delta, tau_delta, k_db;
  double check_points[20];   /* car_park body check points (10 x 2) */
  double w_running[8], w_terminal[8];
  cacto_chain chain;
} cacto_sys_params;

/* MLP parameter blocks: one contiguous float32 buffer per network, Keras order
 * [W1 (in x out, row-major), b1, W2, b2, ...].  Actor: ns->256->256->na (NeuralNetwork.py:51-63).
 * Critic 'sine': ns->64->64->128->128->1 (NeuralNetwork.py:95-108). */
int64_t cacto_actor_param_count(int32_t ns, int32_t na);
int64_t cacto_critic_param_count(int32_t ns);
int32_t cacto_abi_version(void);

/* ---- K1': Env.simulate_batch (environment.py:134-138; per system :235,:437,:584, robot_utils.py:399-405) */
int cacto_dyn_step(const cacto_sys_params* p, int dtype, int layout, const void* state, const void* action,
                   void* state_next, int64_t B, void* stream);

/* ---- K2: Env.derivative_batch (environment.py:140-144,93-109): Fu[B][ns][na], normalised, time row 0 */
int cacto_dyn_derivative(const cacto_sys_params* p, int dtype, int layout, const void* state, const void* action,
                         void* Fu, int64_t B, void* stream);

/* ---- K2: Env.augmented_derivative over a batch (environment.py:111-132,:221,:420,:567; caller TO.py:181):
 *      Fx[B][nx][nx], Fu[B][nx][na] */
int cacto_dyn_augmented(const cacto_sys_params* p, int dtype, int layout, const void* state, const void* action,
                        void* Fx, void* Fu, int64_t B, void* stream);

/* ---- Env.get_end_effector_position over a batch (environment.py:146-156,:245,:450,:597): ee[B][3] */
int cacto_ee_position(const cacto_sys_params* p, int dtype, int layout, const void* state, void* ee, int64_t B,
                      void* stream);

/* ---- Env.reward / reward_batch (environment.py:252-286 and twins; UR5 :780-816).
 *      weights[B][8] (fp64, conf.cost_weights_*), action may be NULL (reward(w, s)).
 *      ur5_plain_ucost != 0 selects UR5.reward's u.u control cost (quirk Q8) instead of the bounded one.
 *      reward[B]; dr_da[B][na] optional (NULL to skip) = d reward / d action (NeuralNetwork.py:199-204). */
int cacto_reward(const cacto_sys_params* p, int dtype, int layout, const double* weights, const void* state,
                 const void* action, int ur5_plain_ucost, void* reward, void* dr_da, int64_t B, void* stream);

/* ---- K1: RL_AC.create_TO_init over a batch (RL.py:197-233) fused with the actor forward
 *      (NeuralNetwork.py:130-138, utils.py:17-24) and Env.simulate.
 *      ics[B][ns] fp64; horizon[B] int32 (NSTEPS_SH per rollout, <= T_max); use_actor = (ep != 0).
 *      states  [T_max+1][ns][B] fp64 (SoA, time-major), controls [T_max][na][B] fp64,
 *      flags[B] int32: 1 ok, 0 NaN met (RL.py:229-231).  Entries past a rollout's horizon are left untouched.
 *      If reward_weights != NULL also writes rewards[T_max+1][B] = Env.step's reward at the current
 *      state/action with the running weights, terminal weights at the last knot (plot_utils.py:261-268). */
int cacto_rollout(const cacto_sys_params* p, const float* actor_params, int use_actor, const double* ics,
                  const int32_t* horizon, int32_t T_max, double* states, double* controls, int32_t* flags,
                  double* rewards, int64_t B, void* stream);

/* ---- K1 on tcgen05 tensor cores: same contract as cacto_rollout (use_actor = 1), with the 256x256 hidden layer
 *      computed by tcgen05.mma kind::tf32 with 3xTF32 operand splitting (fp32-class accuracy, accumulators in TMEM).
 *      w2img (cacto_actor_tc_image_floats() floats, 128-byte aligned, caller-owned) is the hi/lo-split, UMMA-laid-out
 *      image of the actor's W2 built by cacto_actor_tc_prepare; rebuild it whenever the actor changes. */
int64_t cacto_actor_tc_image_floats(void);
int cacto_actor_tc_prepare(const float* actor_params, int32_t ns, int32_t na, float* w2img, void* stream);
int cacto_rollout_tc(const cacto_sys_params* p, const float* actor_params, const float* w2img, const double* ics,
                     const int32_t* horizon, int32_t T_max, double* states, double* controls, int32_t* flags,
                     double* rewards, int64_t B, void* stream);

/* ---- K1 on tcgen05 at the fp16 rate (default rollout engine): same contract as cacto_rollout (use_actor = 1).
 *      The 256x256 hidden layer runs as 3 x tcgen05.mma kind::f16 per K-step on fp16 hi/lo operand pairs
 *      (a = a_hi + a_lo, w = w_hi + w_lo; a w ~= a_hi w_hi + a_hi w_lo + a_lo w_hi, fp32 accumulation in TMEM: the
 *      accuracy class of 3xTF32 at twice the rate) by persistent CTAs that keep two 128-rollout tiles in flight.
 *      Range limit: hidden activations beyond +-2047 overflow the fp16 high part; such a rollout is flagged failed.
 *      The five systems with ns <= 8 and na <= 3; any other, UR5 included, returns CACTO_E_SYSTEM (cacto_rollout_tc runs UR5).
 *      w2img (cacto_actor_tc16_image_bytes() bytes, 128-byte aligned, caller-owned) is the scaled, split, UMMA-laid-out
 *      image of the actor's W2 built by cacto_actor_tc16_prepare; rebuild it whenever the actor changes. */
int64_t cacto_actor_tc16_image_bytes(void);
int cacto_actor_tc16_prepare(const float* actor_params, int32_t ns, int32_t na, void* w2img, void* stream);
int cacto_rollout_tc16(const cacto_sys_params* p, const float* actor_params, const void* w2img, const double* ics,
                       const int32_t* horizon, int32_t T_max, double* states, double* controls, int32_t* flags,
                       double* rewards, int64_t B, void* stream);

/* ---- K6: TO_Casadi.backward_pass (TO.py:119-202) over a batch of ragged TO trajectories: the DDP value recursion that
 *      produces dVdx for the Sobolev critic (TO.py:109, main.py:237-240).  Trajectory e owns knots offsets[e] .. offsets[e+1]-1
 *      of states[n_knots][nx] (no time column, as TO.py:123-125) and controls[n_knots][na] (the row of a trajectory's last
 *      knot is ignored).  Per knot: A, B = Env.augmented_derivative (environment.py:111-132), l_x / l_xx = gradient / Hessian
 *      of the reward -CAMS.cost (environment_TO.py cost_fun; running weights, terminal weights at the last knot) by
 *      hyper-dual evaluation, l_u / l_uu of the bounded control cost; then Q_*, pinv(Q_uu + mu I), V_x, V_xx
 *      (TO.py:182-200).  V_x[n_knots][nx+1], last column 0 (TO.py:166).  workspace: caller-owned,
 *      cacto_backward_pass_workspace_bytes(nx, na, n_knots) bytes, 8-byte aligned. */
int64_t cacto_backward_pass_workspace_bytes(int32_t nx, int32_t na, int64_t n_knots);
int cacto_backward_pass(const cacto_sys_params* p, const int64_t* offsets, int32_t E, const double* states,
                        const double* controls, int64_t n_knots, double mu, void* workspace, double* V_x, void* stream);

/* ---- K7: the TO solve (TO.py:35-100 solves it with ipopt on the host) as batched iLQR on the GPU, an opt-in alternative.
 *      Problem, per trajectory e with knots offsets[e] .. offsets[e+1]-1 (T_e = knots - 1 controls): from x_0 = states[offsets[e]]
 *      (kept fixed) minimise over u_0 .. u_{T-1}
 *          J = sum_{k<T} c_run(x_k, u_k) + c_term(x_T),   x_{k+1} = Env.simulate(x_k, u_k) in fp64,
 *      c = -reward (running / terminal weights) with the bounded control cost a^2 + w_b (a/u_max)^10 for every system (UR5
 *      included): the cost K6 differentiates, with the sign flipped.  No hard bounds (the reference's TO has only the penalty).
 *      One iteration per trajectory still running: per-knot derivatives at the iterate (K6's knot code); a warp-per-trajectory
 *      backward recursion with a Cholesky factor of Q_uu + mu I (not positive definite at some knot: the pass fails, mu grows)
 *      giving k_t = -Quu~^-1 Q_u, K_t = -Quu~^-1 Q_ux and the expected change dV(a) = a dV1 + a^2/2 dV2 (dV1 = sum k'Q_u,
 *      dV2 = sum k'Q_uu k); CACTO_DDP_N_ALPHA closed-loop probes u = u_bar + a k + K (x - x_bar), a = 2^-j, cost only;
 *      then the largest a with (J - J(a)) >= CACTO_DDP_C1 (-dV(a)) is re-rolled with the same arithmetic and committed.
 *      mu: / CACTO_DDP_MU_FACTOR (floor CACTO_DDP_MU_MIN) on success, * CACTO_DDP_MU_FACTOR on failure.
 *      Status: CONVERGED when |dV(1)| < tol |J| (no step) or an accepted step improved J by < tol |J|; FAILED when mu exceeds
 *      CACTO_DDP_MU_MAX or the warm start's cost is not finite (the iterate is the last accepted one: the best).
 *      states[n_knots][nx] (no time column) and controls[n_knots][na] hold the iterate in place (the control row of a
 *      trajectory's last knot is not used); cost[E] fp64, status[E] int32, iters[E] int32.
 *      workspace: cacto_ddp_workspace_bytes(nx, na, n_knots, E) bytes, 8-byte aligned, caller-owned: per knot K6's block
 *      [l_x | l_xx | A | B | l_u | l_uu] followed by [k | K], then per trajectory CACTO_DDP_TRAJ_DOUBLES doubles
 *      [mu, dV1, dV2, backward ok, probe costs[CACTO_DDP_N_ALPHA], accepted alpha index of iterations 1..CACTO_DDP_HISTORY
 *      (j >= 0; CACTO_DDP_H_* otherwise)].
 *      cacto_ddp_init: re-simulates every iterate from x_0 (states written from knot 1 on), sets cost, status, iters = 0, mu.
 *      cacto_ddp_iterate: n_iter iterations, enqueued without host synchronisation; finished trajectories are skipped. */
#define CACTO_DDP_N_ALPHA 8
#define CACTO_DDP_C1 1e-4
#define CACTO_DDP_MU_INIT 1e-6
#define CACTO_DDP_MU_MIN 1e-9
#define CACTO_DDP_MU_MAX 1e10
#define CACTO_DDP_MU_FACTOR 10.0
#define CACTO_DDP_HISTORY 8
#define CACTO_DDP_TRAJ_DOUBLES 24
enum { CACTO_DDP_RUNNING = 0, CACTO_DDP_CONVERGED = 1, CACTO_DDP_FAILED = 2 };
enum { CACTO_DDP_H_BACKWARD_FAILED = -1, CACTO_DDP_H_NO_STEP = -2, CACTO_DDP_H_CONVERGED = -3, CACTO_DDP_H_NOT_RUN = -4 };
int64_t cacto_ddp_workspace_bytes(int32_t nx, int32_t na, int64_t n_knots, int32_t E);
int cacto_ddp_init(const cacto_sys_params* p, const int64_t* offsets, int32_t E, double* states, const double* controls,
                   int64_t n_knots, void* workspace, double* cost, int32_t* status, int32_t* iters, void* stream);
int cacto_ddp_iterate(const cacto_sys_params* p, const int64_t* offsets, int32_t E, double* states, double* controls,
                      int64_t n_knots, int32_t n_iter, double tol, void* workspace, double* cost, int32_t* status, int32_t* iters,
                      void* stream);

/* ---- plumbing for the host feeder (main.py:216-233 hands warm-starts to the TO pool): strided device-to-host copy of a
 *      column block, rows x width_bytes, on the copy engine. */
int cacto_copy2d_to_host(void* dst_host, int64_t dst_pitch, const void* src_dev, int64_t src_pitch, int64_t width_bytes,
                         int64_t rows, void* stream);
/*      The same for `slabs` stacked column blocks: slab k of the source has src_rows rows of which the first `rows` go to slab k of
 *      the destination (dst_rows rows); and the exact fp64 -> fp32 narrowing of the controls (fp32 actor outputs widened for the
 *      fp64 dynamics, RL.py:223).  Together: the compact transfer format of the warm-start hand-off (no time row, fp32 controls). */
int cacto_copy3d_to_host(void* dst_host, int64_t dst_pitch, int64_t dst_rows, const void* src_dev, int64_t src_pitch, int64_t src_rows,
                         int64_t width_bytes, int64_t rows, int64_t slabs, void* stream);
int cacto_narrow_f64_to_f32(const double* src, float* dst, int64_t n, void* stream);

/* ---- host helper of the PER sampler (replay_buffer.py:142-147: `random.random()` once per stratum): n draws from a copy of the
 *      interpreter's MT19937 state (random.getstate()[1]: 624 words + position), advanced in place -- same stream, same bits. */
int cacto_host_mt19937_random(uint32_t* state625, double* out, int64_t n);

/* ---- Generic dense networks: the critic variants of NeuralNetwork.py besides 'sine' (create_critic_elu :65-78,
 *      create_critic_sine_elu :80-93, create_critic_relu :110-128), or any stack of <= CACTO_MLP_MAX_LAYERS dense layers of
 *      <= 256 units (the actor of cacto_actor_grad_generic: <= CACTO_ACTOR_MAX_WIDTH units).  Parameter block in Keras order
 *      [W1 (in x out), b1, ...]; act[l] is the activation after layer l (the last one CACTO_ACT_LINEAR).  One CTA per sample
 *      (latency-oriented); same semantics, arguments and outputs as cacto_critic_forward / cacto_critic_grad / cacto_actor_grad, without the transposed parameter copies. */
#define CACTO_MLP_MAX_LAYERS 8
enum { CACTO_ACT_LINEAR = 0, CACTO_ACT_SIN = 1, CACTO_ACT_ELU = 2, CACTO_ACT_LEAKY = 3 };
typedef struct cacto_mlp_desc {
  int32_t n_layers;                          /* dense layers L */
  int32_t dims[CACTO_MLP_MAX_LAYERS + 1];    /* dims[0] = nb_state, dims[L] = outputs */
  int32_t act[CACTO_MLP_MAX_LAYERS];
} cacto_mlp_desc;
int cacto_mlp_forward_generic(const cacto_sys_params* p, const cacto_mlp_desc* d, const float* params, const float* state,
                              float* out, float* dout_ds, int64_t B, void* stream);
int cacto_critic_grad_generic(const cacto_sys_params* p, const cacto_mlp_desc* d, const float* critic_params,
                              const float* target_params, float w_S, int mc, const float* state, const float* state_next,
                              const float* partial_rtg, const float* dVdx, const float* done, const float* weights, float inv_B,
                              float* grad, float* rtg, float* V, float* V_target_s, float* loss, int64_t B, void* stream);
/* state_next = Env.simulate_batch(state, actor(state)), Fu = Env.derivative_batch (normalised, [B][ns][na]) and
 * dr_da = d reward_batch / d action come from cacto_dyn_step / cacto_dyn_derivative / cacto_reward (NeuralNetwork.py:185-204). */
int cacto_actor_grad_generic(const cacto_sys_params* p, const cacto_mlp_desc* d_actor, const float* actor_params,
                             const cacto_mlp_desc* d_critic, const float* critic_params, const float* state,
                             const float* state_next, const float* Fu, const float* dr_da, float inv_B, float* grad, int64_t B,
                             void* stream);

/* ---- The actor at any hidden width (conf.NH1 / conf.NH2; NeuralNetwork.py:51-63: ns -> nh1 -> nh2 -> na, LeakyReLU(0.3)),
 *      1 <= nh1, nh2 <= CACTO_ACTOR_MAX_WIDTH, on fp32 CUDA-core kernels that take the widths at run time (csrc/actor_width.cu).
 *      actor_params: the Keras-layout block of cacto_actor_width_param_count(ns, na, nh1, nh2) floats, 16-byte aligned; no
 *      transposed or prepared copy.  cacto_actor_width_param_count returns CACTO_E_SIZE for widths out of range.
 *      cacto_rollout_width: the contract of cacto_rollout with use_actor = 1 (RL.py:197-233; outputs may be pinned host memory).
 *      cacto_actor_forward_width: the contract of cacto_actor_forward (NeuralNetwork.py:130-138).
 *      cacto_actor_grad_width: the contract of cacto_actor_grad with the 'sine' critic (NeuralNetwork.py:180-232), one launch;
 *      grad is accumulated into. */
#define CACTO_ACTOR_MAX_WIDTH 512
int64_t cacto_actor_width_param_count(int32_t ns, int32_t na, int32_t nh1, int32_t nh2);
int cacto_rollout_width(const cacto_sys_params* p, const float* actor_params, int32_t nh1, int32_t nh2, const double* ics,
                        const int32_t* horizon, int32_t T_max, double* states, double* controls, int32_t* flags, double* rewards,
                        int64_t B, void* stream);
int cacto_actor_forward_width(const cacto_sys_params* p, const float* actor_params, int32_t nh1, int32_t nh2, const float* state,
                              float* out, int64_t B, void* stream);
int cacto_actor_grad_width(const cacto_sys_params* p, const float* actor_params, int32_t nh1, int32_t nh2, const float* critic_params,
                           const float* critic_params_T, const float* state, const double* term, float inv_B, float* grad,
                           float* actions /* [B][na] or NULL */, int64_t B, void* stream);

/* ---- N4: NN.eval over a batch (NeuralNetwork.py:130-138): out[B][na] (actor) / out[B][1] (critic) */
int cacto_actor_forward(const cacto_sys_params* p, const float* actor_params, const float* state, float* out,
                        int64_t B, void* stream);
int cacto_critic_forward(const cacto_sys_params* p, const float* critic_params, const float* state, float* value,
                         float* dV_ds /* [B][ns] or NULL */, int64_t B, void* stream);

/* ---- N6: NN.compute_critic_grad (NeuralNetwork.py:150-178).
 *      grad (float32, critic_param_count) is ACCUMULATED into (caller zeroes it); inv_B = 1/global batch.
 *      Outputs rtg[B], V[B], V_target_s[B] (the reference's return tuple). */
int cacto_critic_grad(const cacto_sys_params* p, const float* critic_params, const float* critic_params_T,
                      const float* target_params, float w_S, int mc, const float* state, const float* state_next,
                      const float* partial_rtg, const float* dVdx, const float* done, const float* weights,
                      float inv_B, float* grad, float* rtg, float* V, float* V_target_s, float* loss,
                      int64_t B, void* stream);

/* ---- N7: NN.compute_actor_grad (NeuralNetwork.py:180-232) incl. simulate_batch / derivative_batch /
 *      reward_batch inside the kernel.  term[B] fp64 as the reference keeps it. */
int cacto_actor_grad(const cacto_sys_params* p, const float* actor_params, const float* actor_params_T,
                     const float* critic_params, const float* critic_params_T, const float* state,
                     const double* term, float inv_B, float* grad, float* actions /* [B][na] or NULL */,
                     int64_t B, void* stream);

/* ---- N6 / N7 at large batch (B >= ~2 k: the PER batch 4096 and critic batch 16 384 of BASELINE configs 2, 3, 5) on tcgen05
 *      tensor cores (csrc/update_tc.cu): same arguments, outputs and accumulate-into-grad contract as cacto_critic_grad /
 *      cacto_actor_grad (NeuralNetwork.py:150-178 / :180-232), computed layer by layer over 128-sample tiles with fp16-split
 *      operands (fp32-class products, fp32 accumulation in TMEM) and batch-reduction GEMMs for the weight gradients.  No
 *      transposed parameter copies are needed.  workspace: caller-owned, 256-byte aligned, at least
 *      cacto_update_tc_workspace_bytes(B, ns, na) bytes (~19 KB per sample; both calls of an update may share it: the actor
 *      call reuses nothing of the critic call's contents). */
int64_t cacto_update_tc_workspace_bytes(int64_t B, int32_t ns, int32_t na);
int cacto_critic_grad_tc(const cacto_sys_params* p, const float* critic_params, const float* target_params, float w_S, int mc,
                         const float* state, const float* state_next, const float* partial_rtg, const float* dVdx,
                         const float* done, const float* weights, float inv_B, float* grad, float* rtg, float* V,
                         float* V_target_s, float* loss /* [1], accumulated, or NULL */, int64_t B, void* workspace,
                         int64_t workspace_bytes, void* stream);
int cacto_actor_grad_tc(const cacto_sys_params* p, const float* actor_params, const float* critic_params, const float* state,
                        const double* term, float inv_B, float* grad, float* actions /* [B][na] or NULL */, int64_t B,
                        void* workspace, int64_t workspace_bytes, void* stream);

/* ---- Deterministic N6 / N7 (NN(..., deterministic=True)): the contracts of cacto_critic_grad, cacto_actor_grad and
 *      cacto_actor_grad_width on the same fused fp32 kernels, but with every cross-CTA and cross-warp float sum taken in a fixed
 *      order, so that the same inputs give the same bits in grad, rtg, V, V_target_s and loss however the CTAs are scheduled.
 *      Each CTA (one tile of samples) writes its sums into its own slice of `partials`; one reduce kernel then adds the slices
 *      into grad in slice order, starting from 0.0f, and adds that into what grad holds (the accumulate-into-grad contract is
 *      kept; loss, if not NULL, receives the summed loss the same way).  Results differ from the default entry points only in
 *      summation order; they depend on the batch size (the tile size and the slice count follow it).
 *      partials: caller-owned, 16-byte aligned, at least cacto_det_partials_floats(net, B, ns, na, nh1, nh2) floats, where net is
 *      CACTO_DET_CRITIC, CACTO_DET_ACTOR (nh1, nh2 ignored) or CACTO_DET_ACTOR_WIDTH.  A slice holds the network's gradient block
 *      plus one loss partial (rounded up to 4 floats); there are min(tiles, CACTO_DET_MAX_SLICES) slices, so the workspace stops
 *      growing with B once the batch has more tiles than that (more tiles run as successive launches of at most
 *      CACTO_DET_MAX_SLICES CTAs, CTA j of each adding into slice j).  Critic and actor calls that may run concurrently need
 *      separate workspaces.  The size query returns CACTO_E_SIZE for out-of-range arguments.  No host synchronisation;
 *      capturable.
 *      cacto_critic_grad_tc_det / cacto_actor_grad_tc_det: the same for the tcgen05 engine (contracts of cacto_critic_grad_tc /
 *      cacto_actor_grad_tc, same workspace).  Its weight matrices are already summed in a fixed order; the bias and head column
 *      sums and the loss are summed per warp, then in warp order inside a CTA, and each CTA writes them into its own slice of
 *      `partials` (net CACTO_DET_CRITIC_TC / CACTO_DET_ACTOR_TC: at most 3 / 2 regions of min(B / 128 tiles, CACTO_DET_MAX_SLICES)
 *      slices of 648 floats, every entry written, so no clearing), which one reduce kernel adds into grad in slice order. */
#define CACTO_DET_MAX_SLICES 296
enum { CACTO_DET_CRITIC = 0, CACTO_DET_ACTOR = 1, CACTO_DET_ACTOR_WIDTH = 2, CACTO_DET_CRITIC_TC = 3, CACTO_DET_ACTOR_TC = 4 };
int64_t cacto_det_partials_floats(int32_t net, int64_t B, int32_t ns, int32_t na, int32_t nh1, int32_t nh2);
int cacto_critic_grad_det(const cacto_sys_params* p, const float* critic_params, const float* critic_params_T,
                          const float* target_params, float w_S, int mc, const float* state, const float* state_next,
                          const float* partial_rtg, const float* dVdx, const float* done, const float* weights,
                          float inv_B, float* grad, float* rtg, float* V, float* V_target_s, float* loss,
                          int64_t B, float* partials, int64_t partials_floats, void* stream);
int cacto_actor_grad_det(const cacto_sys_params* p, const float* actor_params, const float* actor_params_T,
                         const float* critic_params, const float* critic_params_T, const float* state,
                         const double* term, float inv_B, float* grad, float* actions /* [B][na] or NULL */,
                         int64_t B, float* partials, int64_t partials_floats, void* stream);
int cacto_actor_grad_width_det(const cacto_sys_params* p, const float* actor_params, int32_t nh1, int32_t nh2, const float* critic_params,
                               const float* critic_params_T, const float* state, const double* term, float inv_B, float* grad,
                               float* actions /* [B][na] or NULL */, int64_t B, float* partials, int64_t partials_floats, void* stream);
int cacto_critic_grad_tc_det(const cacto_sys_params* p, const float* critic_params, const float* target_params, float w_S, int mc,
                             const float* state, const float* state_next, const float* partial_rtg, const float* dVdx,
                             const float* done, const float* weights, float inv_B, float* grad, float* rtg, float* V,
                             float* V_target_s, float* loss /* [1], accumulated, or NULL */, int64_t B, void* workspace,
                             int64_t workspace_bytes, float* partials, int64_t partials_floats, void* stream);
int cacto_actor_grad_tc_det(const cacto_sys_params* p, const float* actor_params, const float* critic_params, const float* state,
                            const double* term, float inv_B, float* grad, float* actions /* [B][na] or NULL */, int64_t B,
                            void* workspace, int64_t workspace_bytes, float* partials, int64_t partials_floats, void* stream);

/* ---- N8/N9: tf.keras Adam step (RL.py:105,109; TF 2.11: m += (g-m)(1-b1), v += (g^2-v)(1-b2),
 *      p -= alpha_t m / (sqrt(v) + eps)) fused with the optional Polyak target update (RL.py:113-118:
 *      target = tau p + (1-tau) target), the refresh of the transposed copy and the zeroing of `grad`.
 *      alpha_t = lr(t-1) sqrt(1-b2^t)/(1-b1^t) is computed by the caller. n must equal the network's
 *      parameter count; with params_T_or_null == NULL (generic networks, no transposed copy) any flat block of n
 *      parameters is accepted and is_critic / ns / na are ignored. */
int cacto_adam_step(float* params, float* grad, float* m, float* v, float alpha_t, const float* alpha_dev_or_null,
                    float beta1, float beta2, float eps, float* target_or_null, float tau, float* params_T_or_null,
                    int32_t is_critic, int32_t ns, int32_t na, int64_t n, void* stream);

/* Device-side learning-rate schedule for CUDA-graph replays of the update: reads the step counter, writes
 * alpha_out[0] = values[#{boundaries < step}] sqrt(1-b2^t)/(1-b1^t) with t = step+1 (PiecewiseConstantDecay,
 * RL.py:82-85; nb = 0 for a constant rate values[0]), increments the counter and clears zero_or_null[0]. */
int cacto_adam_schedule(int64_t* step, const float* boundaries, const float* values, int32_t nb, float beta1,
                        float beta2, float* alpha_out, float* zero_or_null, void* stream);
/* The same for the two optimizers of an update (critic: _a, actor: _b) in one launch: RL_AC.update runs both Adam steps
 * (RL.py:101-111), and at the reference's batch of 64 every launch on the update's critical path is 4 % of it. */
int cacto_adam_schedule2(int64_t* step_a, const float* boundaries_a, const float* values_a, int32_t nb_a, float beta1_a,
                         float beta2_a, float* alpha_a, int64_t* step_b, const float* boundaries_b, const float* values_b,
                         int32_t nb_b, float beta1_b, float beta2_b, float* alpha_b, float* zero_or_null, void* stream);

/* ---- Data-parallel update (SURVEY.md 8e; the reference is single-GPU, main.py:59): cacto_adam_step with the gradient
 *      all-reduce fused in over NVLink peer memory.  peer_grads[r] / peer_flags[r] (HOST arrays of `world` device pointers)
 *      are rank r's gradient block of this network (n floats) and its flag row (32 zero-initialised uint32: CACTO_MAX_PEERS
 *      arrival words, a launch counter, a CTA ticket), both inside regions obtained from cacto_peer_alloc and mapped with
 *      cacto_peer_open; entry [rank] is the caller's own.  Every rank must issue the same sequence of calls.  The kernel
 *      announces its launch number to every peer, waits for all of them, sums the
 *      blocks in rank order (bit-identical replicas) and applies the step.  It does NOT clear the caller's gradient block
 *      (peers may still read it); it clears zero_other_or_null[0..n_other), the block of the network whose step precedes
 *      this one (critic and actor steps alternate, RL.py:104-109).  max_ctas > 0 bounds the CTAs of the launch (grid-stride
 *      over the parameters; 0 = one thread per parameter): the CTAs spin while they wait, which matters only when several
 *      ranks share one device, as the single-GPU test does.  Traps after 20 s if a peer never arrives. */
int cacto_adam_step_peer(float* params, const float* const* peer_grads, uint32_t* const* peer_flags, int32_t world,
                         int32_t rank, float* zero_other_or_null, int64_t n_other, float* m,
                         float* v, const float* alpha_dev, float beta1, float beta2, float eps, float* target_or_null,
                         float tau, float* params_T_or_null, int32_t is_critic, int32_t ns, int32_t na, int64_t n,
                         int32_t max_ctas, void* stream);

/* Peer-memory regions: cudaMalloc'ed (zero-filled) blocks that other processes of the box map through CUDA IPC.
 * export writes CACTO_IPC_HANDLE_BYTES bytes; open maps a handle received from another process (peer access over
 * NVLink is enabled lazily) and close unmaps it.  Host-synchronous; not for use inside stream capture. */
int cacto_peer_alloc(int64_t bytes, void** dev_ptr_out);
int cacto_peer_free(void* dev_ptr);
int cacto_peer_export(void* dev_ptr, void* handle_out);
int cacto_peer_open(const void* handle, void** dev_ptr_out);
int cacto_peer_close(void* dev_ptr);

/* Rebuild the per-layer transposed copy of a parameter block (W^T per layer, biases copied). */
int cacto_transpose_params(const float* params, float* params_T, int32_t is_critic, int32_t ns, int32_t na,
                           void* stream);

/* ---- R3/K4: segment_tree.py.  Trees are fp64 arrays of 2*capacity nodes, root at 1.
 *      update: tree[idx[i]] = value[i] in batch order (last duplicate wins), then every touched ancestor is
 *      recomputed level by level (SegmentTree.__setitem__, segment_tree.py:76-86).  Either tree may be NULL. */
int cacto_segtree_update(double* sum_tree, double* min_tree, int32_t capacity, const int64_t* idx,
                         const double* value, int32_t n, int32_t* stamp /* [capacity] workspace, all -1 */,
                         void* stream);
/* SumSegmentTree.sum(start, end) / MinSegmentTree.min(start, end): out[0] = sum, out[1] = min,
 * Python slice semantics of segment_tree.py:51-74 (end exclusive, negative end wraps). */
int cacto_segtree_reduce(const double* sum_tree, const double* min_tree, int32_t capacity, int32_t start,
                         int32_t end, double* out, void* stream);
/* PrioritizedReplayBuffer._sample_proportional (replay_buffer.py:139-157) + the leaf read of :175:
 * uniforms[n] are the host's random.random() draws; idx[n] int64, leaf[n] fp64 = sum_tree[idx],
 * totals[0] = sum(0, max_idx-1) used for the strata, totals[1] = sum(), totals[2] = min(). */
int cacto_segtree_sample(const double* sum_tree, const double* min_tree, int32_t capacity, int32_t max_idx,
                         const double* uniforms, int32_t n, int64_t* idx, double* leaf, double* totals,
                         void* stream);

/* SumSegmentTree.find_prefixsum_idx (segment_tree.py:105-131) for n given prefix sums. */
int cacto_segtree_find(const double* sum_tree, int32_t capacity, const double* prefix, int32_t n, int64_t* idx,
                       void* stream);

/* Host-side helper of PrioritizedReplayBuffer.update_priorities (replay_buffer.py:210-216): out[i] = pow(x[i], exponent) with
 * the C library's pow -- what CPython's `priority ** alpha` evaluates -- on HOST arrays (the one entry point that takes host
 * pointers and launches nothing: the bits of p ** alpha must be the host libm's for the trees to stay bit-exact). */
int cacto_host_pow(const double* x_host, double exponent, double* out_host, int64_t n);

/* ---- R1/R2: gather of sampled rows (replay_buffer.py:47-61,178-188): storage[cap][3ns+3] fp64 ->
 *      float32 blocks; term stays fp64.  exp_counter (fp64[cap]) is incremented once per distinct index
 *      when non-NULL (replay_buffer.py:174). */
int cacto_buffer_gather(const double* storage, int32_t ns, const int64_t* idx, int32_t n, float* state,
                        float* partial_rtg, float* state_next, float* dVdx, float* done, double* term,
                        double* exp_counter, int32_t* stamp, void* stream);

/* ---- G1/K5: RL_AC.RL_Solve windows (RL.py:173-187) for a ragged batch of trajectories.
 *      offsets[E+1] (knot offsets, trajectory e has T_e+1 = offsets[e+1]-offsets[e] knots),
 *      rwrd[total] fp64, states[total][ns] fp64 ->
 *      partial[total], total_rtg[total] (float32-rounded, stored fp64), s_next[total][ns], done[total],
 *      term[total], ep_return[E]. */
int cacto_rtg_window(const int64_t* offsets, int32_t E, const double* rwrd, const double* states, int32_t ns,
                     int32_t nsteps_td, int32_t mc, double* partial, double* total_rtg, double* s_next,
                     double* done, double* term, double* ep_return, void* stream);

/* ---- measurement only (bench.py): blocks x 256 threads each issue iters x 16 independent-chain fp32 FMAs;
 *      flops = blocks * 256 * iters * 16 * 2.  The in-run FP32-FMA roofline denominator (SURVEY.md 8d). */
int cacto_peak_fma_fp32(float* out, int32_t iters, int32_t blocks, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CACTO_B200_H */
