// torch_ops.cpp -- PyTorch custom-op shims over the C ABI of libcacto_b200.so (include/cacto_b200.h): TORCH_LIBRARY(cacto, ...).
//
// north_star / SURVEY.md 8b: "the host calls CUDA through a thin C-ABI layer exposed as PyTorch custom ops".  Every op takes torch
// tensors, checks device / dtype / contiguity / element count, passes raw pointers and the CURRENT CUDA stream to the extern "C" symbol
// of the same name and turns a non-zero return code into a RuntimeError (TORCH_CHECK).  Nothing is computed here and no torch
// type crosses the C boundary.  The system constants (cacto_sys_params, a POD) travel as a CPU uint8 tensor holding the struct's
// bytes.  Outputs are pre-sized by the caller (mutable arguments), exactly as the C ABI wants them.
// Built in-tree by cacto_b200/build.py into cacto_b200/libcacto_b200_torch.so; loaded by cacto_b200/ops.py.
#include <c10/cuda/CUDAStream.h>
#include <torch/library.h>
#include <ATen/ATen.h>
#include "cacto_b200.h"

namespace {

using at::Tensor;
using c10::optional;

const cacto_sys_params* sys(const Tensor& p) {
  TORCH_CHECK(p.device().is_cpu() && p.scalar_type() == at::kByte && p.is_contiguous() && p.numel() == (int64_t)sizeof(cacto_sys_params),
              "cacto: system parameters must be a CPU uint8 tensor of sizeof(cacto_sys_params) = ", sizeof(cacto_sys_params), " bytes");
  return reinterpret_cast<const cacto_sys_params*>(p.data_ptr());
}
void* stream() { return (void*)c10::cuda::getCurrentCUDAStream().stream(); }
void* dev(const Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda() && t.is_contiguous(), "cacto: ", name, " must be a contiguous CUDA tensor");
  return t.data_ptr();
}
void* dev(const Tensor& t, at::ScalarType ty, const char* name) {
  TORCH_CHECK(t.scalar_type() == ty, "cacto: ", name, " has dtype ", t.scalar_type(), ", expected ", ty);
  return dev(t, name);
}
void* opt(const optional<Tensor>& t, at::ScalarType ty, const char* name) { return t.has_value() ? dev(*t, ty, name) : nullptr; }
// element counts: the C ABI takes bare pointers, so a tensor of the wrong size would be read or written out of bounds on the device
void need(const Tensor& t, int64_t n, const char* name) {
  TORCH_CHECK(t.numel() == n, "cacto: ", name, " has ", t.numel(), " elements, expected ", n);
}
void need(const optional<Tensor>& t, int64_t n, const char* name) {
  if (t.has_value()) need(*t, n, name);
}
void need_at_least(const Tensor& t, int64_t n, const char* name) {
  TORCH_CHECK(t.numel() >= n, "cacto: ", name, " has ", t.numel(), " elements, at least ", n, " needed");
}
// batch size of a [B][ns] (layout 0) or [ns][B] (layout 1) state block
int64_t batch_of(const Tensor& state, int64_t layout, int64_t ns) {
  TORCH_CHECK(state.dim() == 2 && state.size(layout ? 0 : 1) == ns, "cacto: state must be [B][", ns, "] (layout 0) or [", ns, "][B] (layout 1)");
  return state.size(layout ? 1 : 0);
}
int64_t rows_of(const Tensor& state, int64_t ns, const char* name) {
  TORCH_CHECK(state.dim() == 2 && state.size(1) == ns, "cacto: ", name, " must be [B][", ns, "]");
  return state.size(0);
}
int dtype_code(const Tensor& t) {
  TORCH_CHECK(t.scalar_type() == at::kFloat || t.scalar_type() == at::kDouble, "cacto: float32 or float64 expected");
  return t.scalar_type() == at::kDouble ? 1 : 0;
}
void ok(int rc, const char* what) {
  TORCH_CHECK(rc >= 0, "cacto_", what, ": ", rc == CACTO_E_ARG ? "bad argument" : rc == CACTO_E_SYSTEM ? "unknown system" : rc == CACTO_E_DTYPE ? "unsupported dtype"
                                              : rc == CACTO_E_SIZE ? "bad size" : "misaligned buffer");
  TORCH_CHECK(rc == 0, "cacto_", what, ": CUDA error ", rc);
}
#define F32 at::kFloat
#define F64 at::kDouble

// ---- environment (K1', K2, reward, EE)
void dyn_step(const Tensor& p, int64_t layout, const Tensor& state, const Tensor& action, Tensor out) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = batch_of(state, layout, P_->ns);
  need(action, B * P_->na, "action"); need(out, B * P_->ns, "out");
  ok(cacto_dyn_step(P_, dtype_code(state), (int)layout, dev(state, "state"), dev(action, state.scalar_type(), "action"), dev(out, state.scalar_type(), "out"), B,
                    stream()), "dyn_step");
}
void dyn_derivative(const Tensor& p, int64_t layout, const Tensor& state, const Tensor& action, Tensor Fu) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = batch_of(state, layout, P_->ns);
  need(action, B * P_->na, "action"); need(Fu, B * P_->ns * P_->na, "Fu");
  ok(cacto_dyn_derivative(P_, dtype_code(state), (int)layout, dev(state, "state"), dev(action, state.scalar_type(), "action"), dev(Fu, state.scalar_type(), "Fu"), B,
                          stream()), "dyn_derivative");
}
void dyn_augmented(const Tensor& p, int64_t layout, const Tensor& state, const Tensor& action, Tensor Fx, Tensor Fu) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = batch_of(state, layout, P_->ns);
  need(action, B * P_->na, "action"); need(Fx, B * P_->nx * P_->nx, "Fx"); need(Fu, B * P_->nx * P_->na, "Fu");
  ok(cacto_dyn_augmented(P_, dtype_code(state), (int)layout, dev(state, "state"), dev(action, state.scalar_type(), "action"), dev(Fx, state.scalar_type(), "Fx"),
                         dev(Fu, state.scalar_type(), "Fu"), B, stream()), "dyn_augmented");
}
void ee_position(const Tensor& p, int64_t layout, const Tensor& state, Tensor ee) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = batch_of(state, layout, P_->ns);
  need(ee, B * 3, "ee");
  ok(cacto_ee_position(P_, dtype_code(state), (int)layout, dev(state, "state"), dev(ee, state.scalar_type(), "ee"), B, stream()), "ee_position");
}
void reward(const Tensor& p, int64_t layout, const Tensor& weights, const Tensor& state, const optional<Tensor>& action, int64_t ur5_plain_ucost, Tensor r,
            const optional<Tensor>& dr_da) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = batch_of(state, layout, P_->ns);
  need(weights, B * 8, "weights"); need(action, B * P_->na, "action"); need(r, B, "reward"); need(dr_da, B * P_->na, "dr_da");
  ok(cacto_reward(P_, dtype_code(state), (int)layout, (const double*)dev(weights, F64, "weights"), dev(state, "state"), opt(action, state.scalar_type(), "action"),
                  (int)ur5_plain_ucost, dev(r, state.scalar_type(), "reward"), opt(dr_da, state.scalar_type(), "dr_da"), B, stream()), "reward");
}

// ---- rollouts (K1)
void rollout(const Tensor& p, const optional<Tensor>& actor, int64_t use_actor, const Tensor& ics, const Tensor& horizon, int64_t T_max, Tensor states, Tensor controls,
             Tensor flags, const optional<Tensor>& rewards) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(ics, P_->ns, "ics");
  TORCH_CHECK(T_max >= 0, "cacto: T_max < 0");
  if (actor.has_value()) need(*actor, cacto_actor_param_count(P_->ns, P_->na), "actor");
  need(horizon, B, "horizon"); need(states, (T_max + 1) * P_->ns * B, "states"); need(controls, T_max * P_->na * B, "controls"); need(flags, B, "flags");
  need(rewards, (T_max + 1) * B, "rewards");
  ok(cacto_rollout(P_, (const float*)opt(actor, F32, "actor"), (int)use_actor, (const double*)dev(ics, F64, "ics"), (const int32_t*)dev(horizon, at::kInt, "horizon"),
                   (int32_t)T_max, (double*)dev(states, F64, "states"), (double*)dev(controls, F64, "controls"), (int32_t*)dev(flags, at::kInt, "flags"),
                   (double*)opt(rewards, F64, "rewards"), B, stream()), "rollout");
}
void actor_tc16_prepare(const Tensor& actor, int64_t ns, int64_t na, Tensor w2img) {
  need(actor, cacto_actor_param_count((int32_t)ns, (int32_t)na), "actor"); need_at_least(w2img, cacto_actor_tc16_image_bytes(), "w2img");
  ok(cacto_actor_tc16_prepare((const float*)dev(actor, F32, "actor"), (int32_t)ns, (int32_t)na, dev(w2img, at::kByte, "w2img"), stream()), "actor_tc16_prepare");
}
void rollout_tc16(const Tensor& p, const Tensor& actor, const Tensor& w2img, const Tensor& ics, const Tensor& horizon, int64_t T_max, Tensor states, Tensor controls,
                  Tensor flags, const optional<Tensor>& rewards) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(ics, P_->ns, "ics");
  TORCH_CHECK(T_max >= 0, "cacto: T_max < 0");
  need(actor, cacto_actor_param_count(P_->ns, P_->na), "actor"); need_at_least(w2img, cacto_actor_tc16_image_bytes(), "w2img");
  need(horizon, B, "horizon"); need(states, (T_max + 1) * P_->ns * B, "states"); need(controls, T_max * P_->na * B, "controls"); need(flags, B, "flags");
  need(rewards, (T_max + 1) * B, "rewards");
  ok(cacto_rollout_tc16(P_, (const float*)dev(actor, F32, "actor"), dev(w2img, at::kByte, "w2img"), (const double*)dev(ics, F64, "ics"),
                        (const int32_t*)dev(horizon, at::kInt, "horizon"), (int32_t)T_max, (double*)dev(states, F64, "states"), (double*)dev(controls, F64, "controls"),
                        (int32_t*)dev(flags, at::kInt, "flags"), (double*)opt(rewards, F64, "rewards"), B, stream()), "rollout_tc16");
}

// ---- the actor at any hidden width (K1, N4, N7 of csrc/actor_width.cu)
int64_t actor_width_count(const cacto_sys_params* P_, int64_t nh1, int64_t nh2) {
  const int64_t n = cacto_actor_width_param_count(P_->ns, P_->na, (int32_t)nh1, (int32_t)nh2);
  TORCH_CHECK(n > 0, "cacto: actor widths (", nh1, ", ", nh2, ") outside 1..", CACTO_ACTOR_MAX_WIDTH);
  return n;
}
void rollout_width(const Tensor& p, const Tensor& actor, int64_t nh1, int64_t nh2, const Tensor& ics, const Tensor& horizon, int64_t T_max, Tensor states,
                   Tensor controls, Tensor flags, const optional<Tensor>& rewards) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(ics, P_->ns, "ics");
  TORCH_CHECK(T_max >= 0, "cacto: T_max < 0");
  need(actor, actor_width_count(P_, nh1, nh2), "actor");
  need(horizon, B, "horizon"); need(states, (T_max + 1) * P_->ns * B, "states"); need(controls, T_max * P_->na * B, "controls"); need(flags, B, "flags");
  need(rewards, (T_max + 1) * B, "rewards");
  ok(cacto_rollout_width(P_, (const float*)dev(actor, F32, "actor"), (int32_t)nh1, (int32_t)nh2, (const double*)dev(ics, F64, "ics"),
                         (const int32_t*)dev(horizon, at::kInt, "horizon"), (int32_t)T_max, (double*)dev(states, F64, "states"), (double*)dev(controls, F64, "controls"),
                         (int32_t*)dev(flags, at::kInt, "flags"), (double*)opt(rewards, F64, "rewards"), B, stream()), "rollout_width");
}
void actor_forward_width(const Tensor& p, const Tensor& actor, int64_t nh1, int64_t nh2, const Tensor& state, Tensor out) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(state, P_->ns, "state");
  need(actor, actor_width_count(P_, nh1, nh2), "actor"); need(out, B * P_->na, "out");
  ok(cacto_actor_forward_width(P_, (const float*)dev(actor, F32, "actor"), (int32_t)nh1, (int32_t)nh2, (const float*)dev(state, F32, "state"),
                               (float*)dev(out, F32, "out"), B, stream()), "actor_forward_width");
}
void actor_grad_width(const Tensor& p, const Tensor& actor, int64_t nh1, int64_t nh2, const Tensor& critic, const Tensor& critic_T, const Tensor& state,
                      const Tensor& term, double inv_B, Tensor grad, const optional<Tensor>& actions) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(state, P_->ns, "state"), nact = actor_width_count(P_, nh1, nh2), nc = cacto_critic_param_count(P_->ns);
  need(actor, nact, "actor"); need(grad, nact, "grad"); need(critic, nc, "critic"); need(critic_T, nc, "critic_T"); need(term, B, "term");
  need(actions, B * P_->na, "actions");
  ok(cacto_actor_grad_width(P_, (const float*)dev(actor, F32, "actor"), (int32_t)nh1, (int32_t)nh2, (const float*)dev(critic, F32, "critic"),
                            (const float*)dev(critic_T, F32, "critic_T"), (const float*)dev(state, F32, "state"), (const double*)dev(term, F64, "term"), (float)inv_B,
                            (float*)dev(grad, F32, "grad"), (float*)opt(actions, F32, "actions"), B, stream()), "actor_grad_width");
}

// ---- networks (N4, N6-N9)
void actor_forward(const Tensor& p, const Tensor& actor, const Tensor& state, Tensor out) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(state, P_->ns, "state");
  need(actor, cacto_actor_param_count(P_->ns, P_->na), "actor"); need(out, B * P_->na, "out");
  ok(cacto_actor_forward(P_, (const float*)dev(actor, F32, "actor"), (const float*)dev(state, F32, "state"), (float*)dev(out, F32, "out"), B, stream()),
     "actor_forward");
}
void critic_forward(const Tensor& p, const Tensor& critic, const Tensor& state, Tensor value, const optional<Tensor>& dV_ds) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(state, P_->ns, "state");
  need(critic, cacto_critic_param_count(P_->ns), "critic"); need(value, B, "value"); need(dV_ds, B * P_->ns, "dV_ds");
  ok(cacto_critic_forward(P_, (const float*)dev(critic, F32, "critic"), (const float*)dev(state, F32, "state"), (float*)dev(value, F32, "value"),
                          (float*)opt(dV_ds, F32, "dV_ds"), B, stream()), "critic_forward");
}
void critic_grad(const Tensor& p, const Tensor& critic, const Tensor& critic_T, const Tensor& target, double w_S, int64_t mc, const Tensor& state,
                 const optional<Tensor>& state_next, const Tensor& prtg, const optional<Tensor>& dVdx, const optional<Tensor>& done, const Tensor& weights, double inv_B,
                 Tensor grad, Tensor rtg, Tensor V, Tensor Vt, const optional<Tensor>& loss) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(state, P_->ns, "state"), nc = cacto_critic_param_count(P_->ns);
  need(critic, nc, "critic"); need(target, nc, "target"); need(grad, nc, "grad");
  need(state_next, B * P_->ns, "state_next"); need(prtg, B, "partial_rtg"); need(dVdx, B * P_->ns, "dVdx"); need(done, B, "done"); need(weights, B, "weights");
  need(rtg, B, "rtg"); need(V, B, "V"); need(Vt, B, "V_target"); need(loss, 1, "loss");
  need(critic_T, nc, "critic_T");
  ok(cacto_critic_grad(P_, (const float*)dev(critic, F32, "critic"), (const float*)dev(critic_T, F32, "critic_T"), (const float*)dev(target, F32, "target"), (float)w_S,
                       (int)mc, (const float*)dev(state, F32, "state"), (const float*)opt(state_next, F32, "state_next"), (const float*)dev(prtg, F32, "partial_rtg"),
                       (const float*)opt(dVdx, F32, "dVdx"), (const float*)opt(done, F32, "done"), (const float*)dev(weights, F32, "weights"), (float)inv_B,
                       (float*)dev(grad, F32, "grad"), (float*)dev(rtg, F32, "rtg"), (float*)dev(V, F32, "V"), (float*)dev(Vt, F32, "V_target"), (float*)opt(loss, F32, "loss"),
                       B, stream()), "critic_grad");
}
void actor_grad(const Tensor& p, const Tensor& actor, const Tensor& actor_T, const Tensor& critic, const Tensor& critic_T, const Tensor& state, const Tensor& term,
                double inv_B, Tensor grad, const optional<Tensor>& actions) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(state, P_->ns, "state"), nact = cacto_actor_param_count(P_->ns, P_->na);
  need(actor, nact, "actor"); need(grad, nact, "grad"); need(critic, cacto_critic_param_count(P_->ns), "critic"); need(term, B, "term"); need(actions, B * P_->na, "actions");
  need(actor_T, nact, "actor_T"); need(critic_T, cacto_critic_param_count(P_->ns), "critic_T");
  ok(cacto_actor_grad(P_, (const float*)dev(actor, F32, "actor"), (const float*)dev(actor_T, F32, "actor_T"), (const float*)dev(critic, F32, "critic"),
                      (const float*)dev(critic_T, F32, "critic_T"), (const float*)dev(state, F32, "state"), (const double*)dev(term, F64, "term"), (float)inv_B,
                      (float*)dev(grad, F32, "grad"), (float*)opt(actions, F32, "actions"), B, stream()), "actor_grad");
}
// ---- deterministic gradients (fixed-order sums through a partials workspace of det_partials_floats elements)
int64_t det_partials_floats(int64_t net, int64_t B, int64_t ns, int64_t na, int64_t nh1, int64_t nh2) {
  return cacto_det_partials_floats((int32_t)net, B, (int32_t)ns, (int32_t)na, (int32_t)nh1, (int32_t)nh2);
}
int64_t det_need(int32_t net, int64_t B, const cacto_sys_params* P_, int64_t nh1, int64_t nh2, const Tensor& partials) {
  const int64_t n = cacto_det_partials_floats(net, B, P_->ns, P_->na, (int32_t)nh1, (int32_t)nh2);
  TORCH_CHECK(n >= 0, "cacto: no deterministic workspace size for these arguments");
  need_at_least(partials, n, "partials");
  return partials.numel();
}
void critic_grad_det(const Tensor& p, const Tensor& critic, const Tensor& critic_T, const Tensor& target, double w_S, int64_t mc, const Tensor& state,
                     const optional<Tensor>& state_next, const Tensor& prtg, const optional<Tensor>& dVdx, const optional<Tensor>& done, const Tensor& weights,
                     double inv_B, Tensor grad, Tensor rtg, Tensor V, Tensor Vt, const optional<Tensor>& loss, Tensor partials) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(state, P_->ns, "state"), nc = cacto_critic_param_count(P_->ns);
  need(critic, nc, "critic"); need(target, nc, "target"); need(grad, nc, "grad");
  need(state_next, B * P_->ns, "state_next"); need(prtg, B, "partial_rtg"); need(dVdx, B * P_->ns, "dVdx"); need(done, B, "done"); need(weights, B, "weights");
  need(rtg, B, "rtg"); need(V, B, "V"); need(Vt, B, "V_target"); need(loss, 1, "loss");
  need(critic_T, nc, "critic_T");
  const int64_t np = det_need(CACTO_DET_CRITIC, B, P_, 0, 0, partials);
  ok(cacto_critic_grad_det(P_, (const float*)dev(critic, F32, "critic"), (const float*)dev(critic_T, F32, "critic_T"), (const float*)dev(target, F32, "target"),
                           (float)w_S, (int)mc, (const float*)dev(state, F32, "state"), (const float*)opt(state_next, F32, "state_next"),
                           (const float*)dev(prtg, F32, "partial_rtg"), (const float*)opt(dVdx, F32, "dVdx"), (const float*)opt(done, F32, "done"),
                           (const float*)dev(weights, F32, "weights"), (float)inv_B, (float*)dev(grad, F32, "grad"), (float*)dev(rtg, F32, "rtg"),
                           (float*)dev(V, F32, "V"), (float*)dev(Vt, F32, "V_target"), (float*)opt(loss, F32, "loss"), B,
                           (float*)dev(partials, F32, "partials"), np, stream()), "critic_grad_det");
}
void actor_grad_det(const Tensor& p, const Tensor& actor, const Tensor& actor_T, const Tensor& critic, const Tensor& critic_T, const Tensor& state, const Tensor& term,
                    double inv_B, Tensor grad, const optional<Tensor>& actions, Tensor partials) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(state, P_->ns, "state"), nact = cacto_actor_param_count(P_->ns, P_->na);
  need(actor, nact, "actor"); need(grad, nact, "grad"); need(critic, cacto_critic_param_count(P_->ns), "critic"); need(term, B, "term"); need(actions, B * P_->na, "actions");
  need(actor_T, nact, "actor_T"); need(critic_T, cacto_critic_param_count(P_->ns), "critic_T");
  const int64_t np = det_need(CACTO_DET_ACTOR, B, P_, 0, 0, partials);
  ok(cacto_actor_grad_det(P_, (const float*)dev(actor, F32, "actor"), (const float*)dev(actor_T, F32, "actor_T"), (const float*)dev(critic, F32, "critic"),
                          (const float*)dev(critic_T, F32, "critic_T"), (const float*)dev(state, F32, "state"), (const double*)dev(term, F64, "term"), (float)inv_B,
                          (float*)dev(grad, F32, "grad"), (float*)opt(actions, F32, "actions"), B, (float*)dev(partials, F32, "partials"), np, stream()),
     "actor_grad_det");
}
void actor_grad_width_det(const Tensor& p, const Tensor& actor, int64_t nh1, int64_t nh2, const Tensor& critic, const Tensor& critic_T, const Tensor& state,
                          const Tensor& term, double inv_B, Tensor grad, const optional<Tensor>& actions, Tensor partials) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(state, P_->ns, "state"), nact = actor_width_count(P_, nh1, nh2), nc = cacto_critic_param_count(P_->ns);
  need(actor, nact, "actor"); need(grad, nact, "grad"); need(critic, nc, "critic"); need(critic_T, nc, "critic_T"); need(term, B, "term");
  need(actions, B * P_->na, "actions");
  const int64_t np = det_need(CACTO_DET_ACTOR_WIDTH, B, P_, nh1, nh2, partials);
  ok(cacto_actor_grad_width_det(P_, (const float*)dev(actor, F32, "actor"), (int32_t)nh1, (int32_t)nh2, (const float*)dev(critic, F32, "critic"),
                                (const float*)dev(critic_T, F32, "critic_T"), (const float*)dev(state, F32, "state"), (const double*)dev(term, F64, "term"),
                                (float)inv_B, (float*)dev(grad, F32, "grad"), (float*)opt(actions, F32, "actions"), B, (float*)dev(partials, F32, "partials"), np,
                                stream()), "actor_grad_width_det");
}
void critic_grad_tc_det(const Tensor& p, const Tensor& critic, const Tensor& target, double w_S, int64_t mc, const Tensor& state,
                        const optional<Tensor>& state_next, const Tensor& prtg, const optional<Tensor>& dVdx, const optional<Tensor>& done, const Tensor& weights,
                        double inv_B, Tensor grad, Tensor rtg, Tensor V, Tensor Vt, const optional<Tensor>& loss, Tensor workspace, Tensor partials) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(state, P_->ns, "state"), nc = cacto_critic_param_count(P_->ns);
  need(critic, nc, "critic"); need(target, nc, "target"); need(grad, nc, "grad");
  need(state_next, B * P_->ns, "state_next"); need(prtg, B, "partial_rtg"); need(dVdx, B * P_->ns, "dVdx"); need(done, B, "done"); need(weights, B, "weights");
  need(rtg, B, "rtg"); need(V, B, "V"); need(Vt, B, "V_target"); need(loss, 1, "loss");
  need_at_least(workspace, cacto_update_tc_workspace_bytes(B, P_->ns, P_->na), "workspace");
  const int64_t np = det_need(CACTO_DET_CRITIC_TC, B, P_, 0, 0, partials);
  ok(cacto_critic_grad_tc_det(P_, (const float*)dev(critic, F32, "critic"), (const float*)dev(target, F32, "target"), (float)w_S, (int)mc,
                              (const float*)dev(state, F32, "state"), (const float*)opt(state_next, F32, "state_next"), (const float*)dev(prtg, F32, "partial_rtg"),
                              (const float*)opt(dVdx, F32, "dVdx"), (const float*)opt(done, F32, "done"), (const float*)dev(weights, F32, "weights"), (float)inv_B,
                              (float*)dev(grad, F32, "grad"), (float*)dev(rtg, F32, "rtg"), (float*)dev(V, F32, "V"), (float*)dev(Vt, F32, "V_target"),
                              (float*)opt(loss, F32, "loss"), B, dev(workspace, at::kByte, "workspace"), workspace.numel(),
                              (float*)dev(partials, F32, "partials"), np, stream()), "critic_grad_tc_det");
}
void actor_grad_tc_det(const Tensor& p, const Tensor& actor, const Tensor& critic, const Tensor& state, const Tensor& term, double inv_B, Tensor grad,
                       const optional<Tensor>& actions, Tensor workspace, Tensor partials) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(state, P_->ns, "state"), nact = cacto_actor_param_count(P_->ns, P_->na);
  need(actor, nact, "actor"); need(grad, nact, "grad"); need(critic, cacto_critic_param_count(P_->ns), "critic"); need(term, B, "term"); need(actions, B * P_->na, "actions");
  need_at_least(workspace, cacto_update_tc_workspace_bytes(B, P_->ns, P_->na), "workspace");
  const int64_t np = det_need(CACTO_DET_ACTOR_TC, B, P_, 0, 0, partials);
  ok(cacto_actor_grad_tc_det(P_, (const float*)dev(actor, F32, "actor"), (const float*)dev(critic, F32, "critic"), (const float*)dev(state, F32, "state"),
                             (const double*)dev(term, F64, "term"), (float)inv_B, (float*)dev(grad, F32, "grad"), (float*)opt(actions, F32, "actions"), B,
                             dev(workspace, at::kByte, "workspace"), workspace.numel(), (float*)dev(partials, F32, "partials"), np, stream()),
     "actor_grad_tc_det");
}
int64_t update_tc_workspace_bytes(int64_t B, int64_t ns, int64_t na) { return cacto_update_tc_workspace_bytes(B, (int32_t)ns, (int32_t)na); }
void critic_grad_tc(const Tensor& p, const Tensor& critic, const Tensor& target, double w_S, int64_t mc, const Tensor& state, const optional<Tensor>& state_next,
                    const Tensor& prtg, const optional<Tensor>& dVdx, const optional<Tensor>& done, const Tensor& weights, double inv_B, Tensor grad, Tensor rtg, Tensor V,
                    Tensor Vt, const optional<Tensor>& loss, Tensor workspace) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(state, P_->ns, "state"), nc = cacto_critic_param_count(P_->ns);
  need(critic, nc, "critic"); need(target, nc, "target"); need(grad, nc, "grad");
  need(state_next, B * P_->ns, "state_next"); need(prtg, B, "partial_rtg"); need(dVdx, B * P_->ns, "dVdx"); need(done, B, "done"); need(weights, B, "weights");
  need(rtg, B, "rtg"); need(V, B, "V"); need(Vt, B, "V_target"); need(loss, 1, "loss");
  need_at_least(workspace, cacto_update_tc_workspace_bytes(B, P_->ns, P_->na), "workspace");
  ok(cacto_critic_grad_tc(P_, (const float*)dev(critic, F32, "critic"), (const float*)dev(target, F32, "target"), (float)w_S, (int)mc,
                          (const float*)dev(state, F32, "state"), (const float*)opt(state_next, F32, "state_next"), (const float*)dev(prtg, F32, "partial_rtg"),
                          (const float*)opt(dVdx, F32, "dVdx"), (const float*)opt(done, F32, "done"), (const float*)dev(weights, F32, "weights"), (float)inv_B,
                          (float*)dev(grad, F32, "grad"), (float*)dev(rtg, F32, "rtg"), (float*)dev(V, F32, "V"), (float*)dev(Vt, F32, "V_target"),
                          (float*)opt(loss, F32, "loss"), B, dev(workspace, at::kByte, "workspace"), workspace.numel(), stream()), "critic_grad_tc");
}
void actor_grad_tc(const Tensor& p, const Tensor& actor, const Tensor& critic, const Tensor& state, const Tensor& term, double inv_B, Tensor grad,
                   const optional<Tensor>& actions, Tensor workspace) {
  const cacto_sys_params* P_ = sys(p);      // checked before anything else is touched
  const int64_t B = rows_of(state, P_->ns, "state"), nact = cacto_actor_param_count(P_->ns, P_->na);
  need(actor, nact, "actor"); need(grad, nact, "grad"); need(critic, cacto_critic_param_count(P_->ns), "critic"); need(term, B, "term"); need(actions, B * P_->na, "actions");
  need_at_least(workspace, cacto_update_tc_workspace_bytes(B, P_->ns, P_->na), "workspace");
  ok(cacto_actor_grad_tc(P_, (const float*)dev(actor, F32, "actor"), (const float*)dev(critic, F32, "critic"), (const float*)dev(state, F32, "state"),
                         (const double*)dev(term, F64, "term"), (float)inv_B, (float*)dev(grad, F32, "grad"), (float*)opt(actions, F32, "actions"), B,
                         dev(workspace, at::kByte, "workspace"), workspace.numel(), stream()), "actor_grad_tc");
}
void adam_schedule(Tensor step, const Tensor& boundaries, const Tensor& values, int64_t nb, double beta1, double beta2, Tensor alpha, const optional<Tensor>& zero) {
  TORCH_CHECK(nb >= 0, "cacto: nb < 0");
  need(step, 1, "step"); need_at_least(boundaries, nb, "boundaries"); need_at_least(values, nb + 1, "values"); need(alpha, 1, "alpha"); need(zero, 1, "zero");
  ok(cacto_adam_schedule((int64_t*)dev(step, at::kLong, "step"), (const float*)dev(boundaries, F32, "boundaries"), (const float*)dev(values, F32, "values"), (int32_t)nb,
                         (float)beta1, (float)beta2, (float*)dev(alpha, F32, "alpha"), (float*)opt(zero, F32, "zero"), stream()), "adam_schedule");
}
void adam_schedule2(Tensor step_a, const Tensor& boundaries_a, const Tensor& values_a, int64_t nb_a, double beta1_a, double beta2_a, Tensor alpha_a, Tensor step_b,
                    const Tensor& boundaries_b, const Tensor& values_b, int64_t nb_b, double beta1_b, double beta2_b, Tensor alpha_b, const optional<Tensor>& zero) {
  TORCH_CHECK(nb_a >= 0 && nb_b >= 0, "cacto: nb < 0");
  need(step_a, 1, "step_a"); need_at_least(boundaries_a, nb_a, "boundaries_a"); need_at_least(values_a, nb_a + 1, "values_a"); need(alpha_a, 1, "alpha_a");
  need(step_b, 1, "step_b"); need_at_least(boundaries_b, nb_b, "boundaries_b"); need_at_least(values_b, nb_b + 1, "values_b"); need(alpha_b, 1, "alpha_b");
  need(zero, 1, "zero");
  ok(cacto_adam_schedule2((int64_t*)dev(step_a, at::kLong, "step_a"), (const float*)dev(boundaries_a, F32, "boundaries_a"), (const float*)dev(values_a, F32, "values_a"),
                          (int32_t)nb_a, (float)beta1_a, (float)beta2_a, (float*)dev(alpha_a, F32, "alpha_a"), (int64_t*)dev(step_b, at::kLong, "step_b"),
                          (const float*)dev(boundaries_b, F32, "boundaries_b"), (const float*)dev(values_b, F32, "values_b"), (int32_t)nb_b, (float)beta1_b, (float)beta2_b,
                          (float*)dev(alpha_b, F32, "alpha_b"), (float*)opt(zero, F32, "zero"), stream()), "adam_schedule2");
}
void adam_step(Tensor params, Tensor grad, Tensor m, Tensor v, double alpha_t, const optional<Tensor>& alpha_dev, double beta1, double beta2, double eps,
               const optional<Tensor>& target, double tau, const optional<Tensor>& params_T, int64_t is_critic, int64_t ns, int64_t na) {
  const int64_t n = params.numel();
  need(grad, n, "grad"); need(m, n, "m"); need(v, n, "v"); need(target, n, "target"); need(params_T, n, "params_T"); need(alpha_dev, 1, "alpha_dev");
  ok(cacto_adam_step((float*)dev(params, F32, "params"), (float*)dev(grad, F32, "grad"), (float*)dev(m, F32, "m"), (float*)dev(v, F32, "v"), (float)alpha_t,
                     (const float*)opt(alpha_dev, F32, "alpha_dev"), (float)beta1, (float)beta2, (float)eps, (float*)opt(target, F32, "target"), (float)tau,
                     (float*)opt(params_T, F32, "params_T"), (int32_t)is_critic, (int32_t)ns, (int32_t)na, params.numel(), stream()), "adam_step");
}
void transpose_params(const Tensor& params, Tensor params_T, int64_t is_critic, int64_t ns, int64_t na) {
  const int64_t n = is_critic ? cacto_critic_param_count((int32_t)ns) : cacto_actor_param_count((int32_t)ns, (int32_t)na);
  need(params, n, "params"); need(params_T, n, "params_T");
  ok(cacto_transpose_params((const float*)dev(params, F32, "params"), (float*)dev(params_T, F32, "params_T"), (int32_t)is_critic, (int32_t)ns, (int32_t)na, stream()),
     "transpose_params");
}

// ---- replay (K4) and reward-to-go (K5)
void segtree_update(const optional<Tensor>& sum_tree, const optional<Tensor>& min_tree, int64_t capacity, const Tensor& idx, const Tensor& value, Tensor stamp) {
  need(sum_tree, 2 * capacity, "sum_tree"); need(min_tree, 2 * capacity, "min_tree"); need(value, idx.numel(), "value"); need_at_least(stamp, capacity, "stamp");
  ok(cacto_segtree_update((double*)opt(sum_tree, F64, "sum_tree"), (double*)opt(min_tree, F64, "min_tree"), (int32_t)capacity, (const int64_t*)dev(idx, at::kLong, "idx"),
                          (const double*)dev(value, F64, "value"), (int32_t)idx.numel(), (int32_t*)dev(stamp, at::kInt, "stamp"), stream()), "segtree_update");
}
void segtree_sample(const Tensor& sum_tree, const Tensor& min_tree, int64_t capacity, int64_t max_idx, const Tensor& uniforms, Tensor idx, Tensor leaf, Tensor totals) {
  const int64_t n = uniforms.numel();
  need(sum_tree, 2 * capacity, "sum_tree"); need(min_tree, 2 * capacity, "min_tree"); need(idx, n, "idx"); need(leaf, n, "leaf"); need_at_least(totals, 3, "totals");
  ok(cacto_segtree_sample((const double*)dev(sum_tree, F64, "sum_tree"), (const double*)dev(min_tree, F64, "min_tree"), (int32_t)capacity, (int32_t)max_idx,
                          (const double*)dev(uniforms, F64, "uniforms"), (int32_t)uniforms.numel(), (int64_t*)dev(idx, at::kLong, "idx"), (double*)dev(leaf, F64, "leaf"),
                          (double*)dev(totals, F64, "totals"), stream()), "segtree_sample");
}
void buffer_gather(const Tensor& storage, int64_t ns, const Tensor& idx, Tensor state, Tensor prtg, Tensor state_next, Tensor dVdx, Tensor done, Tensor term,
                   const optional<Tensor>& exp_counter, const optional<Tensor>& stamp) {
  const int64_t n = idx.numel();
  TORCH_CHECK(storage.dim() == 2 && storage.size(1) == 3 * ns + 3, "cacto: storage must be [rows][3 ns + 3]");
  need(state, n * ns, "state"); need(prtg, n, "partial_rtg"); need(state_next, n * ns, "state_next"); need(dVdx, n * ns, "dVdx"); need(done, n, "done"); need(term, n, "term");
  ok(cacto_buffer_gather((const double*)dev(storage, F64, "storage"), (int32_t)ns, (const int64_t*)dev(idx, at::kLong, "idx"), (int32_t)idx.numel(),
                         (float*)dev(state, F32, "state"), (float*)dev(prtg, F32, "partial_rtg"), (float*)dev(state_next, F32, "state_next"), (float*)dev(dVdx, F32, "dVdx"),
                         (float*)dev(done, F32, "done"), (double*)dev(term, F64, "term"), (double*)opt(exp_counter, F64, "exp_counter"), (int32_t*)opt(stamp, at::kInt, "stamp"),
                         stream()), "buffer_gather");
}
void rtg_window(const Tensor& offsets, const Tensor& rwrd, const Tensor& states, int64_t ns, int64_t nsteps_td, int64_t mc, Tensor partial, Tensor total_, Tensor s_next,
                Tensor done, Tensor term, Tensor ep_return) {
  const int64_t total = rwrd.numel(), E = offsets.numel() - 1;
  TORCH_CHECK(E >= 0, "cacto: offsets must hold E + 1 entries");
  need(states, total * ns, "states"); need(partial, total, "partial"); need(total_, total, "total"); need(s_next, total * ns, "s_next"); need(done, total, "done");
  need(term, total, "term"); need(ep_return, E, "ep_return");
  ok(cacto_rtg_window((const int64_t*)dev(offsets, at::kLong, "offsets"), (int32_t)(offsets.numel() - 1), (const double*)dev(rwrd, F64, "rwrd"),
                      (const double*)dev(states, F64, "states"), (int32_t)ns, (int32_t)nsteps_td, (int32_t)mc, (double*)dev(partial, F64, "partial"),
                      (double*)dev(total_, F64, "total"), (double*)dev(s_next, F64, "s_next"), (double*)dev(done, F64, "done"), (double*)dev(term, F64, "term"),
                      (double*)dev(ep_return, F64, "ep_return"), stream()), "rtg_window");
}
int64_t abi_version() { return cacto_abi_version(); }

}  // namespace

TORCH_LIBRARY(cacto, m) {
  m.def("abi_version() -> int", abi_version);
  m.def("dyn_step(Tensor p, int layout, Tensor state, Tensor action, Tensor(a!) out) -> ()", dyn_step);
  m.def("dyn_derivative(Tensor p, int layout, Tensor state, Tensor action, Tensor(a!) Fu) -> ()", dyn_derivative);
  m.def("dyn_augmented(Tensor p, int layout, Tensor state, Tensor action, Tensor(a!) Fx, Tensor(b!) Fu) -> ()", dyn_augmented);
  m.def("ee_position(Tensor p, int layout, Tensor state, Tensor(a!) ee) -> ()", ee_position);
  m.def("reward(Tensor p, int layout, Tensor weights, Tensor state, Tensor? action, int ur5_plain_ucost, Tensor(a!) r, Tensor(b!)? dr_da) -> ()", reward);
  m.def("rollout(Tensor p, Tensor? actor, int use_actor, Tensor ics, Tensor horizon, int T_max, Tensor(a!) states, Tensor(b!) controls, Tensor(c!) flags, "
        "Tensor(d!)? rewards) -> ()", rollout);
  m.def("actor_tc16_prepare(Tensor actor, int ns, int na, Tensor(a!) w2img) -> ()", actor_tc16_prepare);
  m.def("rollout_tc16(Tensor p, Tensor actor, Tensor w2img, Tensor ics, Tensor horizon, int T_max, Tensor(a!) states, Tensor(b!) controls, Tensor(c!) flags, "
        "Tensor(d!)? rewards) -> ()", rollout_tc16);
  m.def("rollout_width(Tensor p, Tensor actor, int nh1, int nh2, Tensor ics, Tensor horizon, int T_max, Tensor(a!) states, Tensor(b!) controls, "
        "Tensor(c!) flags, Tensor(d!)? rewards) -> ()", rollout_width);
  m.def("actor_forward_width(Tensor p, Tensor actor, int nh1, int nh2, Tensor state, Tensor(a!) out) -> ()", actor_forward_width);
  m.def("actor_grad_width(Tensor p, Tensor actor, int nh1, int nh2, Tensor critic, Tensor critic_T, Tensor state, Tensor term, float inv_B, Tensor(a!) grad, "
        "Tensor(b!)? actions) -> ()", actor_grad_width);
  m.def("actor_forward(Tensor p, Tensor actor, Tensor state, Tensor(a!) out) -> ()", actor_forward);
  m.def("critic_forward(Tensor p, Tensor critic, Tensor state, Tensor(a!) value, Tensor(b!)? dV_ds) -> ()", critic_forward);
  m.def("critic_grad(Tensor p, Tensor critic, Tensor critic_T, Tensor target, float w_S, int mc, Tensor state, Tensor? state_next, Tensor prtg, Tensor? dVdx, "
        "Tensor? done, Tensor weights, float inv_B, Tensor(a!) grad, Tensor(b!) rtg, Tensor(c!) V, Tensor(d!) Vt, Tensor(e!)? loss) -> ()", critic_grad);
  m.def("actor_grad(Tensor p, Tensor actor, Tensor actor_T, Tensor critic, Tensor critic_T, Tensor state, Tensor term, float inv_B, Tensor(a!) grad, "
        "Tensor(b!)? actions) -> ()", actor_grad);
  m.def("update_tc_workspace_bytes(int B, int ns, int na) -> int", update_tc_workspace_bytes);
  m.def("critic_grad_tc(Tensor p, Tensor critic, Tensor target, float w_S, int mc, Tensor state, Tensor? state_next, Tensor prtg, Tensor? dVdx, Tensor? done, "
        "Tensor weights, float inv_B, Tensor(a!) grad, Tensor(b!) rtg, Tensor(c!) V, Tensor(d!) Vt, Tensor(e!)? loss, Tensor(f!) workspace) -> ()", critic_grad_tc);
  m.def("actor_grad_tc(Tensor p, Tensor actor, Tensor critic, Tensor state, Tensor term, float inv_B, Tensor(a!) grad, Tensor(b!)? actions, Tensor(c!) workspace) -> ()",
        actor_grad_tc);
  m.def("det_partials_floats(int net, int B, int ns, int na, int nh1, int nh2) -> int", det_partials_floats);
  m.def("critic_grad_det(Tensor p, Tensor critic, Tensor critic_T, Tensor target, float w_S, int mc, Tensor state, Tensor? state_next, Tensor prtg, "
        "Tensor? dVdx, Tensor? done, Tensor weights, float inv_B, Tensor(a!) grad, Tensor(b!) rtg, Tensor(c!) V, Tensor(d!) Vt, Tensor(e!)? loss, "
        "Tensor(f!) partials) -> ()", critic_grad_det);
  m.def("actor_grad_det(Tensor p, Tensor actor, Tensor actor_T, Tensor critic, Tensor critic_T, Tensor state, Tensor term, float inv_B, Tensor(a!) grad, "
        "Tensor(b!)? actions, Tensor(c!) partials) -> ()", actor_grad_det);
  m.def("actor_grad_width_det(Tensor p, Tensor actor, int nh1, int nh2, Tensor critic, Tensor critic_T, Tensor state, Tensor term, float inv_B, "
        "Tensor(a!) grad, Tensor(b!)? actions, Tensor(c!) partials) -> ()", actor_grad_width_det);
  m.def("critic_grad_tc_det(Tensor p, Tensor critic, Tensor target, float w_S, int mc, Tensor state, Tensor? state_next, Tensor prtg, Tensor? dVdx, "
        "Tensor? done, Tensor weights, float inv_B, Tensor(a!) grad, Tensor(b!) rtg, Tensor(c!) V, Tensor(d!) Vt, Tensor(e!)? loss, Tensor(f!) workspace, "
        "Tensor(g!) partials) -> ()", critic_grad_tc_det);
  m.def("actor_grad_tc_det(Tensor p, Tensor actor, Tensor critic, Tensor state, Tensor term, float inv_B, Tensor(a!) grad, Tensor(b!)? actions, "
        "Tensor(c!) workspace, Tensor(d!) partials) -> ()", actor_grad_tc_det);
  m.def("adam_schedule(Tensor(a!) step, Tensor boundaries, Tensor values, int nb, float beta1, float beta2, Tensor(b!) alpha, Tensor(c!)? zero) -> ()", adam_schedule);
  m.def("adam_schedule2(Tensor(a!) step_a, Tensor boundaries_a, Tensor values_a, int nb_a, float beta1_a, float beta2_a, Tensor(b!) alpha_a, Tensor(c!) step_b, "
        "Tensor boundaries_b, Tensor values_b, int nb_b, float beta1_b, float beta2_b, Tensor(d!) alpha_b, Tensor(e!)? zero) -> ()", adam_schedule2);
  m.def("adam_step(Tensor(a!) params, Tensor(b!) grad, Tensor(c!) m, Tensor(d!) v, float alpha_t, Tensor? alpha_dev, float beta1, float beta2, float eps, "
        "Tensor(e!)? target, float tau, Tensor(f!)? params_T, int is_critic, int ns, int na) -> ()", adam_step);
  m.def("transpose_params(Tensor params, Tensor(a!) params_T, int is_critic, int ns, int na) -> ()", transpose_params);
  m.def("segtree_update(Tensor(a!)? sum_tree, Tensor(b!)? min_tree, int capacity, Tensor idx, Tensor value, Tensor(c!) stamp) -> ()", segtree_update);
  m.def("segtree_sample(Tensor sum_tree, Tensor min_tree, int capacity, int max_idx, Tensor uniforms, Tensor(a!) idx, Tensor(b!) leaf, Tensor(c!) totals) -> ()",
        segtree_sample);
  m.def("buffer_gather(Tensor storage, int ns, Tensor idx, Tensor(a!) state, Tensor(b!) prtg, Tensor(c!) state_next, Tensor(d!) dVdx, Tensor(e!) done, Tensor(f!) term, "
        "Tensor(g!)? exp_counter, Tensor(h!)? stamp) -> ()", buffer_gather);
  m.def("rtg_window(Tensor offsets, Tensor rwrd, Tensor states, int ns, int nsteps_td, int mc, Tensor(a!) partial, Tensor(b!) total, Tensor(c!) s_next, Tensor(d!) done, "
        "Tensor(e!) term, Tensor(f!) ep_return) -> ()", rtg_window);
}
