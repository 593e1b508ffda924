// TORCH_LIBRARY layer over the C ABI of librrnco_b200.so (include/rrnco_b200.h): the same entry points as dispatcher ops
// `torch.ops.rrnco_b200.*` with CUDA kernels registered for them, so that the hot path is visible to the PyTorch
// dispatcher (torch.compile treats the ops as opaque leaves instead of graph-breaking on ctypes calls, autocast / functorch
// see tensors, profilers see op names) and a call costs no Python marshalling of structs.  The ops allocate their outputs
// through the caching allocator and launch on the current CUDA stream of the inputs' device; the C ABI underneath still
// never allocates.  rrnco_b200/torch_ops.py loads this library; the ctypes binding (rrnco_b200/_lib.py) stays as the fallback.
//
// Op                                   reference method it serves
//   minmax_normalize                   env._reset normalisation          rrnco/envs/rcvrp/env.py:138-145
//   gather_submatrix                   Real_World_Sampler.sample         rrnco/envs/rcvrp/sampler.py:84-90
//   atsp_step / rcvrp_step             ATSPEnv._step / RCVRPEnv._step    rrnco/envs/atsp/env.py:79-105, rcvrp/env.py:90-122,183-195
//   tour_reward                        env._get_reward                   rrnco/envs/*/env.py
//   select_action                      DecodingStrategy.step             rrnco/models/decoding.py:219-298
//   rollout                            RRNetPolicy.forward decode loop   rrnco/models/policy.py:203-243
//   beam_select / beam_backtrack       BeamSearch step / _backtrack      rrnco/models/decoding.py:402-542
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/library.h>
#include <torch/types.h>

#include "../../include/rrnco_b200.h"

namespace {

using at::Tensor;
using OptTensor = std::optional<Tensor>;

void check_rc(int rc, const char* what) {
  TORCH_CHECK(rc == RRNCO_OK, "librrnco_b200: ", what, ": ", rrnco_strerror(rc), " (code ", rc, ")");
}
void* stream_of(const Tensor& t) { return at::cuda::getCurrentCUDAStream(t.device().index()).stream(); }
Tensor f32c(const Tensor& t) { return t.to(at::kFloat).contiguous(); }
Tensor u8c(const Tensor& t) {
  Tensor c = t.contiguous();
  return c.scalar_type() == at::kBool ? c.view(at::kByte) : c.to(at::kByte);
}
// top_k above the row length keeps every entry; a negative one reaches the C ABI, which rejects it
int32_t clamp_k(int64_t k) { return k > INT32_MAX ? INT32_MAX : k < 0 ? -1 : (int32_t)k; }
template <typename T>
const T* cptr(const OptTensor& t) { return t.has_value() && t->defined() ? t->data_ptr<T>() : nullptr; }

std::tuple<Tensor, Tensor, Tensor> minmax_normalize(const Tensor& dist) {
  TORCH_CHECK(dist.is_cuda() && dist.dim() == 3 && dist.size(1) == dist.size(2), "distance matrices [B,N,N] on CUDA expected");
  c10::cuda::CUDAGuard guard(dist.device());
  Tensor in = f32c(dist);
  Tensor out = at::empty_like(in), mn = at::empty({in.size(0)}, in.options()), mx = at::empty({in.size(0)}, in.options());
  check_rc(rrnco_minmax_normalize(in.size(0), (int32_t)in.size(1), in.data_ptr<float>(), out.data_ptr<float>(),
                                  mn.data_ptr<float>(), mx.data_ptr<float>(), stream_of(in)), "minmax_normalize");
  return {out, mn, mx};
}

std::tuple<Tensor, Tensor, Tensor> gather_submatrix(const Tensor& city, const Tensor& idx, int64_t normalize) {
  TORCH_CHECK(city.is_cuda() && city.dim() == 2 && city.is_contiguous(), "contiguous city matrix [L,L] on CUDA expected");
  TORCH_CHECK(city.scalar_type() == at::kDouble || city.scalar_type() == at::kFloat, "float64 / float32 city matrix expected");
  c10::cuda::CUDAGuard guard(city.device());
  Tensor ix = idx.to(city.device(), at::kInt).contiguous();
  const int64_t B = ix.size(0), n = ix.size(1);
  auto fopt = city.options().dtype(at::kFloat);
  Tensor out = at::empty({B, n, n}, fopt), mn = at::empty({normalize ? B : 0}, fopt), mx = at::empty({normalize ? B : 0}, fopt);
  float* pmn = normalize ? mn.data_ptr<float>() : nullptr;
  float* pmx = normalize ? mx.data_ptr<float>() : nullptr;
  int rc = city.scalar_type() == at::kDouble
               ? rrnco_gather_submatrix(city.data_ptr<double>(), (int32_t)city.size(0), ix.data_ptr<int32_t>(), B, (int32_t)n,
                                        out.data_ptr<float>(), (int32_t)normalize, pmn, pmx, stream_of(city))
               : rrnco_gather_submatrix_f32(city.data_ptr<float>(), (int32_t)city.size(0), ix.data_ptr<int32_t>(), B, (int32_t)n,
                                            out.data_ptr<float>(), (int32_t)normalize, pmn, pmx, stream_of(city));
  check_rc(rc, "gather_submatrix");
  return {out, mn, mx};
}

// -> (action_mask, first_node, current_node, done)
std::tuple<Tensor, Tensor, Tensor, Tensor> atsp_step(const Tensor& action, const Tensor& step_i, const Tensor& mask_in,
                                                     const Tensor& first_in) {
  TORCH_CHECK(mask_in.is_cuda() && mask_in.dim() == 2, "action_mask [R,N] on CUDA expected");
  c10::cuda::CUDAGuard guard(mask_in.device());
  Tensor act = action.contiguous(), m = mask_in.contiguous(), first = first_in.reshape({-1}).contiguous(), si = step_i.contiguous();
  const int64_t R = m.size(0), N = m.size(1);
  auto iopt = m.options().dtype(at::kLong);
  Tensor mask_out = at::empty_like(m), first_out = at::empty({R}, iopt), cur_out = at::empty({R}, iopt),
         done = at::empty({R}, m.options().dtype(at::kBool));
  check_rc(rrnco_atsp_step(R, (int32_t)N, act.data_ptr<int64_t>(), si.data_ptr<int64_t>(), u8c(m).data_ptr<uint8_t>(),
                           first.data_ptr<int64_t>(), reinterpret_cast<uint8_t*>(mask_out.data_ptr()), first_out.data_ptr<int64_t>(),
                           cur_out.data_ptr<int64_t>(), reinterpret_cast<uint8_t*>(done.data_ptr()), stream_of(m)), "atsp_step");
  return {mask_out, first_out, cur_out, done};
}

// action given: RCVRPEnv._step -> (current_node [R,1], used_capacity [R,1], visited, done, action_mask)
// action None : get_action_mask on (visited, used, current)   -> the same tuple with only action_mask filled
std::tuple<Tensor, Tensor, Tensor, Tensor, Tensor> rcvrp_step(const OptTensor& action, const Tensor& demand,
                                                             const Tensor& capacity, const Tensor& used_in,
                                                             const Tensor& visited_in, const OptTensor& current_in) {
  TORCH_CHECK(visited_in.is_cuda() && visited_in.dim() == 2, "visited [R,N] on CUDA expected");
  c10::cuda::CUDAGuard guard(visited_in.device());
  Tensor vis = u8c(visited_in), dem = f32c(demand), cap = f32c(capacity).reshape({-1}), used = f32c(used_in).reshape({-1});
  const int64_t R = vis.size(0), N = vis.size(1);
  Tensor mask = at::empty({R, N}, vis.options().dtype(at::kBool));
  Tensor cur, used_o, vis_o, done;
  if (action.has_value() && action->defined()) {
    Tensor act = action->contiguous();
    cur = at::empty({R, 1}, vis.options().dtype(at::kLong));
    used_o = at::empty({R, 1}, dem.options());
    vis_o = at::empty_like(vis);
    done = at::empty({R}, vis.options().dtype(at::kBool));
    check_rc(rrnco_rcvrp_step(R, (int32_t)N, dem.size(0), act.data_ptr<int64_t>(), dem.data_ptr<float>(), cap.data_ptr<float>(),
                              cap.size(0), used.data_ptr<float>(), vis.data_ptr<uint8_t>(), nullptr, used_o.data_ptr<float>(),
                              vis_o.data_ptr<uint8_t>(), cur.data_ptr<int64_t>(), reinterpret_cast<uint8_t*>(done.data_ptr()),
                              reinterpret_cast<uint8_t*>(mask.data_ptr()), stream_of(vis)), "rcvrp_step");
  } else {
    TORCH_CHECK(current_in.has_value(), "current_node is needed when no action is given");
    Tensor ci = current_in->reshape({-1}).contiguous();
    check_rc(rrnco_rcvrp_step(R, (int32_t)N, dem.size(0), nullptr, dem.data_ptr<float>(), cap.data_ptr<float>(), cap.size(0),
                              used.data_ptr<float>(), vis.data_ptr<uint8_t>(), ci.data_ptr<int64_t>(), nullptr, nullptr, nullptr,
                              nullptr, reinterpret_cast<uint8_t*>(mask.data_ptr()), stream_of(vis)), "rcvrp_step(mask)");
    cur = used_o = vis_o = done = at::empty({0}, vis.options());
  }
  return {cur, used_o, vis_o, done, mask};
}

// -> (real, normalised); real is empty when min_d / max_d are not given
std::tuple<Tensor, Tensor> tour_reward(const Tensor& actions, const Tensor& distance, bool prepend_depot,
                                       const OptTensor& open_route, const OptTensor& min_d, const OptTensor& max_d) {
  TORCH_CHECK(actions.is_cuda() && actions.dim() == 2 && distance.dim() == 3, "actions [R,T], distance [rows,N,N] on CUDA expected");
  c10::cuda::CUDAGuard guard(actions.device());
  Tensor act = actions.contiguous(), dm = f32c(distance);
  const int64_t R = act.size(0), T = act.size(1);
  Tensor norm = at::empty({R}, dm.options());
  const bool has_mm = min_d.has_value() && min_d->defined();
  Tensor real = at::empty({has_mm ? R : 0}, dm.options());
  Tensor orp, mn, mx;
  if (open_route.has_value() && open_route->defined()) orp = u8c(open_route->reshape({-1}));
  if (has_mm) { mn = f32c(*min_d); mx = f32c(*max_d); }
  check_rc(rrnco_tour_reward(R, (int32_t)T, (int32_t)dm.size(-1), dm.size(0), act.data_ptr<int64_t>(), dm.data_ptr<float>(),
                             prepend_depot ? 1 : 0, orp.defined() ? orp.data_ptr<uint8_t>() : nullptr,
                             has_mm ? mn.data_ptr<float>() : nullptr, has_mm ? mx.data_ptr<float>() : nullptr,
                             norm.data_ptr<float>(), has_mm ? real.data_ptr<float>() : nullptr, stream_of(act)), "tour_reward");
  return {real, norm};
}

// -> (action, log-prob); `status` (int32 [1]) is OR-ed in place
std::tuple<Tensor, Tensor> select_action(const Tensor& logits, const Tensor& mask, int64_t decode_mode, double tanh_clipping,
                                         double temperature, int64_t seed, int64_t step, const OptTensor& forced, Tensor status,
                                         int64_t top_k, double top_p) {
  TORCH_CHECK(logits.is_cuda() && logits.dim() == 2, "logits [R,N] on CUDA expected");
  c10::cuda::CUDAGuard guard(logits.device());
  Tensor lg = f32c(logits), m = u8c(mask);
  const int64_t R = lg.size(0), N = lg.size(1);
  Tensor action = at::empty({R}, lg.options().dtype(at::kLong)), logp = at::empty({R}, lg.options());
  Tensor f;
  if (forced.has_value() && forced->defined()) f = forced->contiguous();
  check_rc(rrnco_select_action_filtered(R, (int32_t)N, lg.data_ptr<float>(), m.data_ptr<uint8_t>(), (int32_t)decode_mode,
                                        (float)tanh_clipping, (float)temperature, (uint64_t)seed, (int32_t)step,
                                        f.defined() ? f.data_ptr<int64_t>() : nullptr, action.data_ptr<int64_t>(),
                                        logp.data_ptr<float>(), reinterpret_cast<uint32_t*>(status.data_ptr<int32_t>()),
                                        clamp_k(top_k), (float)top_p, stream_of(lg)), "select_action");
  return {action, logp};
}

// -> (action, parent row, log-prob, new score), rows in (w b) order; `status` (int32 [1]) is OR-ed in place
std::tuple<Tensor, Tensor, Tensor, Tensor> beam_select(const Tensor& logits, const Tensor& mask, const Tensor& score,
                                                       int64_t beam_width, double tanh_clipping, double temperature,
                                                       Tensor status) {
  TORCH_CHECK(logits.is_cuda() && logits.dim() == 2, "logits [R,N] on CUDA expected");
  TORCH_CHECK(beam_width >= 2 && logits.size(0) % beam_width == 0, "beam_select: beam_width >= 2 dividing the rows expected");
  c10::cuda::CUDAGuard guard(logits.device());
  Tensor lg = f32c(logits), m = u8c(mask), sc = f32c(score);
  const int64_t R = lg.size(0), N = lg.size(1);
  TORCH_CHECK(sc.numel() == R, "beam_select: one score per row expected");
  auto lopt = lg.options().dtype(at::kLong);
  Tensor action = at::empty({R}, lopt), parent = at::empty({R}, lopt), logp = at::empty({R}, lg.options()),
         out = at::empty({R}, lg.options());
  check_rc(rrnco_beam_select(R / beam_width, (int32_t)beam_width, (int32_t)N, lg.data_ptr<float>(), m.data_ptr<uint8_t>(),
                             sc.data_ptr<float>(), (float)tanh_clipping, (float)temperature, action.data_ptr<int64_t>(),
                             parent.data_ptr<int64_t>(), logp.data_ptr<float>(), out.data_ptr<float>(),
                             reinterpret_cast<uint32_t*>(status.data_ptr<int32_t>()), stream_of(lg)), "beam_select");
  return {action, parent, logp, out};
}

// step-major [T, R] actions / parents / log-probs -> (actions [R, T], log-probs [R, T] | empty, log-likelihood [R]);
// `status` (int32 [1]) is OR-ed in place
std::tuple<Tensor, Tensor, Tensor> beam_backtrack(const Tensor& actions, const Tensor& parents, const Tensor& logprobs,
                                                  bool per_step_logprobs, Tensor status) {
  TORCH_CHECK(actions.is_cuda() && actions.dim() == 2 && parents.sizes() == actions.sizes() &&
              logprobs.sizes() == actions.sizes(), "actions / parents / logprobs [T,R] on CUDA expected");
  c10::cuda::CUDAGuard guard(actions.device());
  Tensor a = actions.to(at::kLong).contiguous(), p = parents.to(at::kLong).contiguous(), l = f32c(logprobs);
  const int64_t T = a.size(0), R = a.size(1);
  Tensor a_out = at::empty({R, T}, a.options());
  Tensor l_out = at::empty({per_step_logprobs ? R : 0, per_step_logprobs ? T : 0}, l.options());
  Tensor ll = at::empty({R}, l.options());
  check_rc(rrnco_beam_backtrack(R, (int32_t)T, a.data_ptr<int64_t>(), p.data_ptr<int64_t>(), l.data_ptr<float>(),
                                a_out.data_ptr<int64_t>(), per_step_logprobs ? l_out.data_ptr<float>() : nullptr,
                                ll.data_ptr<float>(), reinterpret_cast<uint32_t*>(status.data_ptr<int32_t>()), stream_of(a)),
           "beam_backtrack");
  return {a_out, l_out, ll};
}

// weights: [ffn_w1, ffn_b1, ffn_w2, ffn_b2, ctx_state_w?, ctx_placeholder_q?]
// cache  : [glimpse_key, glimpse_val, logit_key, ctx_node_proj, ctx_node_proj2?]
// data   : [distance, duration?, demand?, demand_backhaul?, time_windows?, service_time?, vehicle_capacity?, distance_limit?,
//           open_route?, backhaul_class?, min_distance?, max_distance?]   (the members of rrnco_instance_data_t, in order)
// -> (actions [R, t_cap], logprob [R, t_cap] | empty, log_likelihood [R], normalised reward [R], real reward [R] | empty,
//     info int32 [2] = (longest rollout T, device status word), tile_steps int32 [n_inst * ceil(S / rrnco_rollout_tile_rows)])
std::tuple<Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor> rollout(
    int64_t env, int64_t n_starts, bool multistart, int64_t decode_mode, int64_t seed, const c10::List<OptTensor>& weights,
    double alpha, double beta, double tanh_clipping, double temperature, const c10::List<OptTensor>& cache,
    const c10::List<OptTensor>& data, const OptTensor& forced_actions, int64_t t_cap, bool per_step_logprobs, Tensor workspace,
    int64_t top_k, double top_p) {
  TORCH_CHECK(weights.size() == 6 && cache.size() == 5 && data.size() == 12, "rollout: weights[6], cache[5], data[12] expected");
  auto W = [&](size_t i) -> OptTensor { return weights.get(i); };
  auto C = [&](size_t i) -> OptTensor { return cache.get(i); };
  auto D = [&](size_t i) -> OptTensor { return data.get(i); };
  TORCH_CHECK(C(0).has_value() && C(0)->is_cuda() && C(0)->dim() == 3, "cache tensors [n_inst,N,E] on CUDA expected");
  const Tensor& key = *C(0);
  c10::cuda::CUDAGuard guard(key.device());
  const int64_t n_inst = key.size(0), N = key.size(1), R = n_inst * n_starts;
  rrnco_decoder_weights_t w{};
  w.ffn_w1 = cptr<float>(W(0)); w.ffn_b1 = cptr<float>(W(1)); w.ffn_w2 = cptr<float>(W(2)); w.ffn_b2 = cptr<float>(W(3));
  w.ctx_state_w = cptr<float>(W(4)); w.ctx_placeholder_q = cptr<float>(W(5));
  w.alpha = (float)alpha; w.beta = (float)beta; w.tanh_clipping = (float)tanh_clipping; w.temperature = (float)temperature;
  rrnco_decoder_cache_t c{};
  c.glimpse_key = cptr<float>(C(0)); c.glimpse_val = cptr<float>(C(1)); c.logit_key = cptr<float>(C(2));
  c.ctx_node_proj = cptr<float>(C(3)); c.ctx_node_proj2 = cptr<float>(C(4));
  TORCH_CHECK(D(0).has_value(), "data[0] (distance) is required");
  rrnco_instance_data_t d{};
  d.data_rows = D(0)->size(0);
  d.distance = cptr<float>(D(0)); d.duration = cptr<float>(D(1)); d.demand = cptr<float>(D(2)); d.demand_backhaul = cptr<float>(D(3));
  d.time_windows = cptr<float>(D(4)); d.service_time = cptr<float>(D(5)); d.vehicle_capacity = cptr<float>(D(6));
  d.distance_limit = cptr<float>(D(7)); d.open_route = cptr<uint8_t>(D(8)); d.backhaul_class = cptr<float>(D(9));
  d.min_distance = cptr<float>(D(10)); d.max_distance = cptr<float>(D(11));
  const bool has_mm = d.min_distance != nullptr;
  Tensor forced;
  int64_t forced_T = 0;
  if (forced_actions.has_value() && forced_actions->defined()) {
    forced = forced_actions->contiguous();
    forced_T = forced.size(1);
  }
  auto fopt = key.options().dtype(at::kFloat);
  Tensor actions = at::empty({R, t_cap}, key.options().dtype(at::kLong));
  Tensor logprob = at::empty({per_step_logprobs ? R : 0, per_step_logprobs ? t_cap : 0}, fopt);
  Tensor ll = at::empty({R}, fopt), norm = at::empty({R}, fopt), real = at::empty({has_mm ? R : 0}, fopt);
  Tensor info = at::zeros({2}, key.options().dtype(at::kInt));
  const int64_t need = rrnco_rollout_workspace_bytes((int32_t)env, (int32_t)N, n_inst, (int32_t)n_starts);
  TORCH_CHECK(workspace.is_cuda() && workspace.scalar_type() == at::kByte && workspace.numel() >= need,
              "rollout: workspace of >= ", need, " bytes (uint8, CUDA) expected");
  check_rc(rrnco_rollout_filtered((int32_t)env, (int32_t)N, n_inst, (int32_t)n_starts, multistart ? 1 : 0, (int32_t)decode_mode,
                                  (uint64_t)seed, &w, &c, &d, forced.defined() ? forced.data_ptr<int64_t>() : nullptr,
                                  (int32_t)forced_T, (int32_t)t_cap, actions.data_ptr<int64_t>(),
                                  per_step_logprobs ? logprob.data_ptr<float>() : nullptr, ll.data_ptr<float>(),
                                  norm.data_ptr<float>(), has_mm ? real.data_ptr<float>() : nullptr, info.data_ptr<int32_t>(),
                                  reinterpret_cast<uint32_t*>(info.data_ptr<int32_t>() + 1), workspace.data_ptr<uint8_t>(),
                                  clamp_k(top_k), (float)top_p, stream_of(key)), "rollout");
  const int64_t tile_rows = rrnco_rollout_tile_rows((int32_t)env, (int32_t)N, n_inst, (int32_t)n_starts);
  const int64_t n_tiles = n_inst * ((n_starts + tile_rows - 1) / tile_rows);
  Tensor tile_steps = workspace.narrow(0, 2 * R * 8, 4 * n_tiles).view(at::kInt);
  return {actions, logprob, ll, norm, real, info, tile_steps};
}

int64_t rollout_workspace_bytes(int64_t env, int64_t n_nodes, int64_t n_inst, int64_t n_starts) {
  return rrnco_rollout_workspace_bytes((int32_t)env, (int32_t)n_nodes, n_inst, (int32_t)n_starts);
}

}  // namespace

TORCH_LIBRARY(rrnco_b200, m) {
  m.def("minmax_normalize(Tensor dist) -> (Tensor, Tensor, Tensor)");
  m.def("gather_submatrix(Tensor city, Tensor idx, int normalize) -> (Tensor, Tensor, Tensor)");
  m.def("atsp_step(Tensor action, Tensor step_i, Tensor mask_in, Tensor first_in) -> (Tensor, Tensor, Tensor, Tensor)");
  m.def("rcvrp_step(Tensor? action, Tensor demand, Tensor capacity, Tensor used_in, Tensor visited_in, Tensor? current_in) -> "
        "(Tensor, Tensor, Tensor, Tensor, Tensor)");
  m.def("tour_reward(Tensor actions, Tensor distance, bool prepend_depot, Tensor? open_route, Tensor? min_d, Tensor? max_d) -> "
        "(Tensor, Tensor)");
  m.def("select_action(Tensor logits, Tensor mask, int decode_mode, float tanh_clipping, float temperature, int seed, int step, "
        "Tensor? forced, Tensor(a!) status, int top_k=0, float top_p=0.0) -> (Tensor, Tensor)");
  m.def("rollout(int env, int n_starts, bool multistart, int decode_mode, int seed, Tensor?[] weights, float alpha, float beta, "
        "float tanh_clipping, float temperature, Tensor?[] cache, Tensor?[] data, Tensor? forced_actions, int t_cap, "
        "bool per_step_logprobs, Tensor(a!) workspace, int top_k=0, float top_p=0.0) -> "
        "(Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor)");
  m.def("beam_select(Tensor logits, Tensor mask, Tensor score, int beam_width, float tanh_clipping, float temperature, "
        "Tensor(a!) status) -> (Tensor, Tensor, Tensor, Tensor)");
  m.def("beam_backtrack(Tensor actions, Tensor parents, Tensor logprobs, bool per_step_logprobs, Tensor(a!) status) -> "
        "(Tensor, Tensor, Tensor)");
  m.def("rollout_workspace_bytes(int env, int n_nodes, int n_inst, int n_starts) -> int", &rollout_workspace_bytes);
}

TORCH_LIBRARY_IMPL(rrnco_b200, CUDA, m) {
  m.impl("minmax_normalize", &minmax_normalize);
  m.impl("gather_submatrix", &gather_submatrix);
  m.impl("atsp_step", &atsp_step);
  m.impl("rcvrp_step", &rcvrp_step);
  m.impl("tour_reward", &tour_reward);
  m.impl("select_action", &select_action);
  m.impl("rollout", &rollout);
  m.impl("beam_select", &beam_select);
  m.impl("beam_backtrack", &beam_backtrack);
}
