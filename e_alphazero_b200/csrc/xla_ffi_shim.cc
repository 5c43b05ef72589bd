// xla_ffi_shim.cc -- XLA typed-FFI custom-call handlers over the C ABI of libeaz_b200.so (include/eaz_b200.h).
//
// This is the binding a maintainer of emcts/e-alphazero adds to call the library from inside the jitted / pmapped JAX program
// (SURVEY.md 8b "Who calls it (2)"): one handler per entry point of the hot path,
//
//   eaz_search          emctx.epistemic_gumbel_muzero_policy + Tree.epistemic_summary   selfplay.py:100-121, reanalyze.py:70-86,
//                       (DeepSea and Subleq; recurrent_fn of context.py:109-157 fused)    evaluate.py:29-45
//   eaz_evaluate        the evaluate() episode loop (search + env step + reward sum under  evaluate.py:13-57
//                       a device-decided while condition)
//   eaz_selfplay        the selfplay() scan (T steps of search + auto-reset env step, every  selfplay.py:78-149
//                       output stacked over the steps)
//   eaz_env_step        pgx Env.step / selfplay.auto_reset                               selfplay.py:26-75,135, evaluate.py:47
//   eaz_env_init        pgx Env.init (vmapped)                                           selfplay.py:161,166, main.py:205
//   eaz_mlp_forward_states   forward.apply(params, state, states.observation)            selfplay.py:89, reanalyze.py:67,90
//   eaz_reanalyze_targets    the target arithmetic after the search                      reanalyze.py:86-129
//   eaz_hash_update     BaseHash.update on the observations of a training batch           network/hashes.py:45-50, train.py:22
//   eaz_replay_init / _add / _add_sequence / _sample / _set_priorities / _status
//                       flashbax make_prioritised_flat_buffer on the compact ring         main.py:217-225, 383-385, 413-414, 454
//                       (_add_sequence: a whole self-play scan's states, add_sequences=True)
//                       (csrc/replay.cu: the write cursor lives in the tree header, sampling is keyed and reads nothing it writes)
//
// XLA owns every buffer (results and the workspace are XLA-allocated), the stream comes from PlatformStream, errors travel as
// ffi::Error carrying eaz_last_error().  The handlers hold no state.
//
// Build (where jaxlib is installed; its headers are NOT in the image this repository was developed in, so `make xla_ffi` is
// a no-op there and tests/test_abi_cpu.py compiles this file against tests/xla_ffi_stub/, a minimal stand-in of the API):
//   g++ -std=c++17 -O2 -shared -fPIC -I$(python -c "import jax.ffi; print(jax.ffi.include_dir())") -I/usr/local/cuda/include ...
//       -I../../include xla_ffi_shim.cc -o ../libeaz_xla_ffi.so -L.. -leaz_b200 -L/usr/local/cuda/lib64 -lcudart -Wl,-rpath,'$ORIGIN'
// Python side: e_alphazero_b200/jax_ffi.py registers the symbols and wraps them in the reference's call shapes.
//
// Argument convention shared by all handlers
//   * the env instance is described by int attributes (env_kind, size, word_size, binary_encoding, reward_fn) plus the
//     `action_map` buffer (DeepSea: bool [N,N]; Subleq: any 1-element dummy);
//   * a pgx.State travels as its information-carrying leaves, in the field order of `eaz_state`:
//       step_count S32[B], rewards F32[B,1], terminated PRED[B], truncated PRED[B],
//       DeepSea: col S32[B]            Subleq: memory S32[B,ws], task S32[B], solved PRED[B], input_after S32[B,8], output_after S32[B,8]
//   * the haiku parameters travel as 24 F32 buffers: for head in (value, ube, exploit, explore) for layer in 0..2: w, b
//     (module order fc_az_net/linear, linear_1 .. linear_11, fully_connected.py:49-81), then the hash state `binary_set` U8.
#include <cuda_runtime_api.h>

#include <algorithm>
#include <cstdint>
#include <string>

#include "eaz_b200.h"
#include "xla/ffi/api/ffi.h"

namespace ffi = xla::ffi;

namespace {

ffi::Error EazError(int rc, const char* what) {
  if (rc == EAZ_OK) return ffi::Error::Success();
  const std::string msg = std::string(what) + ": " + eaz_last_error();
  switch (rc) {
    case EAZ_ERR_INVALID_ARG: return ffi::Error(ffi::ErrorCode::kInvalidArgument, msg);
    case EAZ_ERR_WORKSPACE: return ffi::Error(ffi::ErrorCode::kResourceExhausted, msg);
    case EAZ_ERR_UNSUPPORTED: return ffi::Error(ffi::ErrorCode::kUnimplemented, msg);
    default: return ffi::Error(ffi::ErrorCode::kInternal, msg);
  }
}
ffi::Error Bad(const std::string& msg) { return ffi::Error(ffi::ErrorCode::kInvalidArgument, msg); }

#define EAZ_FFI_TRY(expr)                \
  do {                                   \
    ffi::Error _e = (expr);              \
    if (_e.failure()) return _e;         \
  } while (0)

template <typename T>
ffi::Error GetArg(ffi::RemainingArgs& args, size_t i, const char* name, T** out, int64_t min_elems) {
  if (i >= args.size()) return Bad(std::string("missing argument: ") + name);
  auto buf = args.get<ffi::AnyBuffer>(i);
  if (!buf.has_value()) return buf.error();
  if ((int64_t)buf->size_bytes() < min_elems * (int64_t)sizeof(T))
    return Bad(std::string(name) + ": buffer smaller than expected");
  *out = reinterpret_cast<T*>(buf->untyped_data());
  return ffi::Error::Success();
}
template <typename T>
ffi::Error GetRet(ffi::RemainingRets& rets, size_t i, const char* name, T** out, int64_t min_elems) {
  if (i >= rets.size()) return Bad(std::string("missing result: ") + name);
  auto buf = rets.get<ffi::AnyBuffer>(i);
  if (!buf.has_value()) return buf.error();
  if ((int64_t)(*buf)->size_bytes() < min_elems * (int64_t)sizeof(T))
    return Bad(std::string(name) + ": result buffer smaller than expected");
  *out = reinterpret_cast<T*>((*buf)->untyped_data());
  return ffi::Error::Success();
}

eaz_env MakeEnv(int32_t env_kind, int32_t size, int32_t word_size, int32_t binary_encoding, int32_t reward_fn, const void* action_map) {
  eaz_env env{};
  env.kind = env_kind;
  env.size = size;
  env.action_map = env_kind == EAZ_ENV_DEEPSEA ? static_cast<const uint8_t*>(action_map) : nullptr;
  env.word_size = word_size;
  env.binary_encoding = binary_encoding;
  env.reward_fn = reward_fn;
  return env;
}
constexpr size_t kCommonLeaves = 4;
size_t NumLeaves(const eaz_env& env) { return kCommonLeaves + (env.kind == EAZ_ENV_DEEPSEA ? 1 : 5); }

// pgx.State leaves (see the header comment) starting at args[*i] -> eaz_state of device pointers; advances *i
template <typename Src, typename Getter>
ffi::Error ReadState(Src& src, Getter get, size_t* i, const eaz_env& env, int64_t B, eaz_state* st) {
  *st = eaz_state{};
  EAZ_FFI_TRY(get(src, (*i)++, "state.step_count", &st->step_count, B));
  EAZ_FFI_TRY(get(src, (*i)++, "state.rewards", &st->rewards, B));
  EAZ_FFI_TRY(get(src, (*i)++, "state.terminated", &st->terminated, B));
  EAZ_FFI_TRY(get(src, (*i)++, "state.truncated", &st->truncated, B));
  if (env.kind == EAZ_ENV_DEEPSEA) {
    EAZ_FFI_TRY(get(src, (*i)++, "state.col", &st->col, B));
  } else {
    EAZ_FFI_TRY(get(src, (*i)++, "state.memory", &st->memory, B * env.word_size));
    EAZ_FFI_TRY(get(src, (*i)++, "state.task", &st->task, B));
    EAZ_FFI_TRY(get(src, (*i)++, "state.solved", &st->solved, B));
    EAZ_FFI_TRY(get(src, (*i)++, "state.input_after", &st->input_after, B * EAZ_SUBLEQ_IO_LEN));
    EAZ_FFI_TRY(get(src, (*i)++, "state.output_after", &st->output_after, B * EAZ_SUBLEQ_IO_LEN));
  }
  return ffi::Error::Success();
}
ffi::Error ReadStateArgs(ffi::RemainingArgs& args, size_t* i, const eaz_env& env, int64_t B, eaz_state* st) {
  auto get = [](ffi::RemainingArgs& a, size_t k, const char* nm, auto** out, int64_t n) { return GetArg(a, k, nm, out, n); };
  return ReadState(args, get, i, env, B, st);
}
ffi::Error ReadStateRets(ffi::RemainingRets& rets, size_t* i, const eaz_env& env, int64_t B, eaz_state* st) {
  auto get = [](ffi::RemainingRets& r, size_t k, const char* nm, auto** out, int64_t n) { return GetRet(r, k, nm, out, n); };
  return ReadState(rets, get, i, env, B, st);
}

// element sizes of the leaves, for the device-to-device copies of the functional (non-aliased) env calls
ffi::Error CopyState(const eaz_env& env, const eaz_state& src, const eaz_state& dst, int64_t B, cudaStream_t stream) {
  auto cp = [&](void* d, const void* s, size_t bytes) -> cudaError_t {
    if (d == s || bytes == 0) return cudaSuccess;  // input_output_aliases donated the buffer: already in place
    return cudaMemcpyAsync(d, s, bytes, cudaMemcpyDeviceToDevice, stream);
  };
  cudaError_t e = cudaSuccess;
  auto acc = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
  acc(cp(dst.step_count, src.step_count, B * 4));
  acc(cp(dst.rewards, src.rewards, B * 4));
  acc(cp(dst.terminated, src.terminated, B));
  acc(cp(dst.truncated, src.truncated, B));
  if (env.kind == EAZ_ENV_DEEPSEA) {
    acc(cp(dst.col, src.col, B * 4));
  } else {
    acc(cp(dst.memory, src.memory, B * 4 * env.word_size));
    acc(cp(dst.task, src.task, B * 4));
    acc(cp(dst.solved, src.solved, B));
    acc(cp(dst.input_after, src.input_after, B * 4 * EAZ_SUBLEQ_IO_LEN));
    acc(cp(dst.output_after, src.output_after, B * 4 * EAZ_SUBLEQ_IO_LEN));
  }
  if (e != cudaSuccess) return ffi::Error(ffi::ErrorCode::kInternal, std::string("state copy: ") + cudaGetErrorString(e));
  return ffi::Error::Success();
}

// 24 weight / bias buffers + nothing else, starting at args[*i]
ffi::Error ReadNet(ffi::RemainingArgs& args, size_t* i, const eaz_env& env, const void* binary_set, int32_t hash_bits, int32_t hash_io,
                   float max_u, float novelty_scale, eaz_fc_params* net) {
  *net = eaz_fc_params{};
  const int32_t D = eaz_env_obs_dim(&env), A = eaz_env_num_actions(&env);
  if (D <= 0 || A <= 0) return EazError(EAZ_ERR_INVALID_ARG, "env description");
  if (*i >= args.size()) return Bad("missing network parameters");
  // hidden width from the first bias buffer (fc_az_net/linear: b [hidden])
  {
    auto b0 = args.get<ffi::AnyBuffer>(*i + 1);
    if (!b0.has_value()) return b0.error();
    net->hidden = (int32_t)b0->element_count();
  }
  net->in_dim = D;
  net->num_actions = A;
  const int64_t H = net->hidden;
  for (int h = 0; h < 4; ++h) {
    const int64_t out3 = h >= EAZ_HEAD_EXPLOIT ? A : 1;
    const int64_t ins[3] = {D, H, H}, outs[3] = {H, H, out3};
    for (int l = 0; l < 3; ++l) {
      float *w = nullptr, *b = nullptr;
      EAZ_FFI_TRY(GetArg(args, (*i)++, "params.w", &w, ins[l] * outs[l]));
      EAZ_FFI_TRY(GetArg(args, (*i)++, "params.b", &b, outs[l]));
      net->w[h][l] = w;
      net->b[h][l] = b;
    }
  }
  net->binary_set = static_cast<const uint8_t*>(binary_set);
  net->hash_bits = hash_bits;
  net->hash_io = hash_io;
  net->word_size = env.kind == EAZ_ENV_SUBLEQ ? env.word_size : 0;
  net->max_u = max_u;
  net->novelty_scale = novelty_scale;
  return ffi::Error::Success();
}

void* AlignUp(void* p, size_t a) { return reinterpret_cast<void*>((reinterpret_cast<uintptr_t>(p) + (a - 1)) & ~(uintptr_t)(a - 1)); }

// ------------------------------------------------------------------------------------------------ search
// args : beta F32[B], gumbel F32[B,A], invalid_actions PRED[B,A], action_map, binary_set U8[2^(bits-3)],
//        root prior_logits F32[B,A], root value F32[B], root value_epistemic_variance F32[B]   (ignored when fused_root != 0),
//        workspace_in U8[ws] (pass the previous call's `workspace` result with input_output_aliases to keep the parameter-derived
//        tables across the steps of one selfplay() scan; anything else = scratch),
//        then the root state leaves, then the 24 parameter buffers
// rets : action S32[B], action_weights F32[B,A], value F32[B], value_epistemic_std F32[B], visit_counts F32[B,A],
//        visit_probs F32[B,A], qvalues F32[B,A], qvalues_epistemic_variance F32[B,A], root_value F32[B], root_ube F32[B],
//        workspace U8[eaz_search_workspace_bytes + 256]
ffi::Error SearchImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> beta, ffi::Buffer<ffi::F32> gumbel, ffi::AnyBuffer invalid,
                      ffi::AnyBuffer action_map, ffi::Buffer<ffi::U8> binary_set, ffi::Buffer<ffi::F32> prior_logits,
                      ffi::Buffer<ffi::F32> value, ffi::Buffer<ffi::F32> variance, ffi::Buffer<ffi::U8> workspace_in,
                      ffi::RemainingArgs rest, ffi::ResultBuffer<ffi::S32> action, ffi::ResultBuffer<ffi::F32> action_weights,
                      ffi::ResultBuffer<ffi::F32> out_value, ffi::ResultBuffer<ffi::F32> out_std, ffi::ResultBuffer<ffi::F32> visit_counts,
                      ffi::ResultBuffer<ffi::F32> visit_probs, ffi::ResultBuffer<ffi::F32> qvalues, ffi::ResultBuffer<ffi::F32> qvar,
                      ffi::ResultBuffer<ffi::F32> root_value, ffi::ResultBuffer<ffi::F32> root_ube, ffi::ResultBuffer<ffi::U8> workspace,
                      int32_t env_kind, int32_t size, int32_t word_size, int32_t binary_encoding, int32_t reward_fn,
                      int32_t num_simulations, int32_t max_depth, int32_t max_num_considered_actions, float gumbel_scale, float discount,
                      int32_t two_players_game, int32_t exploration, float value_scale, float maxvisit_init, int32_t rescale_values,
                      int32_t flags, int32_t mlp_mode, int32_t fused_root, int32_t draw_gumbel, int32_t noise_seed, int32_t reuse_prepared,
                      int32_t hash_bits, int32_t hash_io, float max_u, float novelty_scale) {
  const int64_t B = beta.element_count();
  const eaz_env env = MakeEnv(env_kind, size, word_size, binary_encoding, reward_fn, action_map.untyped_data());
  const int32_t A = eaz_env_num_actions(&env);
  if (A <= 0) return EazError(EAZ_ERR_INVALID_ARG, "eaz_search (env)");
  if (!draw_gumbel && gumbel.element_count() != (size_t)(B * A)) return Bad("gumbel must be [B, num_actions]");
  if ((int64_t)action->element_count() != B || (int64_t)action_weights->element_count() != B * A) return Bad("result shapes must be [B] / [B, num_actions]");

  size_t i = 0;
  eaz_state st;
  EAZ_FFI_TRY(ReadStateArgs(rest, &i, env, B, &st));
  eaz_fc_params net;
  EAZ_FFI_TRY(ReadNet(rest, &i, env, binary_set.untyped_data(), hash_bits, hash_io, max_u, novelty_scale, &net));

  eaz_search_config cfg{};
  cfg.batch = (int32_t)B;
  cfg.num_simulations = num_simulations;
  cfg.max_depth = max_depth;
  cfg.max_num_considered_actions = max_num_considered_actions;
  cfg.gumbel_scale = gumbel_scale;
  cfg.discount = discount;
  cfg.two_players_game = two_players_game;
  cfg.exploration = exploration;
  cfg.value_scale = value_scale;
  cfg.maxvisit_init = maxvisit_init;
  cfg.rescale_values = rescale_values;
  cfg.use_mixed_value = 1;
  cfg.epsilon = 1e-8f;
  cfg.flags = flags;
  cfg.mlp_mode = mlp_mode;
  cfg.pb_c_init = 1.25f;
  cfg.pb_c_base = 19652.0f;
  cfg.temperature = 1.0f;
  cfg.noise_seed = (uint32_t)noise_seed;

  const size_t need = eaz_search_workspace_bytes(&cfg, &env);
  if (need == 0) return EazError(EAZ_ERR_INVALID_ARG, "eaz_search_workspace_bytes");
  void* ws = AlignUp(workspace->untyped_data(), 256);
  const size_t ws_bytes = workspace->size_bytes() - (size_t)((uint8_t*)ws - (uint8_t*)workspace->untyped_data());
  if (ws_bytes < need) return Bad("workspace result must hold eaz_search_workspace_bytes + 256 bytes");
  if (reuse_prepared) {  // only meaningful when XLA aliased workspace_in to the result (the tables of the previous call are in it)
    if (workspace_in.untyped_data() != workspace->untyped_data())
      return Bad("reuse_prepared needs input_output_aliases={workspace_in: workspace}: the tables live in the workspace");
    cfg.flags |= EAZ_FLAG_REUSE_PREPARED;
  }

  eaz_search_inputs in{};
  in.prior_logits = fused_root ? nullptr : prior_logits.typed_data();
  in.value = fused_root ? nullptr : value.typed_data();
  in.value_epistemic_variance = fused_root ? nullptr : variance.typed_data();
  in.beta = beta.typed_data();
  in.embedding = &st;
  in.invalid_actions = invalid.element_count() == (size_t)(B * A) ? static_cast<const uint8_t*>(invalid.untyped_data()) : nullptr;
  in.gumbel = draw_gumbel ? nullptr : gumbel.typed_data();
  in.env = &env;
  in.net = &net;

  eaz_search_outputs out{};
  out.action = action->typed_data();
  out.action_weights = action_weights->typed_data();
  out.value = out_value->typed_data();
  out.value_epistemic_std = out_std->typed_data();
  out.visit_counts = visit_counts->typed_data();
  out.visit_probs = visit_probs->typed_data();
  out.qvalues = qvalues->typed_data();
  out.qvalues_epistemic_variance = qvar->typed_data();
  if (fused_root) {
    out.root_value = root_value->typed_data();
    out.root_ube = root_ube->typed_data();
  }
  return EazError(eaz_search_gumbel(&cfg, &in, &out, ws, ws_bytes, stream), "eaz_search_gumbel");
}

// ------------------------------------------------------------------------------------------------ evaluation episodes
// args : beta F32[B], action_map, binary_set U8[2^(bits-3)], workspace_in U8[ws], then the initial state leaves (env.init), then the 24
//        parameter buffers
// rets : the final state leaves, returns F32[B] (sum of rewards per episode), workspace U8[eaz_evaluate_workspace_bytes + 256]
// The loop's CUDA graph is kept with the workspace address: alias workspace_in -> workspace and the state leaves to keep it across calls.
ffi::Error EvaluateImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> beta, ffi::AnyBuffer action_map, ffi::Buffer<ffi::U8> binary_set,
                        ffi::Buffer<ffi::U8> workspace_in, ffi::RemainingArgs rest, ffi::RemainingRets rets, int32_t env_kind, int32_t size,
                        int32_t word_size, int32_t binary_encoding, int32_t reward_fn, int32_t num_simulations, int32_t max_depth,
                        int32_t max_num_considered_actions, float discount, float value_scale, float maxvisit_init, int32_t rescale_values,
                        int32_t flags, int32_t mlp_mode, int32_t hash_bits, int32_t hash_io, float max_u, float novelty_scale,
                        int32_t max_episode_length) {
  (void)workspace_in;  // (only its aliasing matters: the result `workspace` is the buffer the library uses)
  const int64_t B = beta.element_count();
  const eaz_env env = MakeEnv(env_kind, size, word_size, binary_encoding, reward_fn, action_map.untyped_data());
  if (eaz_env_num_actions(&env) <= 0) return EazError(EAZ_ERR_INVALID_ARG, "EazEvaluate (env)");
  const size_t nl = NumLeaves(env);
  if (rest.size() != nl + 24) return Bad("EazEvaluate: expected the state leaves and 24 parameter buffers");
  if (rets.size() != nl + 2) return Bad("EazEvaluate: expected the state leaves, returns and workspace as results");
  size_t i = 0, j = 0;
  eaz_state src, st;
  EAZ_FFI_TRY(ReadStateArgs(rest, &i, env, B, &src));
  eaz_fc_params net;
  EAZ_FFI_TRY(ReadNet(rest, &i, env, binary_set.untyped_data(), hash_bits, hash_io, max_u, novelty_scale, &net));
  EAZ_FFI_TRY(ReadStateRets(rets, &j, env, B, &st));
  float* returns = nullptr;
  EAZ_FFI_TRY(GetRet(rets, j++, "returns", &returns, B));
  auto workspace = rets.get<ffi::AnyBuffer>(j);
  if (!workspace.has_value()) return workspace.error();

  eaz_search_config cfg{};
  cfg.batch = (int32_t)B;
  cfg.num_simulations = num_simulations;
  cfg.max_depth = max_depth;
  cfg.max_num_considered_actions = max_num_considered_actions;
  cfg.gumbel_scale = 0.0f;  // evaluate.py:44
  cfg.discount = discount;
  cfg.exploration = 0;      // the exploitation head (evaluate.py:29-35)
  cfg.value_scale = value_scale;
  cfg.maxvisit_init = maxvisit_init;
  cfg.rescale_values = rescale_values;
  cfg.use_mixed_value = 1;
  cfg.epsilon = 1e-8f;
  cfg.flags = flags & ~EAZ_FLAG_REUSE_PREPARED;
  cfg.mlp_mode = mlp_mode;
  cfg.pb_c_init = 1.25f;
  cfg.pb_c_base = 19652.0f;
  cfg.temperature = 1.0f;

  const size_t need = eaz_evaluate_workspace_bytes(&cfg, &env);
  if (need == 0) return EazError(EAZ_ERR_INVALID_ARG, "eaz_evaluate_workspace_bytes");
  void* ws = AlignUp((*workspace)->untyped_data(), 256);
  const size_t pad = (size_t)((uint8_t*)ws - (uint8_t*)(*workspace)->untyped_data());
  if ((*workspace)->size_bytes() < pad + need) return Bad("workspace result must hold eaz_evaluate_workspace_bytes + 256 bytes");
  EAZ_FFI_TRY(CopyState(env, src, st, B, stream));

  eaz_search_inputs in{};
  in.beta = beta.typed_data();
  in.env = &env;
  return EazError(eaz_evaluate(&cfg, &in, &net, &st, returns, max_episode_length, ws, (*workspace)->size_bytes() - pad, stream), "eaz_evaluate");
}

// ------------------------------------------------------------------------------------------------ self-play scan
// args : beta F32[B], action_map, binary_set U8[2^(bits-3)], gumbel F32[T,B,A], sample_gumbel F32[T,B,A], task_ids S32[T,B] (each of
//        the three: any 1-element dummy = not given -- the noise is then drawn in the search, the task ids are required for Subleq),
//        workspace_in U8[ws] (alias it to `workspace` to keep the graph, and with reuse_prepared the tables, across calls), then the
//        initial state leaves, then the 24 parameter buffers
// rets : the final state leaves, action S32[T,B], root_value F32[T,B], root_epistemic_std F32[T,B], value_prediction F32[T,B],
//        ube_prediction F32[T,B], q_values_epistemic_variance F32[T,B,A], trajectory S32[T,B,4], states U8[T,B,S] (the states after
//        each step, eaz_env_compact records), rewards F32[T,B], workspace U8[eaz_selfplay_workspace_bytes + 256]
ffi::Error SelfplayImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> beta, ffi::AnyBuffer action_map, ffi::Buffer<ffi::U8> binary_set,
                        ffi::Buffer<ffi::F32> gumbel, ffi::Buffer<ffi::F32> sample_gumbel, ffi::Buffer<ffi::S32> task_ids,
                        ffi::Buffer<ffi::U8> workspace_in, ffi::RemainingArgs rest, ffi::RemainingRets rets, int32_t env_kind, int32_t size,
                        int32_t word_size, int32_t binary_encoding, int32_t reward_fn, int32_t num_simulations, int32_t max_depth,
                        int32_t max_num_considered_actions, float gumbel_scale, float discount, int32_t two_players_game, int32_t exploration,
                        float value_scale, float maxvisit_init, int32_t rescale_values, int32_t flags, int32_t mlp_mode, int32_t hash_bits,
                        int32_t hash_io, float max_u, float novelty_scale, int32_t steps, int32_t root_prior, int32_t action_sampling,
                        float temperature, int32_t noise_seed, int32_t reuse_prepared) {
  const int64_t B = beta.element_count(), T = steps;
  const eaz_env env = MakeEnv(env_kind, size, word_size, binary_encoding, reward_fn, action_map.untyped_data());
  const int32_t A = eaz_env_num_actions(&env), S = eaz_env_compact_bytes(&env);
  if (A <= 0 || S <= 0) return EazError(EAZ_ERR_INVALID_ARG, "EazSelfplay (env)");
  if (T < 0) return Bad("EazSelfplay: steps must be >= 0");
  const size_t nl = NumLeaves(env);
  if (rest.size() != nl + 24) return Bad("EazSelfplay: expected the state leaves and 24 parameter buffers");
  if (rets.size() != nl + 10) return Bad("EazSelfplay: expected the state leaves, the 9 stacked outputs and workspace as results");
  const bool noise = (int64_t)gumbel.element_count() == T * B * A, sample = (int64_t)sample_gumbel.element_count() == T * B * A,
             tasks = (int64_t)task_ids.element_count() == T * B;
  if (!noise && gumbel.element_count() != 1) return Bad("EazSelfplay: gumbel must be [steps, B, num_actions] or a 1-element dummy");
  if (!sample && sample_gumbel.element_count() != 1) return Bad("EazSelfplay: sample_gumbel must be [steps, B, num_actions] or a 1-element dummy");
  if (!tasks && task_ids.element_count() != 1) return Bad("EazSelfplay: task_ids must be [steps, B] or a 1-element dummy");
  size_t i = 0, j = 0;
  eaz_state src, st;
  EAZ_FFI_TRY(ReadStateArgs(rest, &i, env, B, &src));
  eaz_fc_params net;
  EAZ_FFI_TRY(ReadNet(rest, &i, env, binary_set.untyped_data(), hash_bits, hash_io, max_u, novelty_scale, &net));
  EAZ_FFI_TRY(ReadStateRets(rets, &j, env, B, &st));
  eaz_selfplay_outputs out{};
  EAZ_FFI_TRY(GetRet(rets, j++, "action", &out.action, T * B));
  EAZ_FFI_TRY(GetRet(rets, j++, "root_value", &out.root_value, T * B));
  EAZ_FFI_TRY(GetRet(rets, j++, "root_epistemic_std", &out.root_epistemic_std, T * B));
  EAZ_FFI_TRY(GetRet(rets, j++, "value_prediction", &out.value_prediction, T * B));
  EAZ_FFI_TRY(GetRet(rets, j++, "ube_prediction", &out.ube_prediction, T * B));
  EAZ_FFI_TRY(GetRet(rets, j++, "q_values_epistemic_variance", &out.q_values_epistemic_variance, T * B * A));
  EAZ_FFI_TRY(GetRet(rets, j++, "trajectory", &out.trajectory, T * B * 4));
  EAZ_FFI_TRY(GetRet(rets, j++, "states", &out.states, T * B * S));
  EAZ_FFI_TRY(GetRet(rets, j++, "rewards", &out.rewards, T * B));
  auto workspace = rets.get<ffi::AnyBuffer>(j);
  if (!workspace.has_value()) return workspace.error();

  eaz_search_config cfg{};
  cfg.batch = (int32_t)B;
  cfg.num_simulations = num_simulations;
  cfg.max_depth = max_depth;
  cfg.max_num_considered_actions = max_num_considered_actions;
  cfg.gumbel_scale = gumbel_scale;
  cfg.discount = discount;
  cfg.two_players_game = two_players_game;
  cfg.exploration = exploration;
  cfg.value_scale = value_scale;
  cfg.maxvisit_init = maxvisit_init;
  cfg.rescale_values = rescale_values;
  cfg.use_mixed_value = 1;
  cfg.epsilon = 1e-8f;
  cfg.flags = flags & ~EAZ_FLAG_REUSE_PREPARED;
  cfg.mlp_mode = mlp_mode;
  cfg.pb_c_init = 1.25f;
  cfg.pb_c_base = 19652.0f;
  cfg.temperature = temperature;
  cfg.noise_seed = (uint32_t)noise_seed;
  cfg.root_prior = root_prior;
  cfg.action_sampling = action_sampling;

  const size_t need = eaz_selfplay_workspace_bytes(&cfg, &env);
  if (need == 0) return EazError(EAZ_ERR_INVALID_ARG, "eaz_selfplay_workspace_bytes");
  void* ws = AlignUp((*workspace)->untyped_data(), 256);
  const size_t pad = (size_t)((uint8_t*)ws - (uint8_t*)(*workspace)->untyped_data());
  if ((*workspace)->size_bytes() < pad + need) return Bad("workspace result must hold eaz_selfplay_workspace_bytes + 256 bytes");
  if (reuse_prepared) {  // only meaningful when XLA aliased workspace_in to the result (the tables of the previous call are in it)
    if (workspace_in.untyped_data() != (*workspace)->untyped_data())
      return Bad("reuse_prepared needs input_output_aliases={workspace_in: workspace}: the tables live in the workspace");
    cfg.flags |= EAZ_FLAG_REUSE_PREPARED;
  }
  EAZ_FFI_TRY(CopyState(env, src, st, B, stream));

  eaz_search_inputs in{};
  in.beta = beta.typed_data();
  in.gumbel = noise ? gumbel.typed_data() : nullptr;
  in.sample_gumbel = sample ? sample_gumbel.typed_data() : nullptr;
  in.env = &env;
  return EazError(eaz_selfplay(&cfg, &in, &net, &st, (int32_t)T, tasks ? task_ids.typed_data() : nullptr, &out, ws,
                               (*workspace)->size_bytes() - pad, stream),
                  "eaz_selfplay");
}

// ------------------------------------------------------------------------------------------------ env step / init
// args : action S32[B], task_ids S32[B] (pre-drawn reset tasks; any 1-element dummy for DeepSea), action_map, then the state leaves
// rets : the stepped state leaves (same order).  With input_output_aliases the step runs in place, else the leaves are copied first.
ffi::Error EnvStepImpl(cudaStream_t stream, ffi::Buffer<ffi::S32> action, ffi::Buffer<ffi::S32> task_ids, ffi::AnyBuffer action_map,
                       ffi::RemainingArgs leaves, ffi::RemainingRets out_leaves, int32_t env_kind, int32_t size, int32_t word_size,
                       int32_t binary_encoding, int32_t reward_fn, int32_t auto_reset) {
  const int64_t B = action.element_count();
  const eaz_env env = MakeEnv(env_kind, size, word_size, binary_encoding, reward_fn, action_map.untyped_data());
  if (leaves.size() != NumLeaves(env) || out_leaves.size() != NumLeaves(env)) return Bad("eaz_env_step: wrong number of state leaves");
  size_t i = 0, j = 0;
  eaz_state src, dst;
  EAZ_FFI_TRY(ReadStateArgs(leaves, &i, env, B, &src));
  EAZ_FFI_TRY(ReadStateRets(out_leaves, &j, env, B, &dst));
  EAZ_FFI_TRY(CopyState(env, src, dst, B, stream));
  const int32_t* tasks = (env.kind == EAZ_ENV_SUBLEQ && (int64_t)task_ids.element_count() == B) ? task_ids.typed_data() : nullptr;
  return EazError(eaz_env_step(&env, &dst, action.typed_data(), auto_reset, tasks, (int32_t)B, stream), "eaz_env_step");
}

// args : task_ids S32[B], action_map;  rets : the initial state leaves
ffi::Error EnvInitImpl(cudaStream_t stream, ffi::Buffer<ffi::S32> task_ids, ffi::AnyBuffer action_map, ffi::RemainingRets out_leaves,
                       int32_t env_kind, int32_t size, int32_t word_size, int32_t binary_encoding, int32_t reward_fn, int32_t batch) {
  const eaz_env env = MakeEnv(env_kind, size, word_size, binary_encoding, reward_fn, action_map.untyped_data());
  if (out_leaves.size() != NumLeaves(env)) return Bad("eaz_env_init: wrong number of state leaves");
  size_t j = 0;
  eaz_state dst;
  EAZ_FFI_TRY(ReadStateRets(out_leaves, &j, env, batch, &dst));
  const int32_t* tasks = (env.kind == EAZ_ENV_SUBLEQ && (int64_t)task_ids.element_count() == batch) ? task_ids.typed_data() : nullptr;
  return EazError(eaz_env_init(&env, tasks, &dst, batch, stream), "eaz_env_init");
}

// ------------------------------------------------------------------------------------------------ network on env states
// args : action_map, binary_set, then the state leaves, then the 24 parameter buffers
// rets : exploit_logits F32[B,A], explore_logits F32[B,A], value F32[B], ube F32[B], novelty F32[B], scratch U8[B * compact_bytes + 16]
ffi::Error MlpForwardStatesImpl(cudaStream_t stream, ffi::AnyBuffer action_map, ffi::Buffer<ffi::U8> binary_set, ffi::RemainingArgs rest,
                                ffi::ResultBuffer<ffi::F32> exploit_logits, ffi::ResultBuffer<ffi::F32> explore_logits,
                                ffi::ResultBuffer<ffi::F32> value, ffi::ResultBuffer<ffi::F32> ube, ffi::ResultBuffer<ffi::F32> novelty,
                                ffi::ResultBuffer<ffi::U8> scratch, int32_t env_kind, int32_t size, int32_t word_size,
                                int32_t binary_encoding, int32_t reward_fn, int32_t hash_bits, int32_t hash_io, float max_u,
                                float novelty_scale) {
  const int64_t B = value->element_count();
  const eaz_env env = MakeEnv(env_kind, size, word_size, binary_encoding, reward_fn, action_map.untyped_data());
  size_t i = 0;
  eaz_state st;
  EAZ_FFI_TRY(ReadStateArgs(rest, &i, env, B, &st));
  eaz_fc_params net;
  EAZ_FFI_TRY(ReadNet(rest, &i, env, binary_set.untyped_data(), hash_bits, hash_io, max_u, novelty_scale, &net));
  void* ws = AlignUp(scratch->untyped_data(), 16);
  const size_t ws_bytes = scratch->size_bytes() - (size_t)((uint8_t*)ws - (uint8_t*)scratch->untyped_data());
  return EazError(eaz_mlp_forward_states(&net, &env, &st, (int32_t)B, exploit_logits->typed_data(), explore_logits->typed_data(),
                                         value->typed_data(), ube->typed_data(), novelty->typed_data(), ws, ws_bytes, stream),
                  "eaz_mlp_forward_states");
}

// ------------------------------------------------------------------------------------------------ reanalyze targets
ffi::Error ReanalyzeTargetsImpl(cudaStream_t stream, ffi::Buffer<ffi::S32> action, ffi::Buffer<ffi::F32> qvalues, ffi::Buffer<ffi::F32> qvar,
                                ffi::Buffer<ffi::F32> visit_counts, ffi::Buffer<ffi::F32> value, ffi::Buffer<ffi::F32> value_std,
                                ffi::Buffer<ffi::F32> next_state_value, ffi::Buffer<ffi::F32> next_rewards, ffi::AnyBuffer next_terminated,
                                ffi::AnyBuffer terminated, ffi::AnyBuffer invalid_actions, ffi::ResultBuffer<ffi::F32> value_target,
                                ffi::ResultBuffer<ffi::F32> ube_target, ffi::ResultBuffer<ffi::F32> exploration_policy_target,
                                float discount, float exploration_beta, int32_t exploration_ube_target, float temperature) {
  const int64_t B = action.element_count();
  if (B <= 0 || qvalues.element_count() % (size_t)B != 0) return Bad("qvalues must be [B, A]");
  const int64_t A = (int64_t)qvalues.element_count() / B;
  eaz_reanalyze_config cfg{discount, exploration_beta, exploration_ube_target, temperature};
  const uint8_t* inv = (int64_t)invalid_actions.element_count() == B * A ? static_cast<const uint8_t*>(invalid_actions.untyped_data()) : nullptr;
  return EazError(eaz_reanalyze_targets(&cfg, (int32_t)B, (int32_t)A, action.typed_data(), qvalues.typed_data(), qvar.typed_data(),
                                        visit_counts.typed_data(), value.typed_data(), value_std.typed_data(), next_state_value.typed_data(),
                                        next_rewards.typed_data(), static_cast<const uint8_t*>(next_terminated.untyped_data()),
                                        static_cast<const uint8_t*>(terminated.untyped_data()), inv, value_target->typed_data(),
                                        ube_target->typed_data(), exploration_policy_target->typed_data(), stream),
                  "eaz_reanalyze_targets");
}

// ------------------------------------------------------------------------------------------------ hash update (train.py:22)
// args : x F32[B,D] (the hashed observation rows as float32), binary_set_in U8[..];  rets : binary_set U8[..] (alias it to the input)
ffi::Error HashUpdateImpl(cudaStream_t stream, ffi::Buffer<ffi::F32> x, ffi::Buffer<ffi::U8> binary_set_in, ffi::ResultBuffer<ffi::U8> binary_set,
                          int32_t bits) {
  const auto dims = x.dimensions();
  if (dims.size() != 2) return Bad("x must be [B, D]");
  if (binary_set->untyped_data() != binary_set_in.untyped_data()) {
    const cudaError_t e = cudaMemcpyAsync(binary_set->untyped_data(), binary_set_in.untyped_data(), binary_set_in.size_bytes(),
                                          cudaMemcpyDeviceToDevice, stream);
    if (e != cudaSuccess) return ffi::Error(ffi::ErrorCode::kInternal, cudaGetErrorString(e));
  }
  return EazError(eaz_hash_update(x.typed_data(), (int32_t)dims[0], (int32_t)dims[1], bits, binary_set->typed_data(), stream), "eaz_hash_update");
}

// ------------------------------------------------------------------------------------------------ prioritised replay ring
// flashbax's prioritised flat buffer (main.py:217-225, 383-385, 413-414, 454) as three arrays the program threads through its
// calls: ring_states U8[T,B,S] (eaz_env_compact records), ring_rewards F32[T,B] and the sum tree U8[eaz_priority_tree_bytes(T, B)],
// whose header holds the write cursor, so no call needs a host value.  Every check below runs before anything touches a device.

// T >= 2, B >= 1, T * B < 2^31, and a 128-byte aligned tree buffer of at least eaz_priority_tree_bytes(T, B)
template <typename Buf>
ffi::Error CheckTree(const Buf& tree, int64_t T, int64_t B, size_t* bytes) {
  if (T < 2 || B < 1 || T > INT32_MAX || B > INT32_MAX || T * B >= ((int64_t)1 << 31))
    return Bad("replay: need T >= 2 time slots, B >= 1 envs and T * B < 2^31 (got T=" + std::to_string(T) + ", B=" + std::to_string(B) + ")");
  const size_t need = eaz_priority_tree_bytes((int32_t)T, (int32_t)B);
  if (need == 0) return EazError(EAZ_ERR_INVALID_ARG, "eaz_priority_tree_bytes");
  if (tree.size_bytes() < need)
    return Bad("replay: tree buffer of " + std::to_string(tree.size_bytes()) + " bytes, eaz_priority_tree_bytes = " + std::to_string(need));
  if (reinterpret_cast<uintptr_t>(tree.untyped_data()) % 128 != 0) return Bad("replay: the tree buffer must be 128-byte aligned");
  *bytes = tree.size_bytes();
  return ffi::Error::Success();
}

// ring_states [T,B,S] and ring_rewards [T,B] -> T, B, S
template <typename BufS, typename BufR>
ffi::Error RingDims(const BufS& states, const BufR& rewards, int64_t* T, int64_t* B, int64_t* S) {
  const auto ds = states.dimensions();
  const auto dr = rewards.dimensions();
  if (ds.size() != 3 || dr.size() != 2 || dr[0] != ds[0] || dr[1] != ds[1]) return Bad("replay: ring_states must be [T, B, S] and ring_rewards [T, B]");
  *T = ds[0], *B = ds[1], *S = ds[2];
  return ffi::Error::Success();
}

// S must be the env's compact record size
ffi::Error CheckRecord(const eaz_env& env, int64_t S) {
  const int32_t cb = eaz_env_compact_bytes(&env);
  if (cb <= 0) return EazError(EAZ_ERR_INVALID_ARG, "eaz_env_compact_bytes");
  if (S != cb) return Bad("replay: ring_states must be [T, B, eaz_env_compact_bytes = " + std::to_string(cb) + "]");
  return ffi::Error::Success();
}

// the state leaves starting at src[first] hold exactly n envs each
int64_t LeafElems(const eaz_env& env, size_t k) {  // elements per env of leaf k (eaz_state order)
  if (k < kCommonLeaves || env.kind == EAZ_ENV_DEEPSEA) return 1;
  return k == kCommonLeaves ? env.word_size : k >= kCommonLeaves + 3 ? EAZ_SUBLEQ_IO_LEN : 1;
}
ffi::Error CheckLeafRows(ffi::RemainingArgs& args, size_t first, const eaz_env& env, int64_t n) {
  for (size_t k = 0; k < NumLeaves(env); ++k) {
    auto b = args.get<ffi::AnyBuffer>(first + k);
    if (!b.has_value()) return b.error();
    if ((int64_t)b->element_count() != n * LeafElems(env, k)) return Bad("replay: state leaf " + std::to_string(k) + " does not hold " + std::to_string(n) + " envs");
  }
  return ffi::Error::Success();
}
ffi::Error CheckLeafRows(ffi::RemainingRets& rets, size_t first, const eaz_env& env, int64_t n) {
  for (size_t k = 0; k < NumLeaves(env); ++k) {
    auto b = rets.get<ffi::AnyBuffer>(first + k);
    if (!b.has_value()) return b.error();
    if ((int64_t)(*b)->element_count() != n * LeafElems(env, k)) return Bad("replay: result leaf " + std::to_string(k) + " does not hold " + std::to_string(n) + " envs");
  }
  return ffi::Error::Success();
}

// the functional form of an aliased update: without input_output_aliases the result starts as a copy of the input
ffi::Error CopyUnlessAliased(void* dst, const void* src, size_t bytes, cudaStream_t stream) {
  if (dst == src || bytes == 0) return ffi::Error::Success();
  const cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, stream);
  if (e != cudaSuccess) return ffi::Error(ffi::ErrorCode::kInternal, std::string("replay copy: ") + cudaGetErrorString(e));
  return ffi::Error::Success();
}

// rets : ring_states U8[T,B,S], ring_rewards F32[T,B] (both zeroed), tree U8[eaz_priority_tree_bytes(T, B)]
ffi::Error ReplayInitImpl(cudaStream_t stream, ffi::ResultBuffer<ffi::U8> ring_states, ffi::ResultBuffer<ffi::F32> ring_rewards,
                          ffi::ResultBuffer<ffi::U8> tree, int32_t T, int32_t B, float priority_exponent, int32_t seed) {
  size_t tree_bytes = 0;
  EAZ_FFI_TRY(CheckTree(*tree, T, B, &tree_bytes));
  int64_t t, b, S;
  EAZ_FFI_TRY(RingDims(*ring_states, *ring_rewards, &t, &b, &S));
  if (t != T || b != B) return Bad("EazReplayInit: ring_states must be [T, B, S] and ring_rewards [T, B]");
  if (!(priority_exponent >= 0.0f && priority_exponent <= 1.0f)) return Bad("EazReplayInit: priority_exponent must lie in [0, 1]");
  cudaError_t e = cudaMemsetAsync(ring_states->untyped_data(), 0, ring_states->size_bytes(), stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(ring_rewards->untyped_data(), 0, ring_rewards->size_bytes(), stream);
  if (e != cudaSuccess) return ffi::Error(ffi::ErrorCode::kInternal, std::string("ring memset: ") + cudaGetErrorString(e));
  return EazError(eaz_priority_init(tree->untyped_data(), tree_bytes, T, B, priority_exponent, (uint32_t)seed, stream), "eaz_priority_init");
}

// args : action_map, ring_states_in U8[T,B,S], ring_rewards_in F32[T,B], tree_in U8, then the state leaves of the B envs
// rets : ring_states, ring_rewards, tree (alias each to its input; otherwise the inputs are copied first)
ffi::Error ReplayAddImpl(cudaStream_t stream, ffi::AnyBuffer action_map, ffi::Buffer<ffi::U8> states_in, ffi::Buffer<ffi::F32> rewards_in,
                         ffi::Buffer<ffi::U8> tree_in, ffi::RemainingArgs leaves, ffi::ResultBuffer<ffi::U8> ring_states,
                         ffi::ResultBuffer<ffi::F32> ring_rewards, ffi::ResultBuffer<ffi::U8> tree, int32_t env_kind, int32_t size,
                         int32_t word_size, int32_t binary_encoding, int32_t reward_fn) {
  const eaz_env env = MakeEnv(env_kind, size, word_size, binary_encoding, reward_fn, action_map.untyped_data());
  int64_t T, B, S;
  EAZ_FFI_TRY(RingDims(states_in, rewards_in, &T, &B, &S));
  size_t in_bytes = 0, tree_bytes = 0;
  EAZ_FFI_TRY(CheckTree(tree_in, T, B, &in_bytes));
  EAZ_FFI_TRY(CheckTree(*tree, T, B, &tree_bytes));
  EAZ_FFI_TRY(CheckRecord(env, S));
  if (ring_states->size_bytes() != states_in.size_bytes() || ring_rewards->size_bytes() != rewards_in.size_bytes() || tree_bytes != in_bytes)
    return Bad("EazReplayAdd: each result must have the shape of its input");
  if (leaves.size() != NumLeaves(env)) return Bad("EazReplayAdd: wrong number of state leaves");
  EAZ_FFI_TRY(CheckLeafRows(leaves, 0, env, B));
  size_t i = 0;
  eaz_state st;
  EAZ_FFI_TRY(ReadStateArgs(leaves, &i, env, B, &st));
  EAZ_FFI_TRY(CopyUnlessAliased(ring_states->untyped_data(), states_in.untyped_data(), states_in.size_bytes(), stream));
  EAZ_FFI_TRY(CopyUnlessAliased(ring_rewards->untyped_data(), rewards_in.untyped_data(), rewards_in.size_bytes(), stream));
  EAZ_FFI_TRY(CopyUnlessAliased(tree->untyped_data(), tree_in.untyped_data(), in_bytes, stream));
  return EazError(eaz_replay_add(&env, &st, ring_states->typed_data(), ring_rewards->typed_data(), tree->untyped_data(), tree_bytes, (int32_t)T,
                                 (int32_t)B, stream),
                  "eaz_replay_add");
}

// args : action_map, ring_states_in U8[T,B,S], ring_rewards_in F32[T,B], tree_in U8, compact U8[T',B,S], rewards F32[T',B] (a scan's
//        SelfplayOutput.state: T' time steps of the B envs, appended in time order at the device cursor)
// rets : ring_states, ring_rewards, tree (alias each to its input; otherwise the inputs are copied first)
ffi::Error ReplayAddSequenceImpl(cudaStream_t stream, ffi::AnyBuffer action_map, ffi::Buffer<ffi::U8> states_in, ffi::Buffer<ffi::F32> rewards_in,
                                 ffi::Buffer<ffi::U8> tree_in, ffi::Buffer<ffi::U8> compact, ffi::Buffer<ffi::F32> rewards,
                                 ffi::ResultBuffer<ffi::U8> ring_states, ffi::ResultBuffer<ffi::F32> ring_rewards, ffi::ResultBuffer<ffi::U8> tree,
                                 int32_t env_kind, int32_t size, int32_t word_size, int32_t binary_encoding, int32_t reward_fn) {
  const eaz_env env = MakeEnv(env_kind, size, word_size, binary_encoding, reward_fn, action_map.untyped_data());
  int64_t T, B, S;
  EAZ_FFI_TRY(RingDims(states_in, rewards_in, &T, &B, &S));
  size_t in_bytes = 0, tree_bytes = 0;
  EAZ_FFI_TRY(CheckTree(tree_in, T, B, &in_bytes));
  EAZ_FFI_TRY(CheckTree(*tree, T, B, &tree_bytes));
  EAZ_FFI_TRY(CheckRecord(env, S));
  if (ring_states->size_bytes() != states_in.size_bytes() || ring_rewards->size_bytes() != rewards_in.size_bytes() || tree_bytes != in_bytes)
    return Bad("EazReplayAddSequence: each result must have the shape of its input");
  const auto dc = compact.dimensions();
  const auto dr = rewards.dimensions();
  if (dc.size() != 3 || dc[1] != B || dc[2] != S)
    return Bad("EazReplayAddSequence: compact must be [T', B, S] = [T', " + std::to_string(B) + ", " + std::to_string(S) + "] for the ring's B envs");
  if (dr.size() != 2 || dr[0] != dc[0] || dr[1] != B)
    return Bad("EazReplayAddSequence: rewards must be [T', B] = [" + std::to_string(dc[0]) + ", " + std::to_string(B) + "]");
  if (dc[0] >= INT32_MAX) return Bad("EazReplayAddSequence: T' = " + std::to_string(dc[0]) + " time steps, at most 2^31 - 2");
  EAZ_FFI_TRY(CopyUnlessAliased(ring_states->untyped_data(), states_in.untyped_data(), states_in.size_bytes(), stream));
  EAZ_FFI_TRY(CopyUnlessAliased(ring_rewards->untyped_data(), rewards_in.untyped_data(), rewards_in.size_bytes(), stream));
  EAZ_FFI_TRY(CopyUnlessAliased(tree->untyped_data(), tree_in.untyped_data(), in_bytes, stream));
  return EazError(eaz_replay_add_sequence(&env, compact.typed_data(), rewards.typed_data(), (int32_t)dc[0], ring_states->typed_data(),
                                          ring_rewards->typed_data(), tree->untyped_data(), tree_bytes, (int32_t)T, (int32_t)B, (int32_t)S, stream),
                  "eaz_replay_add_sequence");
}

// args : action_map, ring_states U8[T,B,S], ring_rewards F32[T,B], tree U8, key U32[2] = (seed, draw counter); none is aliased or written
// rets : indices S32[K], probabilities F32[K], the decoded `first` state leaves (K envs), the `second` state leaves,
//        scratch U8[2 K (S + 4) + 16] (the gathered compact records and rewards)
ffi::Error ReplaySampleImpl(cudaStream_t stream, ffi::AnyBuffer action_map, ffi::Buffer<ffi::U8> ring_states, ffi::Buffer<ffi::F32> ring_rewards,
                            ffi::Buffer<ffi::U8> tree, ffi::Buffer<ffi::U32> key, ffi::ResultBuffer<ffi::S32> indices,
                            ffi::ResultBuffer<ffi::F32> probabilities, ffi::RemainingRets out, int32_t env_kind, int32_t size, int32_t word_size,
                            int32_t binary_encoding, int32_t reward_fn, int32_t K) {
  const eaz_env env = MakeEnv(env_kind, size, word_size, binary_encoding, reward_fn, action_map.untyped_data());
  int64_t T, B, S;
  EAZ_FFI_TRY(RingDims(ring_states, ring_rewards, &T, &B, &S));
  size_t tree_bytes = 0;
  EAZ_FFI_TRY(CheckTree(tree, T, B, &tree_bytes));
  EAZ_FFI_TRY(CheckRecord(env, S));
  if (K < 1 || K > (1 << 24)) return Bad("EazReplaySample: K = " + std::to_string(K) + " outside [1, 2^24]");
  if (key.element_count() != 2) return Bad("EazReplaySample: key must be U32[2]");
  if ((int64_t)indices->element_count() != K || (int64_t)probabilities->element_count() != K) return Bad("EazReplaySample: indices / probabilities must be [K]");
  const size_t nl = NumLeaves(env);
  if (out.size() != 2 * nl + 1) return Bad("EazReplaySample: wrong number of results (first leaves, second leaves, scratch)");
  EAZ_FFI_TRY(CheckLeafRows(out, 0, env, K));
  EAZ_FFI_TRY(CheckLeafRows(out, nl, env, K));
  size_t j = 0;
  eaz_state first, second;
  EAZ_FFI_TRY(ReadStateRets(out, &j, env, K, &first));
  EAZ_FFI_TRY(ReadStateRets(out, &j, env, K, &second));
  auto scratch = out.get<ffi::AnyBuffer>(j);
  if (!scratch.has_value()) return scratch.error();
  void* ws = AlignUp((*scratch)->untyped_data(), 16);
  const size_t ws_bytes = (*scratch)->size_bytes() - std::min((*scratch)->size_bytes(), (size_t)((uint8_t*)ws - (uint8_t*)(*scratch)->untyped_data()));
  if (ws_bytes < (size_t)2 * K * (S + 4)) return Bad("EazReplaySample: scratch must hold 2 K (S + 4) + 16 bytes");
  float* first_r = static_cast<float*>(ws);
  float* second_r = first_r + K;
  uint8_t* first_c = reinterpret_cast<uint8_t*>(second_r + K);
  uint8_t* second_c = first_c + (size_t)K * S;
  EAZ_FFI_TRY(EazError(eaz_priority_sample_keyed(tree.untyped_data(), tree_bytes, (int32_t)T, (int32_t)B, K, key.typed_data(),
                                                 ring_states.typed_data(), ring_rewards.typed_data(), (int32_t)S, indices->typed_data(),
                                                 probabilities->typed_data(), first_c, first_r, second_c, second_r, stream),
                       "eaz_priority_sample_keyed"));
  EAZ_FFI_TRY(EazError(eaz_env_uncompact(&env, first_c, first_r, &first, K, stream), "eaz_env_uncompact"));
  return EazError(eaz_env_uncompact(&env, second_c, second_r, &second, K, stream), "eaz_env_uncompact");
}

// args : indices S32[K], priorities F32[K], tree_in U8;  rets : tree (alias it to tree_in)
ffi::Error ReplaySetPrioritiesImpl(cudaStream_t stream, ffi::Buffer<ffi::S32> indices, ffi::Buffer<ffi::F32> priorities, ffi::Buffer<ffi::U8> tree_in,
                                   ffi::ResultBuffer<ffi::U8> tree, int32_t T, int32_t B) {
  size_t in_bytes = 0, tree_bytes = 0;
  EAZ_FFI_TRY(CheckTree(tree_in, T, B, &in_bytes));
  EAZ_FFI_TRY(CheckTree(*tree, T, B, &tree_bytes));
  if (tree_bytes != in_bytes) return Bad("EazReplaySetPriorities: the tree result must have the shape of tree_in");
  const size_t K = indices.element_count();
  if (priorities.element_count() != K) return Bad("EazReplaySetPriorities: indices and priorities differ in length");
  if (K > (size_t)INT32_MAX) return Bad("EazReplaySetPriorities: more than 2^31 - 1 entries");
  EAZ_FFI_TRY(CopyUnlessAliased(tree->untyped_data(), tree_in.untyped_data(), in_bytes, stream));
  return EazError(eaz_priority_set(tree->untyped_data(), tree_bytes, T, B, indices.typed_data(), priorities.typed_data(), (int32_t)K, stream),
                  "eaz_priority_set");
}

// args : tree U8;  rets : flags S32[1], the sticky EAZ_PRIORITY_* bits (copied on the stream, no synchronisation)
ffi::Error ReplayStatusImpl(cudaStream_t stream, ffi::Buffer<ffi::U8> tree, ffi::ResultBuffer<ffi::S32> flags) {
  if (reinterpret_cast<uintptr_t>(tree.untyped_data()) % 128 != 0) return Bad("replay: the tree buffer must be 128-byte aligned");
  if (flags->element_count() != 1) return Bad("EazReplayStatus: flags must be S32[1]");
  return EazError(eaz_priority_status_async(tree.untyped_data(), tree.size_bytes(), flags->typed_data(), stream), "eaz_priority_status_async");
}

}  // namespace

#define EAZ_ENV_ATTRS() \
  .Attr<int32_t>("env_kind").Attr<int32_t>("size").Attr<int32_t>("word_size").Attr<int32_t>("binary_encoding").Attr<int32_t>("reward_fn")

XLA_FFI_DEFINE_HANDLER_SYMBOL(EazSearch, SearchImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()  // beta
                                  .Arg<ffi::Buffer<ffi::F32>>()  // gumbel
                                  .Arg<ffi::AnyBuffer>()         // invalid_actions
                                  .Arg<ffi::AnyBuffer>()         // action_map
                                  .Arg<ffi::Buffer<ffi::U8>>()   // binary_set
                                  .Arg<ffi::Buffer<ffi::F32>>()  // root prior_logits
                                  .Arg<ffi::Buffer<ffi::F32>>()  // root value
                                  .Arg<ffi::Buffer<ffi::F32>>()  // root value_epistemic_variance
                                  .Arg<ffi::Buffer<ffi::U8>>()   // workspace_in
                                  .RemainingArgs()               // state leaves, 24 parameter buffers
                                  .Ret<ffi::Buffer<ffi::S32>>()  // action
                                  .Ret<ffi::Buffer<ffi::F32>>()  // action_weights
                                  .Ret<ffi::Buffer<ffi::F32>>()  // value
                                  .Ret<ffi::Buffer<ffi::F32>>()  // value_epistemic_std
                                  .Ret<ffi::Buffer<ffi::F32>>()  // visit_counts
                                  .Ret<ffi::Buffer<ffi::F32>>()  // visit_probs
                                  .Ret<ffi::Buffer<ffi::F32>>()  // qvalues
                                  .Ret<ffi::Buffer<ffi::F32>>()  // qvalues_epistemic_variance
                                  .Ret<ffi::Buffer<ffi::F32>>()  // root_value
                                  .Ret<ffi::Buffer<ffi::F32>>()  // root_ube
                                  .Ret<ffi::Buffer<ffi::U8>>()   // workspace
                                  EAZ_ENV_ATTRS()
                                  .Attr<int32_t>("num_simulations")
                                  .Attr<int32_t>("max_depth")
                                  .Attr<int32_t>("max_num_considered_actions")
                                  .Attr<float>("gumbel_scale")
                                  .Attr<float>("discount")
                                  .Attr<int32_t>("two_players_game")
                                  .Attr<int32_t>("exploration")
                                  .Attr<float>("value_scale")
                                  .Attr<float>("maxvisit_init")
                                  .Attr<int32_t>("rescale_values")
                                  .Attr<int32_t>("flags")
                                  .Attr<int32_t>("mlp_mode")
                                  .Attr<int32_t>("fused_root")
                                  .Attr<int32_t>("draw_gumbel")
                                  .Attr<int32_t>("noise_seed")
                                  .Attr<int32_t>("reuse_prepared")
                                  .Attr<int32_t>("hash_bits")
                                  .Attr<int32_t>("hash_io")
                                  .Attr<float>("max_u")
                                  .Attr<float>("novelty_scale"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(EazEvaluate, EvaluateImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()  // beta
                                  .Arg<ffi::AnyBuffer>()         // action_map
                                  .Arg<ffi::Buffer<ffi::U8>>()   // binary_set
                                  .Arg<ffi::Buffer<ffi::U8>>()   // workspace_in
                                  .RemainingArgs()               // initial state leaves, 24 parameter buffers
                                  .RemainingRets()               // final state leaves, returns, workspace
                                  EAZ_ENV_ATTRS()
                                  .Attr<int32_t>("num_simulations")
                                  .Attr<int32_t>("max_depth")
                                  .Attr<int32_t>("max_num_considered_actions")
                                  .Attr<float>("discount")
                                  .Attr<float>("value_scale")
                                  .Attr<float>("maxvisit_init")
                                  .Attr<int32_t>("rescale_values")
                                  .Attr<int32_t>("flags")
                                  .Attr<int32_t>("mlp_mode")
                                  .Attr<int32_t>("hash_bits")
                                  .Attr<int32_t>("hash_io")
                                  .Attr<float>("max_u")
                                  .Attr<float>("novelty_scale")
                                  .Attr<int32_t>("max_episode_length"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(EazSelfplay, SelfplayImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()  // beta
                                  .Arg<ffi::AnyBuffer>()         // action_map
                                  .Arg<ffi::Buffer<ffi::U8>>()   // binary_set
                                  .Arg<ffi::Buffer<ffi::F32>>()  // gumbel
                                  .Arg<ffi::Buffer<ffi::F32>>()  // sample_gumbel
                                  .Arg<ffi::Buffer<ffi::S32>>()  // task_ids
                                  .Arg<ffi::Buffer<ffi::U8>>()   // workspace_in
                                  .RemainingArgs()               // initial state leaves, 24 parameter buffers
                                  .RemainingRets()               // final state leaves, 9 stacked outputs, workspace
                                  EAZ_ENV_ATTRS()
                                  .Attr<int32_t>("num_simulations")
                                  .Attr<int32_t>("max_depth")
                                  .Attr<int32_t>("max_num_considered_actions")
                                  .Attr<float>("gumbel_scale")
                                  .Attr<float>("discount")
                                  .Attr<int32_t>("two_players_game")
                                  .Attr<int32_t>("exploration")
                                  .Attr<float>("value_scale")
                                  .Attr<float>("maxvisit_init")
                                  .Attr<int32_t>("rescale_values")
                                  .Attr<int32_t>("flags")
                                  .Attr<int32_t>("mlp_mode")
                                  .Attr<int32_t>("hash_bits")
                                  .Attr<int32_t>("hash_io")
                                  .Attr<float>("max_u")
                                  .Attr<float>("novelty_scale")
                                  .Attr<int32_t>("steps")
                                  .Attr<int32_t>("root_prior")
                                  .Attr<int32_t>("action_sampling")
                                  .Attr<float>("temperature")
                                  .Attr<int32_t>("noise_seed")
                                  .Attr<int32_t>("reuse_prepared"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(EazEnvStep, EnvStepImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::S32>>()  // action
                                  .Arg<ffi::Buffer<ffi::S32>>()  // task_ids
                                  .Arg<ffi::AnyBuffer>()         // action_map
                                  .RemainingArgs()
                                  .RemainingRets()
                                  EAZ_ENV_ATTRS()
                                  .Attr<int32_t>("auto_reset"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(EazEnvInit, EnvInitImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::S32>>()  // task_ids
                                  .Arg<ffi::AnyBuffer>()         // action_map
                                  .RemainingRets()
                                  EAZ_ENV_ATTRS()
                                  .Attr<int32_t>("batch"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(EazMlpForwardStates, MlpForwardStatesImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::AnyBuffer>()        // action_map
                                  .Arg<ffi::Buffer<ffi::U8>>()  // binary_set
                                  .RemainingArgs()
                                  .Ret<ffi::Buffer<ffi::F32>>()  // exploit_logits
                                  .Ret<ffi::Buffer<ffi::F32>>()  // explore_logits
                                  .Ret<ffi::Buffer<ffi::F32>>()  // value
                                  .Ret<ffi::Buffer<ffi::F32>>()  // ube
                                  .Ret<ffi::Buffer<ffi::F32>>()  // novelty
                                  .Ret<ffi::Buffer<ffi::U8>>()   // scratch
                                  EAZ_ENV_ATTRS()
                                  .Attr<int32_t>("hash_bits")
                                  .Attr<int32_t>("hash_io")
                                  .Attr<float>("max_u")
                                  .Attr<float>("novelty_scale"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(EazReanalyzeTargets, ReanalyzeTargetsImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::S32>>()  // action
                                  .Arg<ffi::Buffer<ffi::F32>>()  // qvalues
                                  .Arg<ffi::Buffer<ffi::F32>>()  // qvalues_epistemic_variance
                                  .Arg<ffi::Buffer<ffi::F32>>()  // visit_counts
                                  .Arg<ffi::Buffer<ffi::F32>>()  // value
                                  .Arg<ffi::Buffer<ffi::F32>>()  // value_epistemic_std
                                  .Arg<ffi::Buffer<ffi::F32>>()  // next_state_value
                                  .Arg<ffi::Buffer<ffi::F32>>()  // next_rewards
                                  .Arg<ffi::AnyBuffer>()         // next_terminated
                                  .Arg<ffi::AnyBuffer>()         // terminated
                                  .Arg<ffi::AnyBuffer>()         // invalid_actions
                                  .Ret<ffi::Buffer<ffi::F32>>()  // value_target
                                  .Ret<ffi::Buffer<ffi::F32>>()  // ube_target
                                  .Ret<ffi::Buffer<ffi::F32>>()  // exploration_policy_target
                                  .Attr<float>("discount")
                                  .Attr<float>("exploration_beta")
                                  .Attr<int32_t>("exploration_ube_target")
                                  .Attr<float>("temperature"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(EazHashUpdate, HashUpdateImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::F32>>()  // x
                                  .Arg<ffi::Buffer<ffi::U8>>()   // binary_set_in
                                  .Ret<ffi::Buffer<ffi::U8>>()   // binary_set
                                  .Attr<int32_t>("bits"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(EazReplayInit, ReplayInitImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Ret<ffi::Buffer<ffi::U8>>()   // ring_states
                                  .Ret<ffi::Buffer<ffi::F32>>()  // ring_rewards
                                  .Ret<ffi::Buffer<ffi::U8>>()   // tree
                                  .Attr<int32_t>("T")
                                  .Attr<int32_t>("B")
                                  .Attr<float>("priority_exponent")
                                  .Attr<int32_t>("seed"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(EazReplayAdd, ReplayAddImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::AnyBuffer>()         // action_map
                                  .Arg<ffi::Buffer<ffi::U8>>()   // ring_states_in
                                  .Arg<ffi::Buffer<ffi::F32>>()  // ring_rewards_in
                                  .Arg<ffi::Buffer<ffi::U8>>()   // tree_in
                                  .RemainingArgs()               // state leaves
                                  .Ret<ffi::Buffer<ffi::U8>>()   // ring_states
                                  .Ret<ffi::Buffer<ffi::F32>>()  // ring_rewards
                                  .Ret<ffi::Buffer<ffi::U8>>()   // tree
                                  EAZ_ENV_ATTRS());

XLA_FFI_DEFINE_HANDLER_SYMBOL(EazReplayAddSequence, ReplayAddSequenceImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::AnyBuffer>()         // action_map
                                  .Arg<ffi::Buffer<ffi::U8>>()   // ring_states_in
                                  .Arg<ffi::Buffer<ffi::F32>>()  // ring_rewards_in
                                  .Arg<ffi::Buffer<ffi::U8>>()   // tree_in
                                  .Arg<ffi::Buffer<ffi::U8>>()   // compact [T',B,S]
                                  .Arg<ffi::Buffer<ffi::F32>>()  // rewards [T',B]
                                  .Ret<ffi::Buffer<ffi::U8>>()   // ring_states
                                  .Ret<ffi::Buffer<ffi::F32>>()  // ring_rewards
                                  .Ret<ffi::Buffer<ffi::U8>>()   // tree
                                  EAZ_ENV_ATTRS());

XLA_FFI_DEFINE_HANDLER_SYMBOL(EazReplaySample, ReplaySampleImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::AnyBuffer>()         // action_map
                                  .Arg<ffi::Buffer<ffi::U8>>()   // ring_states
                                  .Arg<ffi::Buffer<ffi::F32>>()  // ring_rewards
                                  .Arg<ffi::Buffer<ffi::U8>>()   // tree
                                  .Arg<ffi::Buffer<ffi::U32>>()  // key
                                  .Ret<ffi::Buffer<ffi::S32>>()  // indices
                                  .Ret<ffi::Buffer<ffi::F32>>()  // probabilities
                                  .RemainingRets()               // first leaves, second leaves, scratch
                                  EAZ_ENV_ATTRS()
                                  .Attr<int32_t>("K"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(EazReplaySetPriorities, ReplaySetPrioritiesImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::S32>>()  // indices
                                  .Arg<ffi::Buffer<ffi::F32>>()  // priorities
                                  .Arg<ffi::Buffer<ffi::U8>>()   // tree_in
                                  .Ret<ffi::Buffer<ffi::U8>>()   // tree
                                  .Attr<int32_t>("T")
                                  .Attr<int32_t>("B"));

XLA_FFI_DEFINE_HANDLER_SYMBOL(EazReplayStatus, ReplayStatusImpl,
                              ffi::Ffi::Bind()
                                  .Ctx<ffi::PlatformStream<cudaStream_t>>()
                                  .Arg<ffi::Buffer<ffi::U8>>()   // tree
                                  .Ret<ffi::Buffer<ffi::S32>>());  // flags
