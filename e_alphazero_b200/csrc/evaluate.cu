// evaluate.cu -- the evaluation loop of evaluate.py:13-57 as one device program.
//
// The reference runs its episodes in a lax.while_loop: cond_fn (evaluate.py:18-20) = any env not terminated and counter <=
// max_episode_length; body = forward.apply + the greedy search (gumbel_scale = 0) + env.step + the reward sum.  Here the loop is a CUDA
// graph with one WHILE conditional node.  Its body is the fused-root search (the launches eaz_search_gumbel enqueues, captured) and
// eval_step_kernel, which steps the envs, adds the rewards, counts the envs still live and -- in its last CTA -- writes the loop
// condition with cudaGraphSetConditional.  The host launches the graph once per evaluation and never waits inside it.
//
// Workspace: [eaz_evaluate_counters | 256 B][zero Gumbel noise B*A f32][played actions B i32][search workspace], each 256-byte aligned.
#include "loop_graph.cuh"
#include "mlp.cuh"

namespace eaz {

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct EvalLayout {
  size_t gumbel, action, search, search_bytes, total;
};

static bool eval_layout(const eaz_search_config* cfg, const eaz_env* env, EvalLayout* L) {
  EnvDesc d;
  if (!cfg || make_env_desc(env, &d) || cfg->batch < 1) return false;
  eaz_search_config c = *cfg;
  c.flags &= ~EAZ_FLAG_REUSE_PREPARED;
  const size_t s = eaz_search_workspace_bytes(&c, env);
  if (s == 0) return false;
  L->gumbel = 256;
  L->action = L->gumbel + align256((size_t)cfg->batch * d.num_actions * sizeof(float));
  L->search = L->action + align256((size_t)cfg->batch * sizeof(int32_t));
  L->search_bytes = s;
  L->total = L->search + s;
  return true;
}

// One move's end: pgx.Env.step (no auto-reset) on the search's actions, returns += rewards[:, 0], the count of live envs and, in the
// CTA that finishes last, the loop condition.  Outside a graph (in_graph = 0) the handle is not touched; the decision is still written
// to ctr->cont.
template <int kKind>
__global__ void eval_step_kernel(EnvDesc env, StateSoA s, const int32_t* __restrict__ action, float* __restrict__ returns,
                                 eaz_evaluate_counters* ctr, int max_episode_length, int B, cudaGraphConditionalHandle loop, int in_graph) {
  int b, owner;
  if constexpr (kKind == EAZ_ENV_DEEPSEA) {
    b = blockIdx.x * blockDim.x + threadIdx.x;
    owner = b < B;
    if (owner) deepsea_state_step(env, s, action, 0, b);
  } else {
    __shared__ SqShared sh;
    __shared__ int kind[EAZ_SQ_EPB];
    extern __shared__ __align__(16) uint8_t sq_dyn[];
    b = blockIdx.x * EAZ_SQ_EPB + threadIdx.x / 3;
    owner = b < B && threadIdx.x % 3 == 0;
    subleq_block_step(env, s, action, nullptr, 1, B, sh, sq_dyn, kind);
  }
  int live = 0;
  if (owner) {  // (this thread wrote env b's leaves)
    returns[b] = __fadd_rn(returns[b], s.rewards[b]);  // evaluate.py:48-50, one add per move
    live = s.terminated[b] == 0;
  }
  const int n = __syncthreads_count(live);
  if (threadIdx.x != 0) return;
  if (n) atomicAdd(&ctr->live, n);
  __threadfence();
  if (atomicAdd(&ctr->ticket, 1u) != gridDim.x - 1) return;
  __threadfence();  // last CTA: every other CTA's count is in
  const int moves = ctr->moves + 1;
  const int cont = atomicAdd(&ctr->live, 0) > 0 && moves <= max_episode_length;  // cond_fn, evaluate.py:18-20
  ctr->moves = moves;
  ctr->cont = cont;
  ctr->live = 0;  // re-armed for the next move
  ctr->ticket = 0;
  if (in_graph) cudaGraphSetConditional(loop, (unsigned)cont);
}

static int launch_eval_step(const EnvDesc& env, const eaz_state* states, const int32_t* action, float* returns, eaz_evaluate_counters* ctr,
                            int max_episode_length, int B, cudaGraphConditionalHandle loop, int in_graph, cudaStream_t st) {
  const StateSoA s = soa_of(states);
  if (env.kind == EAZ_ENV_DEEPSEA) {
    eval_step_kernel<EAZ_ENV_DEEPSEA><<<ceil_div(B, 256), 256, 0, st>>>(env, s, action, returns, ctr, max_episode_length, B, loop, in_graph);
  } else {
    size_t dyn = 0;
    if (cudaError_t e = sq_prepare_launch(eval_step_kernel<EAZ_ENV_SUBLEQ>, env.ws, &dyn); e != cudaSuccess)
      return cuda_fail(e, "eval_step_kernel attribute");
    eval_step_kernel<EAZ_ENV_SUBLEQ><<<ceil_div(B, EAZ_SQ_EPB), 3 * EAZ_SQ_EPB, dyn, st>>>(env, s, action, returns, ctr, max_episode_length, B, loop,
                                                                                          in_graph);
  }
  EAZ_CHECK_LAUNCH("eval_step_kernel");
  return 0;
}

// what the loop's graph bakes in (the captured launches hold these by value)
struct EvalRec {
  eaz_search_config cfg;
  eaz_env env;
  eaz_fc_params net;
  eaz_state states;
  const float* beta;
  const uint8_t* invalid;
  float* returns;
  int32_t max_episode_length;
  size_t bytes;
  bool same(const EvalRec& o) const {
    return !memcmp(&cfg, &o.cfg, sizeof(cfg)) && same_env(env, o.env) && same_net(net, o.net) && !memcmp(&states, &o.states, sizeof(eaz_state)) &&
           beta == o.beta && invalid == o.invalid && returns == o.returns && max_episode_length == o.max_episode_length && bytes == o.bytes;
  }
};
static LoopGraphs<EvalRec> g_eval_graphs;

}  // namespace eaz

using namespace eaz;

extern "C" {

size_t eaz_evaluate_workspace_bytes(const eaz_search_config* cfg, const eaz_env* env) {
  EvalLayout L;
  return eval_layout(cfg, env, &L) ? L.total : 0;
}

int eaz_evaluate(const eaz_search_config* cfg, const eaz_search_inputs* in, const eaz_fc_params* net, eaz_state* states, float* returns,
                 int32_t max_episode_length, void* workspace, size_t workspace_bytes, void* stream) {
  EAZ_CHECK_ARG(cfg && in && net && states && returns, "eaz_evaluate: NULL config / inputs / net / states / returns");
  EAZ_CHECK_ARG(!in->prior_logits && !in->value && !in->value_epistemic_variance,
                "eaz_evaluate: the root is evaluated inside the loop (prior_logits / value / value_epistemic_variance must be NULL)");
  EAZ_CHECK_ARG(cfg->gumbel_scale == 0.0f, "eaz_evaluate: greedy episodes need gumbel_scale = 0 (evaluate.py:44), got %g", (double)cfg->gumbel_scale);
  EAZ_CHECK_ARG(cfg->action_sampling == EAZ_ACTION_SEARCH, "eaz_evaluate: action_sampling must be EAZ_ACTION_SEARCH");
  EAZ_CHECK_ARG(in->beta != nullptr, "eaz_evaluate: beta must be non-NULL");
  EnvDesc env;
  if (int rc = make_env_desc(in->env, &env)) return rc;
  EAZ_CHECK_ARG(cfg->batch >= 1, "batch must be >= 1");
  EAZ_CHECK_ARG(states->step_count && states->rewards && states->terminated, "eaz_evaluate: state step_count / rewards / terminated must be non-NULL");
  if (env.kind == EAZ_ENV_DEEPSEA) EAZ_CHECK_ARG(states->col != nullptr, "eaz_evaluate: DeepSea state needs col");
  else EAZ_CHECK_ARG(states->memory && states->task && states->solved && states->input_after && states->output_after,
                     "eaz_evaluate: Subleq state needs memory / task / solved / input_after / output_after");
  EvalLayout L;
  if (!eval_layout(cfg, in->env, &L)) {
    set_error("eaz_evaluate: the search configuration was rejected (batch %d, num_simulations %d)", cfg->batch, cfg->num_simulations);
    return EAZ_ERR_INVALID_ARG;
  }
  if (!workspace || workspace_bytes < L.total || ((uintptr_t)workspace & 255)) {
    set_error("evaluate workspace must be >= %zu bytes and 256-byte aligned (got %zu)", L.total, workspace_bytes);
    return EAZ_ERR_WORKSPACE;
  }
  const int B = cfg->batch;
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)workspace;
  auto* ctr = reinterpret_cast<eaz_evaluate_counters*>(ws);
  // counters and zero noise; returns start at 0 (evaluate.py:41)
  if (cudaError_t e = cudaMemsetAsync(ws, 0, L.action, st); e != cudaSuccess) return cuda_fail(e, "evaluate memset");
  if (cudaError_t e = cudaMemsetAsync(returns, 0, (size_t)B * sizeof(float), st); e != cudaSuccess) return cuda_fail(e, "evaluate memset");
  if (max_episode_length < 0) return 0;  // cond_fn is false before the first move

  eaz_search_inputs li{};
  li.beta = in->beta;
  li.embedding = states;
  li.invalid_actions = in->invalid_actions;
  li.gumbel = reinterpret_cast<const float*>(ws + L.gumbel);
  li.env = in->env;
  li.net = net;
  eaz_search_outputs lo{};
  lo.action = reinterpret_cast<int32_t*>(ws + L.action);
  void* search_ws = ws + L.search;

  std::lock_guard<std::mutex> lock(g_eval_graphs.mu);
  // the first move's table preparation, once, outside the loop (the reference's model is constant over the episodes)
  eaz_search_config prep = *cfg;
  prep.flags = (prep.flags & ~EAZ_FLAG_REUSE_PREPARED) | kFlagPrepareOnly;
  if (int rc = eaz_search_gumbel(&prep, &li, &lo, search_ws, L.search_bytes, stream)) return rc;

  eaz_search_config body = *cfg;
  body.flags |= EAZ_FLAG_REUSE_PREPARED;
  const EvalRec rec{body, *in->env, *net, *states, in->beta, in->invalid_actions, returns, max_episode_length, workspace_bytes};
  return g_eval_graphs.launch("evaluate", workspace, rec, st, [&](cudaStream_t cap, cudaGraphConditionalHandle handle) {
    int rc = eaz_search_gumbel(&body, &li, &lo, search_ws, L.search_bytes, cap);
    if (rc == 0) rc = launch_eval_step(env, states, lo.action, returns, ctr, max_episode_length, B, handle, 1, cap);
    return rc;
  });
}

// Test hook (not in the public header): one eval_step_kernel launch outside a graph -- env step on `action`, returns += rewards[:,0],
// counters advanced and the decision written to counters->cont.
int eaz_debug_eval_step(const eaz_env* env_in, eaz_state* states, const int32_t* action, float* returns, eaz_evaluate_counters* counters,
                        int32_t max_episode_length, int32_t B, void* stream) {
  EnvDesc env;
  if (int rc = make_env_desc(env_in, &env)) return rc;
  EAZ_CHECK_ARG(states && action && returns && counters && B >= 1, "eaz_debug_eval_step: bad arguments");
  return launch_eval_step(env, states, action, returns, counters, max_episode_length, B, 0, 0, (cudaStream_t)stream);
}

}  // extern "C"
