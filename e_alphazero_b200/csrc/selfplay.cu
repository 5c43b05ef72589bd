// selfplay.cu -- the self-play scan of selfplay.py:78-149 as one device program.
//
// The reference's selfplay() is lax.scan(step_fn, starting_states, key_seq) over selfplay_steps steps (selfplay.py:148): step_fn
// (:86-143) = forward.apply on the root states + the Gumbel search + its summary + the auto-reset env step, and the scan stacks every
// step's SelfplayOutput.  Here the scan is a CUDA graph with one WHILE conditional node.  Its body is the fused-root search (the
// launches eaz_search_gumbel enqueues, captured) and selfplay_step_kernel, which steps the envs with auto-reset, writes row t of every
// requested stacked output, stages the next step's pre-drawn noise and -- in its last CTA -- advances t and writes t < T into the loop's
// handle.  The host launches the graph once per scan and never waits inside it.
//
// Workspace: [SelfplayWords | 256 B][gumbel B*A f32][sample_gumbel B*A f32][one step's search outputs: action B i32, value, value_std,
// root_value, root_ube B f32 each, qvalues_epistemic_variance B*A f32][search workspace], each 256-byte aligned.
#include "loop_graph.cuh"
#include "mlp.cuh"

namespace eaz {

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct SelfplayWords {
  int32_t t;        // steps done so far in this call
  uint32_t ticket;  // CTAs of the step kernel done with the current step
};

struct SelfplayLayout {
  size_t gumbel, sample, action, value, value_std, root_value, root_ube, qvar, search, search_bytes, total;
};

static bool selfplay_layout(const eaz_search_config* cfg, const eaz_env* env, SelfplayLayout* L) {
  EnvDesc d;
  if (!cfg || make_env_desc(env, &d) || cfg->batch < 1) return false;
  eaz_search_config c = *cfg;
  c.flags &= ~EAZ_FLAG_REUSE_PREPARED;
  const size_t s = eaz_search_workspace_bytes(&c, env);
  if (s == 0) return false;
  const size_t BA = align256((size_t)cfg->batch * d.num_actions * sizeof(float)), B4 = align256((size_t)cfg->batch * 4);
  L->gumbel = 256;
  L->sample = L->gumbel + BA;
  L->action = L->sample + BA;
  L->value = L->action + B4;
  L->value_std = L->value + B4;
  L->root_value = L->value_std + B4;
  L->root_ube = L->root_value + B4;
  L->qvar = L->root_ube + B4;
  L->search = L->qvar + BA;
  L->search_bytes = s;
  L->total = L->search + s;
  return true;
}

// What selfplay_step_kernel reads and writes besides the states.
struct SelfplayStep {
  const int32_t* action;  // this step's search outputs [B] / [B,A] (workspace)
  const float *value, *value_std, *root_value, *root_ube, *qvar;
  const int32_t* task_ids;               // [T,B], NULL for DeepSea
  const float *gumbel_src, *sample_src;  // [T,B,A] or NULL (drawn in the search): row t+1 is staged into gumbel_dst / sample_dst [B,A]
  float *gumbel_dst, *sample_dst;
  eaz_selfplay_outputs out;
  SelfplayWords* words;
  int T, B, A;
};

// Closes step t (t = words->t): the auto-reset env step (selfplay.py:26-75,135) on the played actions, row t of every requested output,
// the staging of row t+1 of the pre-drawn noise, and in the CTA that finishes last t += 1 and the loop condition t < T.
template <int kKind>
__global__ void selfplay_step_kernel(EnvDesc env, StateSoA s, SelfplayStep a, cudaGraphConditionalHandle loop) {
  // the same t in every CTA: only the last CTA advances it, after every CTA has read it and taken its ticket
  const int t = *(volatile int32_t*)&a.words->t;
  const size_t row = (size_t)t * a.B;
  int b, owner, per_cta;
  if constexpr (kKind == EAZ_ENV_DEEPSEA) {
    per_cta = blockDim.x;
    b = blockIdx.x * blockDim.x + threadIdx.x;
    owner = b < a.B;
    if (owner) deepsea_state_step(env, s, a.action, 1, b);
  } else {
    __shared__ SqShared sh;
    __shared__ int kind[EAZ_SQ_EPB];
    extern __shared__ __align__(16) uint8_t sq_dyn[];
    per_cta = EAZ_SQ_EPB;
    b = blockIdx.x * EAZ_SQ_EPB + threadIdx.x / 3;
    owner = b < a.B && threadIdx.x % 3 == 0;
    subleq_block_step(env, s, a.action, a.task_ids + row, 2, a.B, sh, sq_dyn, kind);
  }
  const eaz_selfplay_outputs& o = a.out;
  if (owner) {  // (this thread wrote env b's leaves)
    const size_t r = row + b;
    const int act = a.action[b];
    if (o.action) o.action[r] = act;
    if (o.root_value) o.root_value[r] = a.value[b];
    if (o.root_epistemic_std) o.root_epistemic_std[r] = a.value_std[b];
    if (o.value_prediction) o.value_prediction[r] = a.root_value[b];
    if (o.ube_prediction) o.ube_prediction[r] = a.root_ube[b];
    if (o.trajectory) reinterpret_cast<int4*>(o.trajectory)[r] = pack_trajectory(env, s, a.action, b);
    if (o.states) pack_state(env, s, b, o.states + row * env.compact_bytes);
    if (o.rewards) o.rewards[r] = s.rewards[b];
  }
  // the [B,A] rows of this CTA's envs, all threads: q-value variances out, the next step's noise in (the search that read the
  // staged noise of step t has finished: this kernel is not a programmatic dependent of it)
  const size_t BA = (size_t)a.B * a.A, lo = (size_t)blockIdx.x * per_cta * a.A, hi = min(BA, lo + (size_t)per_cta * a.A);
  const bool stage = t + 1 < a.T;
  for (size_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
    if (o.q_values_epistemic_variance) o.q_values_epistemic_variance[(size_t)t * BA + i] = a.qvar[i];
    if (stage && a.gumbel_src) a.gumbel_dst[i] = a.gumbel_src[(size_t)(t + 1) * BA + i];
    if (stage && a.sample_src) a.sample_dst[i] = a.sample_src[(size_t)(t + 1) * BA + i];
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  __threadfence();
  if (atomicAdd(&a.words->ticket, 1u) != gridDim.x - 1) return;
  __threadfence();  // last CTA: every other CTA has read t
  a.words->t = t + 1;
  a.words->ticket = 0;  // re-armed for the next step
  cudaGraphSetConditional(loop, (unsigned)stage);
}

static int launch_selfplay_step(const EnvDesc& env, const eaz_state* states, const SelfplayStep& a, cudaGraphConditionalHandle loop,
                                cudaStream_t st) {
  const StateSoA s = soa_of(states);
  if (env.kind == EAZ_ENV_DEEPSEA) {
    selfplay_step_kernel<EAZ_ENV_DEEPSEA><<<ceil_div(a.B, 256), 256, 0, st>>>(env, s, a, loop);
  } else {
    size_t dyn = 0;
    if (cudaError_t e = sq_prepare_launch(selfplay_step_kernel<EAZ_ENV_SUBLEQ>, env.ws, &dyn); e != cudaSuccess)
      return cuda_fail(e, "selfplay_step_kernel attribute");
    selfplay_step_kernel<EAZ_ENV_SUBLEQ><<<ceil_div(a.B, EAZ_SQ_EPB), 3 * EAZ_SQ_EPB, dyn, st>>>(env, s, a, loop);
  }
  EAZ_CHECK_LAUNCH("selfplay_step_kernel");
  return 0;
}

// what the scan's graph bakes in (the captured launches hold these by value)
struct SelfplayRec {
  eaz_search_config cfg;
  eaz_env env;
  eaz_fc_params net;
  eaz_state states;
  const float* beta;
  const uint8_t* invalid;
  const int32_t* task_ids;
  const float *gumbel, *sample;
  eaz_selfplay_outputs out;
  int32_t T;
  size_t bytes;
  bool same(const SelfplayRec& o) const {
    return !memcmp(&cfg, &o.cfg, sizeof(cfg)) && same_env(env, o.env) && same_net(net, o.net) && !memcmp(&states, &o.states, sizeof(eaz_state)) &&
           beta == o.beta && invalid == o.invalid && task_ids == o.task_ids && gumbel == o.gumbel && sample == o.sample &&
           !memcmp(&out, &o.out, sizeof(out)) && T == o.T && bytes == o.bytes;
  }
};
static LoopGraphs<SelfplayRec> g_selfplay_graphs;

}  // namespace eaz

using namespace eaz;

extern "C" {

size_t eaz_selfplay_workspace_bytes(const eaz_search_config* cfg, const eaz_env* env) {
  SelfplayLayout L;
  return selfplay_layout(cfg, env, &L) ? L.total : 0;
}

int eaz_selfplay(const eaz_search_config* cfg, const eaz_search_inputs* in, const eaz_fc_params* net, eaz_state* states, int32_t T,
                 const int32_t* task_ids, eaz_selfplay_outputs* out, void* workspace, size_t workspace_bytes, void* stream) {
  EAZ_CHECK_ARG(cfg && in && net && states && out, "eaz_selfplay: NULL config / inputs / net / states / outputs");
  EAZ_CHECK_ARG(!in->prior_logits && !in->value && !in->value_epistemic_variance,
                "eaz_selfplay: the root is evaluated inside the loop (prior_logits / value / value_epistemic_variance must be NULL)");
  EAZ_CHECK_ARG(!(cfg->flags & EAZ_FLAG_PUCT), "eaz_selfplay: self-play searches with the Gumbel policy (selfplay.py:107), not EAZ_FLAG_PUCT");
  EAZ_CHECK_ARG(in->beta != nullptr, "eaz_selfplay: beta must be non-NULL");
  EAZ_CHECK_ARG(T >= 0, "eaz_selfplay: negative number of steps T = %d", T);
  EnvDesc env;
  if (int rc = make_env_desc(in->env, &env)) return rc;
  EAZ_CHECK_ARG(cfg->batch >= 1, "batch must be >= 1");
  EAZ_CHECK_ARG(states->step_count && states->rewards && states->terminated, "eaz_selfplay: state step_count / rewards / terminated must be non-NULL");
  if (env.kind == EAZ_ENV_DEEPSEA) EAZ_CHECK_ARG(states->col != nullptr, "eaz_selfplay: DeepSea state needs col");
  else EAZ_CHECK_ARG(states->memory && states->task && states->solved && states->input_after && states->output_after,
                     "eaz_selfplay: Subleq state needs memory / task / solved / input_after / output_after");
  EAZ_CHECK_ARG(!states->observation, "eaz_selfplay: states->observation must be NULL (the loop does not materialise observations)");
  EAZ_CHECK_ARG(env.kind != EAZ_ENV_SUBLEQ || task_ids, "eaz_selfplay: Subleq resets need task_ids [T,B] (subleq.py:624)");
  // the largest stacked output, T*B rows of max(4A, S, 16) bytes, must have a byte count that size_t holds
  const size_t row_bytes = std::max(std::max((size_t)env.num_actions * sizeof(float), (size_t)env.compact_bytes), (size_t)16);
  if ((size_t)T * (size_t)cfg->batch > SIZE_MAX / row_bytes) {
    set_error("eaz_selfplay: T * B * %zu bytes of stacked output (T = %d, B = %d) overflows", row_bytes, T, cfg->batch);
    return EAZ_ERR_INVALID_ARG;
  }
  SelfplayLayout L;
  if (!selfplay_layout(cfg, in->env, &L)) {
    set_error("eaz_selfplay: the search configuration was rejected (batch %d, num_simulations %d)", cfg->batch, cfg->num_simulations);
    return EAZ_ERR_INVALID_ARG;
  }
  if (!workspace || workspace_bytes < L.total || ((uintptr_t)workspace & 255)) {
    set_error("selfplay workspace must be >= %zu bytes and 256-byte aligned (got %zu)", L.total, workspace_bytes);
    return EAZ_ERR_WORKSPACE;
  }
  if (T == 0) return 0;  // lax.scan of length 0: the carry is unchanged and nothing is stacked

  const int B = cfg->batch, A = env.num_actions;
  const bool sampling = cfg->action_sampling != EAZ_ACTION_SEARCH;
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* ws = (uint8_t*)workspace;
  eaz_search_inputs li{};
  li.beta = in->beta;
  li.embedding = states;
  li.invalid_actions = in->invalid_actions;
  li.gumbel = in->gumbel ? reinterpret_cast<const float*>(ws + L.gumbel) : nullptr;
  li.sample_gumbel = sampling && in->sample_gumbel ? reinterpret_cast<const float*>(ws + L.sample) : nullptr;
  li.env = in->env;
  li.net = net;
  eaz_search_outputs lo{};
  lo.action = reinterpret_cast<int32_t*>(ws + L.action);
  lo.value = reinterpret_cast<float*>(ws + L.value);
  lo.value_epistemic_std = reinterpret_cast<float*>(ws + L.value_std);
  lo.qvalues_epistemic_variance = reinterpret_cast<float*>(ws + L.qvar);
  lo.root_value = reinterpret_cast<float*>(ws + L.root_value);
  lo.root_ube = reinterpret_cast<float*>(ws + L.root_ube);
  void* search_ws = ws + L.search;
  SelfplayStep a{lo.action, lo.value, lo.value_epistemic_std, lo.root_value, lo.root_ube, lo.qvalues_epistemic_variance,
                 env.kind == EAZ_ENV_SUBLEQ ? task_ids : nullptr, in->gumbel, li.sample_gumbel ? in->sample_gumbel : nullptr,
                 reinterpret_cast<float*>(ws + L.gumbel), reinterpret_cast<float*>(ws + L.sample), *out,
                 reinterpret_cast<SelfplayWords*>(ws), T, B, A};

  std::lock_guard<std::mutex> lock(g_selfplay_graphs.mu);
  // the table preparation, once, outside the loop (the model is constant within one scan, selfplay.py:148); it draws no noise
  if (!(cfg->flags & EAZ_FLAG_REUSE_PREPARED)) {
    eaz_search_config prep = *cfg;
    prep.flags |= kFlagPrepareOnly;
    if (int rc = eaz_search_gumbel(&prep, &li, &lo, search_ws, L.search_bytes, stream)) return rc;
  }
  eaz_search_config body = *cfg;
  body.flags |= EAZ_FLAG_REUSE_PREPARED;
  const SelfplayRec rec{body, *in->env, *net, *states, in->beta, in->invalid_actions, a.task_ids, a.gumbel_src, a.sample_src, *out, T,
                        workspace_bytes};
  cudaGraphExec_t exec = nullptr;
  if (int rc = g_selfplay_graphs.build("selfplay", workspace, rec, &exec, [&](cudaStream_t cap, cudaGraphConditionalHandle handle) {
        int rc = eaz_search_gumbel(&body, &li, &lo, search_ws, L.search_bytes, cap);
        if (rc == 0) rc = launch_selfplay_step(env, states, a, handle, cap);
        return rc;
      }))
    return rc;
  // the loop words start at t = 0; row 0 of the pre-drawn noise goes into the staged slots (the step kernel stages the later rows)
  if (cudaError_t e = cudaMemsetAsync(ws, 0, sizeof(SelfplayWords), st); e != cudaSuccess) return cuda_fail(e, "selfplay memset");
  const size_t ba = (size_t)B * A * sizeof(float);
  if (a.gumbel_src)
    if (cudaError_t e = cudaMemcpyAsync(a.gumbel_dst, a.gumbel_src, ba, cudaMemcpyDeviceToDevice, st); e != cudaSuccess) return cuda_fail(e, "selfplay noise copy");
  if (a.sample_src)
    if (cudaError_t e = cudaMemcpyAsync(a.sample_dst, a.sample_src, ba, cudaMemcpyDeviceToDevice, st); e != cudaSuccess) return cuda_fail(e, "selfplay noise copy");
  if (cudaError_t e = cudaGraphLaunch(exec, st); e != cudaSuccess) return cuda_fail(e, "selfplay graph launch");
  return 0;
}

}  // extern "C"
