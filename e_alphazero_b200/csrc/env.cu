// env.cu -- pgx.Env.init / step / observe for DeepSea and Subleq on
// struct-of-arrays pgx.State buffers (the standalone env entry points of
// include/eaz_b200.h; the search uses the same device functions on compact states).
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

namespace eaz {

unsigned long long* g_timeline = nullptr;
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what) {
  set_error("%s: %s", what, cudaGetErrorString(e));
  return EAZ_ERR_CUDA;
}

int make_env_desc(const eaz_env* env, EnvDesc* d) {
  EAZ_CHECK_ARG(env != nullptr, "env is NULL");
  memset(d, 0, sizeof(*d));
  d->kind = env->kind;
  if (env->kind == EAZ_ENV_DEEPSEA) {
    EAZ_CHECK_ARG(env->size >= 1 && env->size <= 4095, "DeepSea size_of_grid %d out of range [1,4095]", env->size);
    d->size = env->size;
    d->action_map = env->action_map;
    d->obs_cols = env->size;
    d->obs_dim = env->size * env->size;
    d->num_actions = 2;
    d->compact_bytes = 4;
  } else if (env->kind == EAZ_ENV_SUBLEQ) {
    EAZ_CHECK_ARG(env->word_size >= 16 && env->word_size <= 256, "Subleq word_size %d violates 16 <= word_size <= 256 (subleq.py:606)",
                  env->word_size);
    EAZ_CHECK_ARG(env->reward_fn == EAZ_SUBLEQ_REWARD_SOLVED || env->reward_fn == EAZ_SUBLEQ_REWARD_LOWEST_BYTES, "unknown reward_fn %d",
                  env->reward_fn);
    d->ws = env->word_size;
    d->binary = env->binary_encoding != 0;
    d->reward_fn = env->reward_fn;
    d->obs_cols = d->binary ? binary_width(d->ws) : d->ws + 1;
    d->obs_dim = (d->ws + 32) * d->obs_cols;
    d->num_actions = d->ws;
    d->compact_bytes = EAZ_SQ_HDR + ((d->ws + 7) / 8) * 8;
  } else {
    set_error("unknown env kind %d", env->kind);
    return EAZ_ERR_INVALID_ARG;
  }
  return 0;
}

// ------------------------------------------------------------------ DeepSea
__global__ void deepsea_init_kernel(StateSoA s, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  s.step_count[b] = 0;
  s.col[b] = 0;
  s.rewards[b] = 0.0f;
  s.terminated[b] = 0;
  if (s.truncated) s.truncated[b] = 0;
}

__global__ void deepsea_step_kernel(EnvDesc env, StateSoA s, const int32_t* __restrict__ action, int auto_reset, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  deepsea_state_step(env, s, action, auto_reset, b);
}

// one-hot [N,N] observation, 16 bytes per thread
__global__ void deepsea_observe_kernel(EnvDesc env, StateSoA s, uint8_t* __restrict__ obs, int B) {
  const int D = env.obs_dim;
  const long long chunks_per_env = (D + 15) / 16;
  const long long total = chunks_per_env * B;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i / chunks_per_env), c = (int)(i % chunks_per_env);
    const int idx = deepsea_obs_index(ds_pack(s.step_count[b], s.col[b], 0, 0), env.size);
    uint8_t* o = obs + (size_t)b * D + (size_t)c * 16;
    const int lim = min(16, D - c * 16);
    for (int j = 0; j < lim; ++j) o[j] = (uint8_t)(c * 16 + j == idx);
  }
}

// ------------------------------------------------------------------ Subleq
// mode: 0 = init (task from task_ids), 1 = step, 2 = step with auto_reset
__global__ void __launch_bounds__(3 * EAZ_SQ_EPB) subleq_kernel(EnvDesc env, StateSoA s, const int32_t* __restrict__ action,
                                                                 const int32_t* __restrict__ task_ids, int mode, int B) {
  __shared__ SqShared sh;
  extern __shared__ __align__(16) uint8_t sq_dyn[];  // per-(env, test) memory images + cycle-detector snapshots
  __shared__ int kind[EAZ_SQ_EPB];
  subleq_block_step(env, s, action, task_ids, mode, B, sh, sq_dyn, kind);
}

// Subleq._observe (subleq.py:679-707): one thread per observation row.
__device__ __forceinline__ int sq_obs_word(const EnvDesc& env, const StateSoA& s, int b, int row) {
  const int ws = env.ws;
  if (row < ws) return s.memory[(size_t)b * ws + row];
  const int r = row - ws, part = r >> 3, i = r & 7;
  const int trow = sq_task_row(s.task[b]);
  if (part == 0) return sq_test_in(trow, 0, i, ws);       // example input
  if (part == 1) return s.input_after[(size_t)b * 8 + i]; // input after
  if (part == 2) return sq_test_out(trow, 0, i, ws);      // example output
  return s.output_after[(size_t)b * 8 + i];               // output after
}

__global__ void subleq_observe_kernel(EnvDesc env, StateSoA s, uint8_t* __restrict__ obs, int B) {
  const int rows = env.ws + 32, w = env.obs_cols, ws = env.ws;
  const long long total = (long long)rows * B;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i / rows), row = (int)(i % rows);
    const int v = sq_obs_word(env, s, b, row);
    uint8_t* o = obs + ((size_t)b * rows + row) * w;
    if (env.binary) {  // subleq.py:88-97
      const unsigned m = (unsigned)floormod(v, ws) & 0xffu;
      for (int bit = 0; bit < w; ++bit) o[bit] = bit < 8 ? (uint8_t)((m >> bit) & 1u) : 0;
      o[w - 1] = (uint8_t)(v == ws);
    } else {  // subleq.py:51-55
      const int hot = v == ws ? ws : floormod(v, ws);
      for (int c = 0; c < w; ++c) o[c] = (uint8_t)(c == hot);
    }
  }
}

}  // namespace eaz

using namespace eaz;

namespace eaz {
// one pack_trajectory record per env
__global__ void trajectory_pack_kernel(EnvDesc env, StateSoA s, const int32_t* __restrict__ action, int4* __restrict__ out, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  out[b] = pack_trajectory(env, s, action, b);
}
}  // namespace eaz

extern "C" {

int eaz_abi_version(void) { return EAZ_ABI_VERSION; }
const char* eaz_last_error(void) { return eaz::g_err; }

int32_t eaz_env_num_actions(const eaz_env* env) {
  EnvDesc d;
  return make_env_desc(env, &d) ? -1 : d.num_actions;
}
int32_t eaz_env_obs_dim(const eaz_env* env) {
  EnvDesc d;
  return make_env_desc(env, &d) ? -1 : d.obs_dim;
}
int32_t eaz_env_obs_cols(const eaz_env* env) {
  EnvDesc d;
  return make_env_desc(env, &d) ? -1 : d.obs_cols;
}
int32_t eaz_env_hash_dim(const eaz_env* env, int32_t hash_io) {
  EnvDesc d;
  if (make_env_desc(env, &d)) return -1;
  return (d.kind == EAZ_ENV_SUBLEQ && hash_io) ? 32 * d.obs_cols : d.obs_dim;  // fully_connected.py:85-89
}
int32_t eaz_env_compact_bytes(const eaz_env* env) {
  EnvDesc d;
  return make_env_desc(env, &d) ? -1 : d.compact_bytes;
}

int eaz_subleq_test_cases(int32_t task, int32_t ws, int32_t* inputs, int32_t* outputs) {
  EAZ_CHECK_ARG(ws >= 16 && ws <= 256, "word_size %d violates 16 <= word_size <= 256", ws);
  EAZ_CHECK_ARG(inputs && outputs, "NULL output");
  SubleqVec hin[6][3], hout[6][3];
  cudaError_t e = cudaMemcpyFromSymbol(hin, c_sq_in, sizeof(hin));
  if (e == cudaSuccess) e = cudaMemcpyFromSymbol(hout, c_sq_out, sizeof(hout));
  if (e != cudaSuccess) return cuda_fail(e, "eaz_subleq_test_cases");
  const int t = task - 1 < 0 ? 0 : (task - 1 > 5 ? 5 : task - 1);
  for (int k = 0; k < 3; ++k)
    for (int i = 0; i < 8; ++i) {
      inputs[k * 8 + i] = i < hin[t][k].len ? floormod(hin[t][k].v[i], ws) : ws;
      outputs[k * 8 + i] = i < hout[t][k].len ? floormod(hout[t][k].v[i], ws) : ws;
    }
  return 0;
}

static int check_state(const EnvDesc& d, const eaz_state* s) {
  EAZ_CHECK_ARG(s && s->step_count && s->rewards && s->terminated, "state: step_count/rewards/terminated must be non-NULL");
  if (d.kind == EAZ_ENV_DEEPSEA) EAZ_CHECK_ARG(s->col != nullptr, "DeepSea state needs col");
  else EAZ_CHECK_ARG(s->memory && s->task && s->solved && s->input_after && s->output_after, "Subleq state needs memory/task/solved/input_after/output_after");
  return 0;
}

int eaz_env_observe(const eaz_env* env, const eaz_state* state, uint8_t* observation, int32_t B, void* stream) {
  EnvDesc d;
  if (int rc = make_env_desc(env, &d)) return rc;
  if (int rc = check_state(d, state)) return rc;
  EAZ_CHECK_ARG(observation && B >= 0, "observe: bad arguments");
  if (B == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const StateSoA s = soa_of(state);
  if (d.kind == EAZ_ENV_DEEPSEA) {
    const long long total = (long long)((d.obs_dim + 15) / 16) * B;
    const int grid = (int)min((long long)148 * 16, (total + 255) / 256);
    deepsea_observe_kernel<<<grid, 256, 0, st>>>(d, s, observation, B);
  } else {
    const long long total = (long long)(d.ws + 32) * B;
    const int grid = (int)min((long long)148 * 16, (total + 255) / 256);
    subleq_observe_kernel<<<grid, 256, 0, st>>>(d, s, observation, B);
  }
  EAZ_CHECK_LAUNCH("eaz_env_observe");
  return 0;
}

int eaz_env_init(const eaz_env* env, const int32_t* task_ids, eaz_state* out, int32_t B, void* stream) {
  EnvDesc d;
  if (int rc = make_env_desc(env, &d)) return rc;
  if (int rc = check_state(d, out)) return rc;
  EAZ_CHECK_ARG(B >= 0, "negative batch");
  if (B == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const StateSoA s = soa_of(out);
  if (d.kind == EAZ_ENV_DEEPSEA) deepsea_init_kernel<<<ceil_div(B, 256), 256, 0, st>>>(s, B);
  else {
    size_t dyn = 0;
    if (cudaError_t e = sq_prepare_launch(subleq_kernel, d.ws, &dyn); e != cudaSuccess) return cuda_fail(e, "subleq_kernel attribute");
    subleq_kernel<<<ceil_div(B, EAZ_SQ_EPB), 3 * EAZ_SQ_EPB, dyn, st>>>(d, s, nullptr, task_ids, 0, B);
  }
  EAZ_CHECK_LAUNCH("eaz_env_init");
  if (out->observation) return eaz_env_observe(env, out, out->observation, B, stream);
  return 0;
}

int eaz_env_step(const eaz_env* env, eaz_state* state, const int32_t* action, int32_t auto_reset, const int32_t* task_ids,
                 int32_t B, void* stream) {
  EnvDesc d;
  if (int rc = make_env_desc(env, &d)) return rc;
  if (int rc = check_state(d, state)) return rc;
  EAZ_CHECK_ARG(action != nullptr && B >= 0, "step: action is NULL or negative batch");
  if (B == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const StateSoA s = soa_of(state);
  if (d.kind == EAZ_ENV_DEEPSEA) deepsea_step_kernel<<<ceil_div(B, 256), 256, 0, st>>>(d, s, action, auto_reset, B);
  else {
    size_t dyn = 0;
    if (cudaError_t e = sq_prepare_launch(subleq_kernel, d.ws, &dyn); e != cudaSuccess) return cuda_fail(e, "subleq_kernel attribute");
    subleq_kernel<<<ceil_div(B, EAZ_SQ_EPB), 3 * EAZ_SQ_EPB, dyn, st>>>(d, s, action, task_ids, auto_reset ? 2 : 1, B);
  }
  EAZ_CHECK_LAUNCH("eaz_env_step");
  if (state->observation) return eaz_env_observe(env, state, state->observation, B, stream);
  return 0;
}

int eaz_trajectory_pack(const eaz_env* env, const eaz_state* state, const int32_t* action, int32_t* out, int32_t B, void* stream) {
  EnvDesc d;
  if (int rc = make_env_desc(env, &d)) return rc;
  if (int rc = check_state(d, state)) return rc;
  EAZ_CHECK_ARG(action != nullptr && out != nullptr && B >= 0, "eaz_trajectory_pack: NULL action / out or negative batch");
  if (B == 0) return 0;
  trajectory_pack_kernel<<<ceil_div(B, 256), 256, 0, (cudaStream_t)stream>>>(d, soa_of(state), action, reinterpret_cast<int4*>(out), B);
  EAZ_CHECK_LAUNCH("trajectory_pack_kernel");
  return 0;
}

}  // extern "C"

// Debug hook (not in the public header): device buffer of >= 8 + 4*records u64; buf[0] must be zeroed by the caller.
extern "C" void eaz_debug_set_timeline(unsigned long long* device_buffer) { eaz::g_timeline = device_buffer; }
