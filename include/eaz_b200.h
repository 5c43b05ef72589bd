/*
 * eaz_b200.h -- C ABI of libeaz_b200.so, the B200 (sm_100a) implementation of
 * the batched self-play / reanalyze search step of emcts/e-alphazero.
 *
 * The reference has no FFI of its own: the hot path is a Python call into two
 * third-party JAX packages (emctx, pgx) plus three in-tree modules.  Each entry
 * point below names the reference interface it replaces (file:line under
 * /root/reference/src unless stated) -- these are what a JAX FFI custom-call
 * binding registers (INTEGRATION.md shows the stub).
 *
 * Conventions
 *   - plain `extern "C"`, POD structs, raw DEVICE pointers, explicit stream
 *     (a cudaStream_t passed as void*); no torch / XLA types.
 *   - every call is asynchronous on `stream`, allocates nothing, and never
 *     synchronises the host; the caller owns all buffers.
 *   - return value: 0 = ok, <0 = EAZ_ERR_*; eaz_last_error() gives a
 *     thread-local message.
 *   - bool arrays are one byte per element (0/1), as XLA lays out PRED.
 *   - batch axis B is outermost in every caller-visible array (emctx/pgx
 *     layout: [B], [B,A], [B,N], [B,N,A]).
 */
#ifndef EAZ_B200_H_
#define EAZ_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EAZ_ABI_VERSION 8

enum {
  EAZ_OK = 0,
  EAZ_ERR_INVALID_ARG = -1, /* mirrors the reference's asserts (subleq.py:606, hashes.py:154,210) */
  EAZ_ERR_WORKSPACE = -2,   /* workspace too small / misaligned */
  EAZ_ERR_CUDA = -3,        /* launch failure, message has cudaGetErrorString */
  EAZ_ERR_UNSUPPORTED = -4  /* configuration outside the fused path (no CPU fallback exists) */
};

#define EAZ_SUBLEQ_IO_LEN 8      /* MAXIMUM_INPUT_LENGTH / MAXIMUM_OUTPUT_LENGTH, envs/subleq.py:15-17 */
#define EAZ_SUBLEQ_NUM_TESTS 3   /* test cases per task, envs/subleq.py:406-454 */
#define EAZ_SUBLEQ_MAX_CYCLES 200 /* MAX_CYCLE_COUNT, envs/subleq.py:19 */
#define EAZ_FC_HIDDEN_MAX 256

int eaz_abi_version(void);
const char* eaz_last_error(void);

/* ------------------------------------------------------------------------ */
/* Environments (pgx.Env.step / init / observe; envs/deep_sea.py, envs/subleq.py) */

enum { EAZ_ENV_DEEPSEA = 0, EAZ_ENV_SUBLEQ = 1 };
enum { EAZ_SUBLEQ_REWARD_SOLVED = 0, EAZ_SUBLEQ_REWARD_LOWEST_BYTES = 1 }; /* subleq.py:535-542 */

/* Static description of the env instance (the pgx.Env object's attributes). */
typedef struct eaz_env {
  int32_t kind;              /* EAZ_ENV_* */
  /* DeepSea(size_of_grid, action_map_key), deep_sea.py:37-52 */
  int32_t size;              /* size_of_grid */
  const uint8_t* action_map; /* device bool [size,size]; NULL = all False */
  /* Subleq(tasks, word_size, reward_fn, use_binary_encoding), subleq.py:599-621 */
  int32_t word_size;         /* 16..256 */
  int32_t binary_encoding;   /* use_binary_encoding */
  int32_t reward_fn;         /* EAZ_SUBLEQ_REWARD_* */
} eaz_env;

/* pgx.State as a struct of device arrays (one per pytree leaf that carries
 * information).  DeepSeaState: deep_sea.py:12-22; SubleqState: subleq.py:545-563.
 * Leaves that are constant for these envs (current_player == 0,
 * legal_action_mask == all True) are not passed.  `observation` may be NULL:
 * it is a pure function of the other leaves (eaz_env_observe materialises it). */
typedef struct eaz_state {
  int32_t* step_count;  /* _step_count [B] */
  float* rewards;       /* rewards [B,1] */
  uint8_t* terminated;  /* [B] */
  uint8_t* truncated;   /* [B] (never set by these envs; honoured by step/auto_reset) */
  uint8_t* observation; /* optional; DeepSea bool [B,N,N]; Subleq bool [B,ws+32,w] */
  /* DeepSea */
  int32_t* col;         /* _horizontal_position [B] */
  /* Subleq */
  int32_t* memory;      /* _memory_state [B,ws] */
  int32_t* task;        /* _task [B] (SubleqTask, 1-based, subleq.py:110-124) */
  uint8_t* solved;      /* _solved [B] */
  int32_t* input_after; /* _example_input_after [B,8] */
  int32_t* output_after;/* _example_output_after [B,8] */
  /* _test_cases / _example_input / _example_output are functions of (_task, ws)
   * (subleq.py:398-501,526-527); eaz_subleq_test_cases exports them. */
} eaz_state;

/* pgx.Env.init (vmapped): DeepSea._init deep_sea.py:54-57, Subleq._init
 * subleq.py:623-646.  `task_ids` replaces jax.random.choice(key, tasks)
 * (subleq.py:624) with pre-drawn task ids [B]; ignored for DeepSea. */
int eaz_env_init(const eaz_env* env, const int32_t* task_ids, eaz_state* out, int32_t B, void* stream);

/* pgx.Env.step (vmapped) on the state in place: context.py:127 (inside the
 * search), selfplay.py:135,161,166, evaluate.py:47,54.
 * auto_reset != 0 applies the reference's own wrapper selfplay.py:26-75:
 * reset-if-already-terminal-else-step (`task_ids` then feeds the resets). */
int eaz_env_step(const eaz_env* env, eaz_state* state, const int32_t* action, int32_t auto_reset,
                 const int32_t* task_ids, int32_t B, void* stream);

/* One int32[4] trajectory record per env for the replay buffer (main.py:217-225,383-385: what the reference gathers from every
 * device after a selfplay() scan): {action, reward bits, terminated | truncated << 8 | solved << 16, first word of the compact
 * state}.  out: int32 [B,4].  A single small kernel, so that a whole self-play step stays graph-capturable without tensor glue. */
int eaz_trajectory_pack(const eaz_env* env, const eaz_state* state, const int32_t* action, int32_t* out, int32_t B, void* stream);

/* pgx.Env.observe: DeepSea._observe deep_sea.py:83-85 (one-hot cell),
 * Subleq._observe subleq.py:679-707 with the encoders subleq.py:26-98.
 * Writes bool [B, obs_dim]. */
int eaz_env_observe(const eaz_env* env, const eaz_state* state, uint8_t* observation, int32_t B, void* stream);

/* Number of actions / flattened observation length / rows x cols for an env. */
int32_t eaz_env_num_actions(const eaz_env* env);
int32_t eaz_env_obs_dim(const eaz_env* env);
int32_t eaz_env_obs_cols(const eaz_env* env);
/* Length of the hash input for the FC net: whole observation, or the IO block
 * only when hash_io (fully_connected.py:85-89). */
int32_t eaz_env_hash_dim(const eaz_env* env, int32_t hash_io);

/* get_test_cases(task, ws), subleq.py:398-501: host-side export of the padded
 * test inputs / outputs, int32 [3,8] each (host pointers). */
int eaz_subleq_test_cases(int32_t task, int32_t word_size, int32_t* inputs, int32_t* outputs);

/* ------------------------------------------------------------------------ */
/* Hash-count novelty (network/hashes.py)                                     */

/* XXHash.get_indices hashes.py:162-229 on float32 rows x[B,D] (D % 4 == 0,
 * hashes.py:210; 0 < bits <= 32, hashes.py:154). */
int eaz_xxhash_indices(const float* x, int32_t B, int32_t D, int32_t bits, uint32_t* indices, void* stream);
/* BaseHash.__call__ hashes.py:29-38: seen[b] = bit `indices[b]` of binary_set. */
int eaz_hash_lookup(const float* x, int32_t B, int32_t D, int32_t bits, const uint8_t* binary_set,
                    uint8_t* seen, void* stream);
/* BaseHash.update hashes.py:45-50 (train-side; atomic OR into binary_set). */
int eaz_hash_update(const float* x, int32_t B, int32_t D, int32_t bits, uint8_t* binary_set, void* stream);

/* ------------------------------------------------------------------------ */
/* EpistemicFullyConnectedAZNet (network/fully_connected.py:41-101)           */

/* haiku parameter pytree `fc_az_net/linear{,_1..11}`: w [in,out] row-major,
 * b [out]; module order = call order in fully_connected.py:49-81:
 * value head (linear, _1, _2), UBE head (_3.._5), exploitation policy head
 * (_6.._8), exploration policy head (_9.._11).  State `fc_az_net/xxhash32`
 * binary_set uint8[2^(bits-3)]. */
enum { EAZ_HEAD_VALUE = 0, EAZ_HEAD_UBE = 1, EAZ_HEAD_EXPLOIT = 2, EAZ_HEAD_EXPLORE = 3 };
typedef struct eaz_fc_params {
  int32_t in_dim;      /* flattened observation length D */
  int32_t hidden;      /* layer_size (config.linear_layer_size, 256) */
  int32_t num_actions;
  const float* w[4][3];
  const float* b[4][3];
  const uint8_t* binary_set; /* hash state */
  int32_t hash_bits;         /* bits_per_hash (24) */
  int32_t hash_io;           /* fully_connected.py:85: hash rows word_size: only */
  int32_t word_size;         /* fully_connected.py:26,86: first row of the hashed IO block (0 for DeepSea) */
  float max_u;               /* max_ube (1.0; context.py:68-75 never forwards config.max_ube) */
  float novelty_scale;       /* max_epistemic_variance_reward (1.0) */
} eaz_fc_params;

/* forward.apply(params, state, observation, is_training=False): the root
 * evaluation of selfplay.py:89, reanalyze.py:67,90, evaluate.py:29.
 * observation: bool [B,D].  Outputs (fully_connected.py:101 order), any may be
 * NULL: exploit logits [B,A], explore logits [B,A], value [B], ube [B]
 * (already max(novelty,u) clipped, :92-96), novelty [B]. */
int eaz_mlp_forward(const eaz_fc_params* net, const uint8_t* observation, int32_t B, float* exploit_logits,
                    float* explore_logits, float* value, float* ube, float* novelty, void* stream);

/* Same network evaluated straight from env states (no materialised
 * observation): what the fused recurrent_fn uses. */
int eaz_mlp_forward_states(const eaz_fc_params* net, const eaz_env* env, const eaz_state* state, int32_t B,
                           float* exploit_logits, float* explore_logits, float* value, float* ube,
                           float* novelty, void* workspace, size_t workspace_bytes, void* stream);
/* workspace for the call above: B * eaz_env_compact_bytes(env), 16-byte aligned */

/* Pack pgx.State leaves into the compact in-tree encoding, out: uint8 [B, eaz_env_compact_bytes]. */
int eaz_env_compact(const eaz_env* env, const eaz_state* state, uint8_t* out, int32_t B, void* stream);

/* Inverse of eaz_env_compact: compact records [B, eaz_env_compact_bytes] (+ the rewards leaf [B], NULL = zeros, which
 * the compact encoding does not carry) -> pgx.State leaves; `out->observation`, if non-NULL, is materialised too.
 * This is the decode step of a compact replay buffer (the reference's flashbax buffer, main.py:217-225,383-385, stores
 * a full pgx.State per step: 25x..2500x larger). */
int eaz_env_uncompact(const eaz_env* env, const uint8_t* compact, const float* rewards, eaz_state* out, int32_t B, void* stream);

/* ------------------------------------------------------------------------ */
/* emctx.epistemic_gumbel_muzero_policy (selfplay.py:107-117,                  */
/* reanalyze.py:77-85, evaluate.py:36-45) with the recurrent_fn of            */
/* context.py:109-157 fused in.                                               */

/* Switches for the emctx details that cannot be pinned in this environment
 * (SURVEY.md Appendix A.8). Defaults (flags = EAZ_SEARCH_DEFAULT_FLAGS) follow
 * Appendix A as written. */
enum {
  EAZ_FLAG_BETA_INTERIOR = 1 << 0, /* beta*sqrt(var) bonus inside the qtransform at interior nodes too */
  EAZ_FLAG_BETA_RAW = 1 << 1,      /* mixed value built from raw + beta*sqrt(raw_var) */
  EAZ_FLAG_BETA_FINAL = 1 << 2,    /* final action / action_weights use the beta-adjusted qtransform */
  EAZ_FLAG_BACKUP_STD = 1 << 3,    /* back up a running mean of std instead of variance */
  /* Not an emctx switch: the workspace still holds the parameter-derived tables (sequential-halving table, DeepSea
   * per-cell novelty table, tensor-path weight images) that an earlier eaz_search_gumbel call with the same cfg / env /
   * net wrote into THIS workspace -- skip rebuilding them.  The model is constant across the steps of one selfplay()
   * scan (selfplay.py:148) and one reanalyze() call; the caller clears the flag after every learner update. */
  EAZ_FLAG_REUSE_PREPARED = 1 << 4,
  /* Also not an emctx switch: bits 8..11 = k (2..8): cut the batch into k sub-batches of whole 128-tree tiles and search them
   * concurrently on library-owned auxiliary streams, forked from and joined back into `stream` (CUDA-graph capturable).  Trees
   * never interact, so the results are bit-identical to k = 0/1; the point is overlap -- one sub-batch's tree kernel runs while
   * another's network kernel does.  eaz_search_workspace_bytes accounts for the k separate layouts. */
  EAZ_FLAG_STREAMS_SHIFT = 8,
  /* emctx.epistemic_muzero_policy instead of the Gumbel policy (named by the task, never called by the reference): PUCT at the
   * root and inside the tree (mctx action_selection.muzero_action_selection with qtransform_by_parent_and_siblings; the
   * beta * sqrt(variance) bonus enters q exactly as in the Gumbel path), action ~ visit counts, action_weights = visit_probs
   * (mctx policies.muzero_policy).  Randomness is supplied / derived, not drawn from a JAX key: the caller mixes the Dirichlet
   * noise into `prior_logits`; `gumbel` is the noise of the final categorical draw; the 1e-7 tie-break noise of every
   * selection is a counter-based stream keyed by (noise_seed, tree, node, visit count of the node, action). */
  EAZ_FLAG_PUCT = 1 << 5,
  EAZ_SEARCH_DEFAULT_FLAGS = (1 << 0) | (1 << 1) | (1 << 2)
};
#define EAZ_FLAG_STREAMS(k) ((k) << EAZ_FLAG_STREAMS_SHIFT)

typedef struct eaz_search_config {
  int32_t batch;            /* B (per device) */
  int32_t num_simulations;  /* n; tree has n+1 nodes */
  int32_t max_depth;        /* 0 = None -> num_simulations (mctx search.py) */
  int32_t max_num_considered_actions; /* 16 */
  float gumbel_scale;       /* 1.0; evaluate.py:44 passes 0.0 */
  float discount;           /* get_epistemic_recurrent_fn(discount=), context.py:114 */
  int32_t two_players_game; /* context.py:115,142-143 */
  int32_t exploration;      /* context.py:113,132: recurrent_fn uses the exploration policy head */
  /* epistemic_qtransform_completed_by_mix_value(value_scale, maxvisit_init,
   * rescale_values, use_mixed_value, epsilon) */
  float value_scale;        /* 0.1 */
  float maxvisit_init;      /* 50.0 */
  int32_t rescale_values;   /* selfplay.py:114-116 */
  int32_t use_mixed_value;  /* 1 */
  float epsilon;            /* 1e-8 */
  int32_t flags;            /* EAZ_FLAG_* */
  int32_t mlp_mode;         /* EAZ_MLP_* */
  /* ABI 2 (appended): mctx muzero_policy parameters, read only with EAZ_FLAG_PUCT */
  float pb_c_init;          /* 1.25 */
  float pb_c_base;          /* 19652 */
  float temperature;        /* 1.0; also the temperature of the draw of action_sampling != EAZ_ACTION_SEARCH */
  uint32_t noise_seed;      /* tie-break noise stream */
  /* ABI 5 (appended): the optional parts of the self-play step (selfplay.py:92-98, 125-134); 0 = off, not with EAZ_FLAG_PUCT */
  int32_t root_prior;       /* EAZ_ROOT_PRIOR_* */
  int32_t action_sampling;  /* EAZ_ACTION_* */
} eaz_search_config;

/* Root prior (selfplay.py:92-98).  UNIFORM: the root's prior logits are 0 for every action (then _mask_invalid_actions: invalid ones get
 * EAZ_F32_MIN), whatever prior_logits holds and also with a fused root; the root value / UBE and every node below the root are
 * unchanged. */
enum { EAZ_ROOT_PRIOR_GIVEN = 0, EAZ_ROOT_PRIOR_UNIFORM = 1 };
/* Played action (selfplay.py:125-134).  SEARCH: the Gumbel policy's action.  VISITS / IMPROVED: a categorical draw from the visit
 * probabilities / from this search's action_weights, as the Gumbel-max argmax over valid, not invalid actions of
 * (x_a - max_a x_a) / max(tiny, temperature) + g_a with x_a = log(max(w_a, tiny)) and g = sample_gumbel (ties: lowest index; a row
 * whose actions are all invalid plays 0).  Only `action` changes; action_weights and the summary are those of the search. */
enum { EAZ_ACTION_SEARCH = 0, EAZ_ACTION_VISITS = 1, EAZ_ACTION_IMPROVED = 2 };

enum {
  EAZ_MLP_EXACT = 0, /* fp32 FMA chains in index order: bit-identical to the oracle */
  EAZ_MLP_TENSOR = 1 /* tcgen05 split-precision tensor-core GEMMs (<=1e-5 rel. of EXACT) */
};

typedef struct eaz_search_inputs {
  /* EpistemicRootFnOutput, selfplay.py:100-106 */
  const float* prior_logits;             /* [B,A] raw root logits.  NULL (together with value and
                                            value_epistemic_variance) = FUSED ROOT: the library evaluates the root
                                            itself, i.e. forward.apply on `embedding` (selfplay.py:89) with the policy
                                            head the recurrent_fn uses (`exploration`), and reports the value / UBE
                                            predictions in eaz_search_outputs.root_value / root_ube */
  const float* value;                    /* [B] */
  const float* value_epistemic_variance; /* [B] */
  const float* beta;                     /* [B] */
  const eaz_state* embedding;            /* root states (pgx.State) */
  const uint8_t* invalid_actions;        /* [B,A] bool, NULL = none (selfplay.py:113) */
  const float* gumbel;                   /* [B,A] pre-drawn standard Gumbel noise (replaces
                                            jax.random.gumbel(gumbel_rng), mctx policies.py); NULL = drawn inside the
                                            search from a counter-based stream keyed by (cfg.noise_seed, number of such
                                            searches run on this workspace so far, tree, action) */
  const eaz_env* env;
  const eaz_fc_params* net;              /* params=model */
  /* ABI 5 (appended) */
  const float* sample_gumbel;            /* [B,A] pre-drawn standard Gumbel noise of the action draw (cfg.action_sampling != 0; not
                                            scaled by gumbel_scale).  NULL = drawn inside the search from the stream of `gumbel`
                                            with one more xx round by 0x53414D50 after the action: (noise_seed, the same draw
                                            counter value, tree, action).  The workspace's draw counter advances once per search
                                            that draws either noise itself */
} eaz_search_inputs;

typedef struct eaz_search_outputs {
  /* PolicyOutput */
  int32_t* action;       /* [B] */
  float* action_weights; /* [B,A] */
  /* search_tree.epistemic_summary(), selfplay.py:119-142, reanalyze.py:86-116 */
  float* value;                      /* [B] */
  float* value_epistemic_std;        /* [B] */
  float* visit_counts;               /* [B,A] (as float, like mctx) */
  float* visit_probs;                /* [B,A] */
  float* qvalues;                    /* [B,A] */
  float* qvalues_epistemic_variance; /* [B,A] */
  /* Optional full tree in emctx layout (all NULL to skip). N = n+1. */
  int32_t* node_visits;                       /* [B,N] */
  float* raw_values;                          /* [B,N] */
  float* node_values;                         /* [B,N] */
  float* raw_values_epistemic_variance;       /* [B,N] */
  float* node_values_epistemic_variance;      /* [B,N] */
  int32_t* parents;                           /* [B,N] */
  int32_t* action_from_parent;                /* [B,N] */
  int32_t* children_index;                    /* [B,N,A] */
  float* children_prior_logits;               /* [B,N,A] */
  int32_t* children_visits;                   /* [B,N,A] */
  float* children_rewards;                    /* [B,N,A] */
  float* children_discounts;                  /* [B,N,A] */
  float* children_values;                     /* [B,N,A] */
  float* children_rewards_epistemic_variance; /* [B,N,A] (identically 0, context.py:149) */
  float* children_values_epistemic_variance;  /* [B,N,A] */
  uint8_t* embeddings;                        /* [B,N,S] compact per-node env states, S = eaz_env_compact_bytes */
  /* fused-root mode only (optional): the root network outputs, selfplay.py:139-140 value_prediction / ube_prediction */
  float* root_value;                          /* [B] */
  float* root_ube;                            /* [B] */
} eaz_search_outputs;

/* Bytes per compact (in-tree) env state. */
int32_t eaz_env_compact_bytes(const eaz_env* env);

size_t eaz_search_workspace_bytes(const eaz_search_config* cfg, const eaz_env* env);

/* One whole search for B roots; async on `stream`.  The launch sequence is
 * fixed for a given (cfg, env), so callers may capture it in a CUDA graph. */
int eaz_search_gumbel(const eaz_search_config* cfg, const eaz_search_inputs* in, eaz_search_outputs* out,
                      void* workspace, size_t workspace_bytes, void* stream);

/* Measurement aid (bench.py's roofline breakdown): the same search with CUDA events recorded around every
 * launch on `stream`; SYNCHRONISES the stream and returns summed milliseconds and launch counts per kernel
 * class (host arrays of EAZ_PROFILE_CLASSES entries: init, select, env step, network, expand+backward,
 * finalize, export). */
#define EAZ_PROFILE_CLASSES 7
int eaz_search_gumbel_profiled(const eaz_search_config* cfg, const eaz_search_inputs* in, eaz_search_outputs* out,
                               void* workspace, size_t workspace_bytes, void* stream, float* ms_by_class,
                               int32_t* launches_by_class);

/* Range guard of mlp_mode TENSOR (the scaled 3xFP16 split, fully_connected.py:41-101 evaluated on tcgen05): every weight image carries
 * a power-of-two scale chosen from the matrix's own max |w|, so weights never saturate; what CAN leave the representable range is a
 * hidden activation above 4094 (clamped) or a non-finite weight.  Both set sticky device flags in the workspace (reset whenever the
 * parameter-derived tables are rebuilt).  This call SYNCHRONISES `stream`, reads them (bit 0: weights non-finite / > 2^20, bit 1:
 * activation clamped) into *flags_out and returns EAZ_ERR_UNSUPPORTED with a message if any is set, 0 otherwise. */
int eaz_search_numeric_status(const eaz_search_config* cfg, const eaz_env* env, const void* workspace, size_t workspace_bytes,
                              void* stream, int32_t* flags_out);

/* Number of kernel launches one eaz_search_gumbel call enqueues (for bench.py's
 * gpu_launches accounting). */
int32_t eaz_search_num_launches(const eaz_search_config* cfg, const eaz_env* env);

/* ------------------------------------------------------------------------ */
/* ABI 6 (appended): the evaluation loop of evaluate.py:13-57 as one device    */
/* program -- a CUDA graph whose WHILE conditional node repeats {fused-root    */
/* search, env step, returns += rewards[:,0]} and whose condition the device   */
/* computes: continue while any env is not terminated and moves <=             */
/* max_episode_length (cond_fn, evaluate.py:18-20).                            */

/* The loop's device words, at the start of the evaluate workspace.  After an eaz_evaluate call has finished: moves = the number of
 * moves it ran, cont = 0, live = ticket = 0. */
typedef struct eaz_evaluate_counters {
  int32_t moves;   /* moves run so far in this call */
  int32_t live;    /* envs not terminated after the current move (summed over the CTAs of the step kernel) */
  uint32_t ticket; /* CTAs of the step kernel done with the current move */
  int32_t cont;    /* the loop condition after the last move */
} eaz_evaluate_counters;

/* Workspace of eaz_evaluate (256-byte aligned): the counters, zero Gumbel noise [B,A], the played actions [B] and the search workspace of
 * `cfg`.  0 if cfg / env are rejected. */
size_t eaz_evaluate_workspace_bytes(const eaz_search_config* cfg, const eaz_env* env);

/* Greedy evaluation episodes (evaluate.py:13-57) from `states` (the output of eaz_env_init: no env terminated, so the first move always
 * runs, as in the reference): while any env is not terminated and moves <= max_episode_length, the fused-root search of `cfg` with
 * zero Gumbel noise picks an action per env (cfg->gumbel_scale must be 0 and cfg->action_sampling EAZ_ACTION_SEARCH), pgx.Env.step
 * advances `states` in place (no auto-reset: terminated envs are absorbing) and returns[b] += rewards[b,0], starting from 0.
 * From `in` it reads env, beta [B] and invalid_actions (may be NULL); prior_logits / value / value_epistemic_variance must be NULL
 * (fused root); the other fields are not read.  A negative max_episode_length runs no move (returns = 0).
 * The parameter-derived tables are rebuilt once per call, before the loop.  The loop is a CUDA graph built on the first call for a
 * workspace and kept with it; a call with another cfg / env / net / buffer address rebuilds it.  Asynchronous on `stream`: no
 * allocation of device memory, no host synchronisation after the graph of the workspace is built. */
int eaz_evaluate(const eaz_search_config* cfg, const eaz_search_inputs* in, const eaz_fc_params* net, eaz_state* states, float* returns,
                 int32_t max_episode_length, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------ */
/* ABI 7 (appended): the self-play scan of selfplay.py:78-149 as one device    */
/* program -- lax.scan(step_fn, starting_states, key_seq) over T steps of      */
/* {fused-root search, auto-reset env step, row t of every stacked output},    */
/* a CUDA graph whose WHILE conditional node the device stops after T steps.   */

/* The stacked per-step outputs of the scan (SelfplayOutput, selfplay.py:17-23, stacked over the steps as lax.scan stacks them).  Row t
 * holds what step t returns; every pointer may be NULL (not written).  A = eaz_env_num_actions, S = eaz_env_compact_bytes. */
typedef struct eaz_selfplay_outputs {
  int32_t* action;                    /* [T,B] the played action (the sampled one with cfg.action_sampling != EAZ_ACTION_SEARCH) */
  float* root_value;                  /* [T,B] search summary value (selfplay.py:137) */
  float* root_epistemic_std;          /* [T,B] search summary value_epistemic_std (:138) */
  float* value_prediction;            /* [T,B] the fused root's network value (:139) */
  float* ube_prediction;              /* [T,B] the fused root's network UBE (:140) */
  float* q_values_epistemic_variance; /* [T,B,A] search summary qvalues_epistemic_variance (:141) */
  int32_t* trajectory;                /* [T,B,4] the eaz_trajectory_pack record of the states AFTER step t and its played action */
  uint8_t* states;                    /* [T,B,S] SelfplayOutput.state: the states AFTER step t (auto-reset applied), eaz_env_compact
                                         encoding -- the replay ring's format, decodable with eaz_env_uncompact */
  float* rewards;                     /* [T,B] rewards[:,0] of the states after step t (the leaf the compact encoding does not carry) */
} eaz_selfplay_outputs;

/* Workspace of eaz_selfplay (256-byte aligned): the loop's device words, the staged noise of one step (gumbel and sample_gumbel, [B,A]
 * each), one step's search outputs and the search workspace of `cfg`.  0 if cfg / env are rejected. */
size_t eaz_selfplay_workspace_bytes(const eaz_search_config* cfg, const eaz_env* env);

/* selfplay() (selfplay.py:78-149): T steps of step_fn (selfplay.py:86-143) from `states`, stepped in place -- on return `states` holds
 * the final carry.  Step t: the fused-root search of `cfg` (forward.apply on the states, selfplay.py:89, with the recurrent_fn's policy
 * head; root_prior / action_sampling / temperature as in eaz_search_gumbel), the auto-reset env step on the played actions
 * (selfplay.py:26-75,135; Subleq resets take their task from row t of task_ids [T,B], required for Subleq, ignored for DeepSea) and
 * row t of every non-NULL output of `out`.
 * From `in` it reads env, beta [B] (non-NULL), invalid_actions [B,A] (may be NULL; the same for every step) and the noise:
 * gumbel / sample_gumbel are [T,B,A] (row t for step t) or NULL = drawn inside the search from (cfg.noise_seed, the workspace's draw
 * counter, which advances once per step whose search draws noise itself, tree, action).  prior_logits / value /
 * value_epistemic_variance must be NULL (fused root); the other fields are not read.  EAZ_FLAG_PUCT is refused (the reference's
 * self-play uses the Gumbel policy).  states->observation must be NULL (the loop does not materialise observations).  T == 0 writes
 * and enqueues nothing.  Every argument is checked before anything is enqueued.
 * The parameter-derived tables are rebuilt once per call, before the loop, unless cfg->flags has EAZ_FLAG_REUSE_PREPARED (an earlier
 * call on this workspace built them for the same net); this does not advance the draw counter.  The loop is a CUDA graph built on the
 * first call for a workspace and kept with it; a call with another cfg / env / net / T / buffer address rebuilds it.  Asynchronous on
 * `stream`: no allocation of device memory, no host synchronisation after the graph of the workspace is built. */
int eaz_selfplay(const eaz_search_config* cfg, const eaz_search_inputs* in, const eaz_fc_params* net, eaz_state* states, int32_t T,
                 const int32_t* task_ids, eaz_selfplay_outputs* out, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------ */
/* Convolutional evaluators (SURVEY 8f-4): EpistemicResidualAZNet               */
/* (network/resnet.py:41-135, the default for every pgx env that is not       */
/* DeepSea / Subleq / MinAtar, context.py:76-82) and EpistemicMinatarAZNet    */
/* (network/minatar.py:11-114) in inference mode: forward.apply(params, state, */
/* observation, is_training=False), the root / leaf evaluation of             */
/* selfplay.py:89 and context.py:128-131.  fp32 in the reference's operation  */
/* order (the EXACT contract of eaz_mlp_forward: bit-identical to the oracle). */

enum { EAZ_CONVNET_RESNET = 0, EAZ_CONVNET_MINATAR = 1 };
#define EAZ_CONVNET_MAX_BLOCKS 8
/* haiku parameter / state leaves as device pointers.  hk.Conv2D: w [kh,kw,in,out] (HWIO), b [out]; hk.Linear: w [in,out], b [out];
 * hk.BatchNorm(create_scale, create_offset, decay 0.9) in inference: scale, offset (params) and the `average` leaves of
 * mean_ema / var_ema (state), eps = 1e-5. */
typedef struct eaz_conv { const float* w; const float* b; } eaz_conv;      /* also hk.Linear */
typedef struct eaz_bn { const float* scale; const float* offset; const float* mean; const float* var; } eaz_bn;
typedef struct eaz_convnet_params {
  int32_t kind;          /* EAZ_CONVNET_* */
  int32_t height, width, in_channels; /* observation [B,H,W,C] bool (pgx board / MinAtar frame) */
  int32_t num_actions;
  int32_t num_channels;  /* resnet: 64; minatar: 16 (conv channels) */
  int32_t hidden;        /* minatar: hidden_layers_size 64; resnet: value / UBE head width = num_channels */
  int32_t num_blocks;    /* resnet: 5 */
  int32_t resnet_v2;     /* resnet.py:50 */
  /* --- resnet (resnet.py:70-135, module call order) */
  eaz_conv stem;                                   /* az_resnet/conv2_d */
  eaz_bn stem_bn;                                  /* v1 only (:73-75) */
  eaz_bn block_bn[EAZ_CONVNET_MAX_BLOCKS][2];      /* block_i/batch_norm, batch_norm_1 */
  eaz_conv block_conv[EAZ_CONVNET_MAX_BLOCKS][2];  /* block_i/conv2_d, conv2_d_1 */
  eaz_bn final_bn;                                 /* v2 only (:80-82) */
  /* heads in call order: [0] main policy, [1] exploration policy, [2] value, [3] ube (:84-124) */
  eaz_conv head_conv[4];                           /* 1x1 conv to 2 / 2 / 1 / 1 channels */
  eaz_bn head_bn[4];
  eaz_conv head_fc[4];                             /* Linear(num_actions) / Linear(num_actions) / Linear(num_channels) x2 */
  eaz_conv head_out[4];                            /* [2], [3] only: Linear(1) */
  /* --- minatar (minatar.py:55-95): towers [0] = x1 (main policy + value), [1] = x2 (exploration policy + ube) */
  eaz_conv tower_conv[2];
  eaz_conv tower_fc[2][2];
  eaz_conv mhead_fc[4][2];                         /* [0] main policy, [1] value, [2] exploration policy, [3] ube: Linear(hidden), Linear(out) */
  /* --- hash-count novelty on the float32 observation (hashes.py:23-38,162-229; H*W*C % 4 == 0) */
  const uint8_t* binary_set;
  int32_t hash_bits;
  float max_u;                /* resnet.py:62 / minatar max_ube */
  float novelty_scale;        /* max_reward_epistemic_variance */
  float local_unc_scale;      /* minatar.py:50: 1 / (1 - min(discount, 0.9997)^2); unused for resnet */
  int32_t mlp_mode;           /* EAZ_MLP_EXACT: fp32 in the reference's order, bit-identical to the oracle.  EAZ_MLP_TENSOR (resnet v2 with
                                 64 channels): the 64 -> 64 convolutions of the residual blocks as tcgen05 implicit GEMMs on the scaled
                                 3xFP16 split (<= 1e-5 of EXACT relative to the magnitude of the terms); stem and heads stay fp32 */
} eaz_convnet_params;

/* Scratch for B observations (activations ping-pong), 256-byte aligned. */
size_t eaz_convnet_workspace_bytes(const eaz_convnet_params* net, int32_t B);
/* observation: bool [B,H,W,C].  Outputs as eaz_mlp_forward (any may be NULL): main policy logits [B,A], exploration policy logits
 * [B,A], value [B] (resnet: tanh, :102; minatar: linear, :69), ube [B] (max(novelty, u), resnet.py:126-128; minatar.py:101-104 with
 * the local-uncertainty scale and the clip), novelty [B]. */
int eaz_convnet_forward(const eaz_convnet_params* net, const uint8_t* observation, int32_t B, float* exploit_logits,
                        float* explore_logits, float* value, float* ube, float* novelty, void* workspace, size_t workspace_bytes,
                        void* stream);
/* Range guard of mlp_mode TENSOR, as eaz_search_numeric_status: SYNCHRONISES `stream`, reads the sticky flags the last
 * eaz_convnet_forward on this workspace left (bit 0: a weight tensor non-finite / > 2^20, bit 1: an activation above 4094 was clamped)
 * and returns EAZ_ERR_UNSUPPORTED with a message if any is set. */
int eaz_convnet_numeric_status(const eaz_convnet_params* net, int32_t B, const void* workspace, size_t workspace_bytes, void* stream,
                               int32_t* flags_out);

/* ------------------------------------------------------------------------ */
/* reanalyze target computation (reanalyze.py:86-129) on the summary of a      */
/* finished search: the epilogue that follows epistemic_gumbel_muzero_policy   */
/* in reanalyze().                                                             */

typedef struct eaz_reanalyze_config {
  float discount;                              /* config.discount (reanalyze.py:94) */
  float exploration_beta;                      /* config.exploration_beta (:114-116) */
  int32_t exploration_ube_target;              /* config.exploration_ube_target (:106): max child uncertainty vs the chosen child's */
  float exploration_policy_target_temperature; /* config.exploration_policy_target_temperature (:121) */
} eaz_reanalyze_config;

/* Inputs: policy_output.action [B]; search_summary.qvalues / qvalues_epistemic_variance / visit_counts [B,A],
 * value / value_epistemic_std [B]; next_state_value [B] = forward.apply(...) on experience_pair.second.observation
 * (:90-92); next_rewards = second.rewards.squeeze() [B]; next_terminated = second.terminated [B]; terminated =
 * states.terminated [B]; invalid_actions = ~states.legal_action_mask [B,A] (NULL = none invalid).
 * Outputs: value_target [B] = max(q[action], r' + discount * v(s') * !term') * !term (:87-111),
 * ube_target [B] (:103-111), exploration_policy_target [B,A] = softmax(mask_invalid(complete_qs(q + beta*sqrt(qvar),
 * visits, value + beta*std)) * temperature) (:113-122).  exploitation_policy_target is policy_output.action_weights. */
int eaz_reanalyze_targets(const eaz_reanalyze_config* cfg, int32_t B, int32_t A, const int32_t* action, const float* qvalues,
                          const float* qvalues_epistemic_variance, const float* visit_counts, const float* value,
                          const float* value_epistemic_std, const float* next_state_value, const float* next_rewards,
                          const uint8_t* next_terminated, const uint8_t* terminated, const uint8_t* invalid_actions,
                          float* value_target, float* ube_target, float* exploration_policy_target, void* stream);

/* ------------------------------------------------------------------------ */
/* Prioritised replay sampling (SURVEY 8f-3): the sum tree of the reference's  */
/* flashbax prioritised flat buffer (main.py:217-225 priority_exponent,        */
/* main.py:413-414 sample + batch.indices, main.py:454 set_priorities) over a  */
/* compact replay ring of T time slots x B envs.  Item i = t * B + b is the    */
/* pair (slot t, slot (t+1) % T) of env b; its weight is priority^exponent.    */
/* The tree, its header (cursor, length, max priority, draw counter, sticky    */
/* status) and the descent / node-sum / stratification order are specified in  */
/* csrc/replay.cu; every call below is asynchronous on `stream`, allocates     */
/* nothing and does not synchronise (except eaz_priority_status).              */

enum {
  EAZ_PRIORITY_BAD_PRIORITY = 1 << 0, /* a negative or non-finite priority was stored as 0 */
  EAZ_PRIORITY_BAD_INDEX = 1 << 1,    /* an index outside [0, T*B) was skipped */
  EAZ_PRIORITY_EMPTY = 1 << 2,        /* sampled a tree whose total weight was 0 (outputs: index 0, probability 0) */
  EAZ_PRIORITY_BAD_ADD = 1 << 3       /* add_step for a slot that is neither the cursor nor the newest slot (ignored) */
};

/* Bytes of the caller-owned tree buffer for T >= 2 slots x B >= 1 envs (T * B < 2^31); 0 (and a message) otherwise.
 * The buffer must be 128-byte aligned. */
size_t eaz_priority_tree_bytes(int32_t T, int32_t B);
/* Zero the tree and write the header: exponent (0 <= alpha <= 1), seed, max priority 1, draw counter 0, cursor 0, length 0. */
int eaz_priority_init(void* tree, size_t tree_bytes, int32_t T, int32_t B, float priority_exponent, uint32_t seed, void* stream);
/* Slot `slot` of the ring has just been written (the ring's add): the items starting at slot-1 get max_priority^alpha, the
 * items starting at `slot` get 0; cursor / length advance (or stay, when the newest slot was rewritten). */
int eaz_priority_add_step(void* tree, size_t tree_bytes, int32_t T, int32_t B, int32_t slot, void* stream);
/* flashbax set_priorities: leaves indices[k] = priorities[k]^alpha for the K device entries (the last occurrence of a duplicated
 * index wins; invalid items keep weight 0), max_priority = max(max_priority, priorities), ancestors recomputed. */
int eaz_priority_set(void* tree, size_t tree_bytes, int32_t T, int32_t B, const int32_t* indices, const float* priorities, int32_t K,
                     void* stream);
/* flashbax sample: K stratified draws (1 <= K <= 2^24) -> indices [K] and probabilities [K] = weight / total.  If `states`
 * (the ring's compact records [T,B,S]) is non-NULL the same kernel gathers both slots of every drawn pair into first / second
 * [K,S] (and `rewards` [T,B], if non-NULL, into first_rewards / second_rewards [K]) for eaz_env_uncompact.  Advances the draw
 * counter. */
int eaz_priority_sample(void* tree, size_t tree_bytes, int32_t T, int32_t B, int32_t K, const uint8_t* states, const float* rewards, int32_t S,
                        int32_t* indices, float* probabilities, uint8_t* first, float* first_rewards, uint8_t* second,
                        float* second_rewards, void* stream);
/* SYNCHRONISES `stream` and reads the sticky EAZ_PRIORITY_* bits into *flags_out; returns EAZ_ERR_UNSUPPORTED with a message if
 * any is set, 0 otherwise. */
int eaz_priority_status(const void* tree, size_t tree_bytes, void* stream, int32_t* flags_out);

/* ABI 4 (appended): the replay ring with its cursor on the device, for callers that cannot keep it on the host (a jitted JAX
 * program, a CUDA graph replayed many times). */

/* The ring's add at the DEVICE cursor (slot = the header's cursor, never read by the host): `state`'s B envs go into
 * ring_states[slot] [B,S] in the eaz_env_compact encoding and rewards[:,0] into ring_rewards[slot] [B], then add_step(slot).  The
 * result equals eaz_env_compact + the row copies + eaz_priority_add_step(tree, ..., cursor) bit for bit.  Two launches. */
int eaz_replay_add(const eaz_env* env, const eaz_state* state, uint8_t* ring_states, float* ring_rewards, void* tree, size_t tree_bytes,
                   int32_t T, int32_t B, void* stream);
/* eaz_priority_sample with (seed, draw counter) taken from `key` (device uint32[2]) instead of the header.  Writes nothing into
 * the tree (no counter advance, no status bit): a pure function of the tree, the ring and the key.  An empty tree gives index 0,
 * probability 0. */
int eaz_priority_sample_keyed(const void* tree, size_t tree_bytes, int32_t T, int32_t B, int32_t K, const uint32_t* key, const uint8_t* states,
                              const float* rewards, int32_t S, int32_t* indices, float* probabilities, uint8_t* first, float* first_rewards,
                              uint8_t* second, float* second_rewards, void* stream);
/* Copies the sticky EAZ_PRIORITY_* word into the device int32 *flags_dev on `stream`; does not synchronise. */
int eaz_priority_status_async(const void* tree, size_t tree_bytes, int32_t* flags_dev, void* stream);

/* ABI 8 (appended): a whole self-play scan into the ring in one call -- flashbax's add with add_sequences=True after the scan
 * (main.py:383-385). */

/* Appends `steps` time steps to the ring at the DEVICE cursor: row j of compact [steps,B,S] (eaz_env_compact records, e.g.
 * eaz_selfplay_outputs.states) and of rewards [steps,B] goes to slot (c + j) % T, c = the header's cursor, so only the last T rows
 * survive when steps > T.  The tree buffer, header included, ends exactly as after `steps` calls of eaz_replay_add (add_step at the
 * header's cursor each time), from any ring state.  S must equal eaz_env_compact_bytes(env); compact / rewards may be NULL only
 * when steps == 0, which enqueues nothing.  Every argument is checked before anything is enqueued.  L + 1 launches for a tree of L
 * levels, independent of `steps`; no allocation, no synchronisation. */
int eaz_replay_add_sequence(const eaz_env* env, const uint8_t* compact, const float* rewards, int32_t steps, uint8_t* ring_states,
                            float* ring_rewards, void* tree, size_t tree_bytes, int32_t T, int32_t B, int32_t S, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EAZ_B200_H_ */
