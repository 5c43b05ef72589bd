// search.cu -- emctx.epistemic_gumbel_muzero_policy for B independent trees
// (call sites: selfplay.py:107-117, reanalyze.py:77-85, evaluate.py:36-45) with
// the recurrent_fn of context.py:109-157 fused in.  Algorithm: mctx search.py /
// action_selection.py / qtransforms.py / seq_halving.py / policies.py plus the
// epistemic extension of SURVEY.md Appendix A (assumptions = EAZ_FLAG_*).
//
// Data layout (workspace): the tree is a struct of arrays, NODE-major:
//   node arrays  [N][B]      visits, raw/node value, raw/node variance, link{parent,action}
//   edge arrays  [N][B][A]   child index, prior logit, visits, reward, discount, value, value variance
//   states       [N][B][S]   compact env state per node
// so that everything written for the node expanded in simulation i (the same
// node index i+1 for every tree) and everything read at the root is contiguous
// across the batch.  G = min(32, pow2(A)) lanes cooperate on one tree: lane g owns
// actions g, g+G, ...; all reductions over actions are warp shuffles in the
// fixed order shared with the oracle (common.cuh).
//
// Per simulation: select (+ fused DeepSea step | Subleq step kernel) -> network
// -> expand + backward.  Everything is enqueued on the caller's stream with no
// host synchronisation, so a whole search is CUDA-graph capturable.
//
// The optional parts of the self-play step (cfg.root_prior / action_sampling,
// selfplay.py:92-98,125-134) live in root_init_kernel and finalize_kernel, which
// every search path (persistent, launch chain, stream sub-batch) runs.
#include "mlp.cuh"

#include <cstdlib>
#include <mutex>
#include <vector>

namespace eaz {

// ---- optional per-kernel-class timing (eaz_search_gumbel_profiled): CUDA events around every launch
enum { CLS_INIT = 0, CLS_SELECT, CLS_ENV, CLS_MLP, CLS_EXPAND, CLS_FINAL, CLS_EXPORT, CLS_COUNT };
struct Prof {
  std::vector<cudaEvent_t> ev;  // begin/end pairs
  std::vector<int> cls;
};
static thread_local Prof* tl_prof = nullptr;
static long long* g_tree_trace = nullptr;  // eaz_debug_set_tree_trace
struct ProfScope {
  cudaStream_t st;
  bool on;
  ProfScope(int c, cudaStream_t s) : st(s), on(tl_prof != nullptr) {
    if (!on) return;
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    tl_prof->ev.push_back(a);
    tl_prof->ev.push_back(b);
    tl_prof->cls.push_back(c);
    cudaEventRecord(a, st);
  }
  ~ProfScope() {
    if (on) cudaEventRecord(tl_prof->ev.back(), st);
  }
};

// Tree records (array of 32-byte structs, node-major): one or two 16-byte vector accesses fetch everything a
// level of the descent / backward needs, instead of one scalar access per emctx array.
// Indices are stored +1 so that an all-zero workspace is the empty tree (0 == UNVISITED / NO_PARENT).
struct __align__(16) NodeRec {
  int visits; float val, var; int pad0;       // half 0: backward operands (node_visits, node_values, node_values_epistemic_variance)
  float raw, rawvar; int parent1, action1;    // half 1: raw_values, raw_values_epistemic_variance, parents+1, action_from_parent+1
};
struct __align__(16) EdgeRec {
  int ci1, vis; float pl, rew;                // half 0: children_index+1, children_visits, children_prior_logits, children_rewards
  float val, vvar, dis; int pad1;             // half 1: children_values, children_values_epistemic_variance, children_discounts
};
struct Tree {
  int B, N, A, S;
  NodeRec* nodes;  // [N][B]
  EdgeRec* edges;  // [N][B][A]
  uint8_t* states;
  // scratch
  float *gumbel, *net_logits, *net_value, *net_ube, *reward;
  int32_t *parent, *action, *leaf;
  int32_t* cell;  // DeepSea: observation cell of the pending leaf (saves the network kernel a dependent load)
  int32_t* table;
  uint8_t* ds_seen;
  float4* ds_out;  // DeepSea, persistent search: per-cell network outputs (psearch.cuh: ds_output_table_kernel)
  uint8_t* wimg;  // tensor-path weight images (mlp_mode TENSOR)
  int2* path;     // [max_depth][B] (node, action) per level of the current descent
  int32_t* path_len;
  int32_t* tile_ctr;  // [2][tiles] completion counters of the tile-flag protocol (common.cuh)
  uint32_t* draw_ctr;  // [0] number of searches that drew their own noise on this workspace (counter-based generator), [1] its value
                       // at this search's root_init (read by finalize_kernel while it advances [0])
};

struct Layout {
  size_t off[32];
  size_t total;
  size_t zero_begin, zero_end, ones_begin, ones_end;
};

static size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

static void make_layout(int B, int N, int A, int S, int table_len, int obs_dim, size_t wimg_bytes, size_t out_table_bytes, int max_depth,
                        Layout* L) {
  const size_t nb = (size_t)N * B, nba = nb * A;
  size_t o = 0;
  int i = 0;
  auto put = [&](size_t bytes) { L->off[i++] = o; o = align_up(o + bytes); };
  L->zero_begin = o;
  put(nb * sizeof(NodeRec));   // 0 nodes
  put(nba * sizeof(EdgeRec));  // 1 edges
  put(nb * S);                 // 2 states
  L->zero_end = o;
  L->ones_begin = L->ones_end = o;
  put((size_t)B * 4);                   // 3 cell
  put(out_table_bytes);                 // 4 ds_out
  for (int k = 5; k < 14; ++k) put(0);  // (slots kept so that the scratch offsets below stay stable)
  put((size_t)B * A * 4);  // 14 gumbel
  put((size_t)B * A * 4);  // 15 net_logits
  put((size_t)B * 4);      // 16 net_value
  put((size_t)B * 4);      // 17 net_ube
  put((size_t)B * 4);      // 18 reward
  put((size_t)B * 4);      // 19 parent
  put((size_t)B * 4);      // 20 action
  put((size_t)B * 4);      // 21 leaf
  put((size_t)table_len * 4);  // 22 table
  put((size_t)obs_dim);        // 23 ds_seen
  put(wimg_bytes);             // 24 tensor weight images
  put((size_t)max_depth * B * 8);  // 25 path
  put((size_t)B * 4);              // 26 path_len
  put((size_t)2 * ceil_div(B, kTileRows) * 4);  // 27 tile counters: [tiles] tree done, [tiles] network done
  put(16);                                      // 28 draw counter of the in-kernel noise, [1] its value for the action draw
  L->total = o;
}

static Tree make_tree(void* ws, const Layout& L, int B, int N, int A, int S) {
  uint8_t* p = (uint8_t*)ws;
  Tree t;
  t.B = B; t.N = N; t.A = A; t.S = S;
  t.nodes = (NodeRec*)(p + L.off[0]);
  t.edges = (EdgeRec*)(p + L.off[1]);
  t.states = p + L.off[2];
  t.cell = (int32_t*)(p + L.off[3]);
  t.gumbel = (float*)(p + L.off[14]);
  t.net_logits = (float*)(p + L.off[15]);
  t.net_value = (float*)(p + L.off[16]);
  t.net_ube = (float*)(p + L.off[17]);
  t.reward = (float*)(p + L.off[18]);
  t.parent = (int32_t*)(p + L.off[19]);
  t.action = (int32_t*)(p + L.off[20]);
  t.leaf = (int32_t*)(p + L.off[21]);
  t.table = (int32_t*)(p + L.off[22]);
  t.ds_seen = p + L.off[23];
  t.ds_out = (float4*)(p + L.off[4]);
  t.wimg = p + L.off[24];
  t.path = (int2*)(p + L.off[25]);
  t.path_len = (int32_t*)(p + L.off[26]);
  t.tile_ctr = (int32_t*)(p + L.off[27]);
  t.draw_ctr = (uint32_t*)(p + L.off[28]);
  return t;
}

constexpr int kFlagManyTrees = 1 << 30;  // internal (set by eaz_search_gumbel): the whole batch is >= kManyTrees trees
constexpr int kManyTrees = 6144;
// Subleq transition inside the tree kernel (tree_step.cuh: subleq_expand_fused) or as its own launch: fused saves a launch boundary
// and a pass over the states per simulation, but parks a whole warp (and the tree kernel's registers) behind three interpreting
// lanes -- measured: 5 % faster at 8192 trees (C3), 7 % slower at 16384 and 35 % slower at 65536 x 128 (C5), where the dense
// 3-threads-per-env kernel wins.  The caller-visible batch decides.
constexpr int kFlagSqFused = 1 << 29;  // internal, like kFlagManyTrees
constexpr int kSqFusedMaxTrees = 8192;
static bool subleq_fused_for(int batch) {
  static const bool separate = getenv("EAZ_SUBLEQ_SEPARATE") != nullptr, fused = getenv("EAZ_SUBLEQ_FUSED") != nullptr;  // measurement knobs
  return !separate && (fused || batch <= kSqFusedMaxTrees);
}

// Search scalars, by value into the kernels.
struct SearchParams {
  int n, max_depth, max_considered;
  float gumbel_scale, discount, value_scale, maxvisit_init, epsilon;
  int two_players, rescale, mixed, flags;
  float pb_c_init, pb_c_base, temperature;  // EAZ_FLAG_PUCT (mctx muzero_policy)
  uint32_t noise_seed;
};

// ------------------------------------------------------------------ state packing
__global__ void pack_states_kernel(EnvDesc env, StateSoA s, uint8_t* __restrict__ out, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  pack_state(env, s, b, out);
}

// inverse of pack_states_kernel: compact records -> pgx.State leaves (replay-buffer decode, SURVEY 8f-3)
__global__ void unpack_states_kernel(EnvDesc env, const uint8_t* __restrict__ in, const float* __restrict__ rewards, StateSoA s, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  s.rewards[b] = rewards ? rewards[b] : 0.0f;
  if (env.kind == EAZ_ENV_DEEPSEA) {
    const uint32_t v = reinterpret_cast<const uint32_t*>(in)[b];
    s.step_count[b] = EAZ_DS_STEP(v);
    s.col[b] = EAZ_DS_COL(v);
    s.terminated[b] = (uint8_t)EAZ_DS_TERM(v);
    if (s.truncated) s.truncated[b] = (uint8_t)EAZ_DS_TRUNC(v);
    return;
  }
  const int S = env.compact_bytes, ws = env.ws;
  const uint8_t* o = in + (size_t)b * S;
  const uint16_t* h = reinterpret_cast<const uint16_t*>(o);
  for (int i = 0; i < 8; ++i) {
    s.input_after[(size_t)b * 8 + i] = h[i];
    s.output_after[(size_t)b * 8 + i] = h[8 + i];
  }
  s.step_count[b] = h[16];
  s.task[b] = o[34];
  s.terminated[b] = (o[35] & EAZ_SQ_FLAG_TERM) ? 1 : 0;
  if (s.truncated) s.truncated[b] = (o[35] & EAZ_SQ_FLAG_TRUNC) ? 1 : 0;
  s.solved[b] = (o[35] & EAZ_SQ_FLAG_SOLVED) ? 1 : 0;
  for (int i = 0; i < ws; ++i) s.memory[(size_t)b * ws + i] = o[EAZ_SQ_HDR + i];
}

// ------------------------------------------------------------------ sequential halving table (mctx seq_halving.py)
__global__ void seq_halving_table_kernel(int max_considered, int n, int32_t* __restrict__ table) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m > max_considered) return;
  int32_t* seq = table + (size_t)m * n;
  if (m <= 1) {
    for (int i = 0; i < n; ++i) seq[i] = i;
    return;
  }
  int log2max = 0;
  while ((1 << log2max) < m) log2max++;
  int visits[256];
  for (int i = 0; i < m; ++i) visits[i] = 0;
  int nc = m, len = 0;
  while (len < n) {
    int extra = max(1, n / (log2max * nc));
    for (int e = 0; e < extra && len < n; ++e) {
      for (int i = 0; i < nc && len < n; ++i) seq[len++] = visits[i];
      for (int i = 0; i < nc; ++i) visits[i] += 1;
    }
    nc = max(2, nc / 2);
  }
}

// ------------------------------------------------------------------ lane-group helpers
template <int G, int J>
struct Edge {
  int32_t ci[J], vis[J];
  float pl[J], rew[J], dis[J], val[J], vvar[J];
};

template <int G, int J>
__device__ __forceinline__ void load_edges(const Tree& t, unsigned node_slot, int gl, bool active, Edge<G, J>& e) {
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int a = gl + G * j;
    if (active && a < t.A) {
      const uint4* p = reinterpret_cast<const uint4*>(t.edges + (size_t)(node_slot * (unsigned)t.A + (unsigned)a));
      const uint4 h0 = p[0], h1 = p[1];
      e.ci[j] = (int)h0.x - 1;
      e.vis[j] = (int)h0.y;
      e.pl[j] = __uint_as_float(h0.z);
      e.rew[j] = __uint_as_float(h0.w);
      e.val[j] = __uint_as_float(h1.x);
      e.vvar[j] = __uint_as_float(h1.y);
      e.dis[j] = __uint_as_float(h1.z);
    } else {
      e.ci[j] = -1; e.vis[j] = 0;
      e.pl[j] = 0.0f; e.rew[j] = 0.0f; e.dis[j] = 0.0f; e.val[j] = 0.0f; e.vvar[j] = 0.0f;
    }
  }
}
// raw_values / raw_values_epistemic_variance of a node (second half of its record)
__device__ __forceinline__ void load_node_raw(const Tree& t, unsigned node_slot, bool active, float& raw, float& raw_var) {
  raw = 0.0f;
  raw_var = 0.0f;
  if (active) {
    const uint4 h1 = reinterpret_cast<const uint4*>(t.nodes + node_slot)[1];
    raw = __uint_as_float(h1.x);
    raw_var = __uint_as_float(h1.y);
  }
}

// softmax over the group's actions (jax.nn.softmax: exp(x - max) / sum)
template <int G, int J>
__device__ __forceinline__ void group_softmax(const float (&x)[J], const bool (&valid)[J], float (&p)[J]) {
  float m = -INFINITY;
#pragma unroll
  for (int j = 0; j < J; ++j) if (valid[j]) m = fmaxf(m, x[j]);
  m = group_max<G>(m);
  float s = 0.0f;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    p[j] = valid[j] ? eaz_exp(__fsub_rn(x[j], m)) : 0.0f;
    s = __fadd_rn(s, p[j]);
  }
  s = group_sum<G>(s);
#pragma unroll
  for (int j = 0; j < J; ++j) p[j] = __fdiv_rn(p[j], s);
}

// epistemic_qtransform_completed_by_mix_value (mctx qtransforms.py + beta; SURVEY A.6)
template <int G, int J>
__device__ __forceinline__ void qtransform(const SearchParams& sp, const Edge<G, J>& e, const bool (&valid)[J], float raw, float raw_var,
                                           float beta, bool use_beta, float (&cq)[J], int& sumN, int& maxN) {
  float q[J];
  int sn = 0, mn = 0;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    q[j] = __fadd_rn(e.rew[j], __fmul_rn(e.dis[j], e.val[j]));
    if (use_beta) {
      const float qv = __fadd_rn(0.0f, __fmul_rn(__fmul_rn(e.dis[j], e.dis[j]), e.vvar[j]));  // reward variance == 0 (context.py:149)
      q[j] = __fadd_rn(q[j], __fmul_rn(beta, __fsqrt_rn(qv)));
    }
    if (valid[j]) { sn += e.vis[j]; mn = max(mn, e.vis[j]); }
  }
  sumN = group_sum_i<G>(sn);
  maxN = group_max_i<G>(mn);
  if (use_beta && (sp.flags & EAZ_FLAG_BETA_RAW)) raw = __fadd_rn(raw, __fmul_rn(beta, __fsqrt_rn(raw_var)));
  float value = raw;
  if (sp.mixed) {  // _compute_mixed_value
    float p[J];
    group_softmax<G, J>(e.pl, valid, p);
    float sP = 0.0f;
#pragma unroll
    for (int j = 0; j < J; ++j) {
      p[j] = eaz_max(EAZ_F32_TINY, p[j]);
      sP = __fadd_rn(sP, (valid[j] && e.vis[j] > 0) ? p[j] : 0.0f);
    }
    sP = group_sum<G>(sP);
    float wq = 0.0f;
#pragma unroll
    for (int j = 0; j < J; ++j) wq = __fadd_rn(wq, (valid[j] && e.vis[j] > 0) ? __fdiv_rn(__fmul_rn(p[j], q[j]), sP) : 0.0f);
    wq = group_sum<G>(wq);
    value = __fdiv_rn(__fadd_rn(raw, __fmul_rn((float)sumN, wq)), (float)(sumN + 1));
  }
  float c[J];
#pragma unroll
  for (int j = 0; j < J; ++j) c[j] = e.vis[j] > 0 ? q[j] : value;  // _complete_qvalues (reanalyze.py:32-40)
  if (sp.rescale) {  // _rescale_qvalues
    float lo = INFINITY, hi = -INFINITY;
#pragma unroll
    for (int j = 0; j < J; ++j) if (valid[j]) { lo = fminf(lo, c[j]); hi = fmaxf(hi, c[j]); }
    lo = group_min<G>(lo);
    hi = group_max<G>(hi);
    const float den = eaz_max(__fsub_rn(hi, lo), sp.epsilon);
#pragma unroll
    for (int j = 0; j < J; ++j) c[j] = __fdiv_rn(__fsub_rn(c[j], lo), den);
  }
  const float scale = __fmul_rn(__fadd_rn(sp.maxvisit_init, (float)maxN), sp.value_scale);
#pragma unroll
  for (int j = 0; j < J; ++j) cq[j] = __fmul_rn(scale, c[j]);
}

// seq_halving.score_considered + masked_argmax
template <int G, int J>
__device__ __forceinline__ int root_argmax(const Edge<G, J>& e, const bool (&valid)[J], const float (&gum)[J], const bool (&inval)[J],
                                           const float (&cq)[J], int considered_visit, int gl) {
  float m = -INFINITY;
#pragma unroll
  for (int j = 0; j < J; ++j) if (valid[j]) m = fmaxf(m, e.pl[j]);
  m = group_max<G>(m);
  float best = -INFINITY;
  int besti = 1 << 30;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int a = gl + G * j;
    float s = -INFINITY;
    if (valid[j]) {
      const float lg = __fsub_rn(e.pl[j], m);
      s = eaz_max(-1e9f, __fadd_rn(__fadd_rn(gum[j], lg), cq[j]));
      s = __fadd_rn(s, e.vis[j] == considered_visit ? 0.0f : -INFINITY);
      if (inval[j]) s = -INFINITY;
    }
    const int ia = valid[j] ? a : (1 << 30);
    if (s > best || (s == best && ia < besti)) { best = s; besti = ia; }
  }
  return group_argmax<G>(best, besti);
}

// ---- emctx.epistemic_muzero_policy (EAZ_FLAG_PUCT): mctx muzero_action_selection + qtransform_by_parent_and_siblings
// tie-break noise stream, identical to oracle/eaz_oracle.c:orc_tie_noise
__device__ __forceinline__ float tie_noise(uint32_t seed, uint32_t b, uint32_t node, uint32_t visits, uint32_t a) {
  uint32_t h = seed + EAZ_XX_P1;
  h = xx_round(h, b);
  h = xx_round(h, node);
  h = xx_round(h, visits);
  h = xx_round(h, a);
  h ^= h >> 15; h *= EAZ_XX_P2; h ^= h >> 13; h *= EAZ_XX_P3; h ^= h >> 16;
  return __fmul_rn((float)(h >> 8), 5.9604644775390625e-08f);
}

template <int G, int J>
__device__ __forceinline__ int puct_select(const SearchParams& sp, const Edge<G, J>& e, const bool (&valid)[J], int node_visits, float node_value,
                                           float node_var, float beta, bool use_beta, unsigned b, unsigned node, const bool (&inval)[J], int gl) {
  if (use_beta && (sp.flags & EAZ_FLAG_BETA_RAW)) node_value = __fadd_rn(node_value, __fmul_rn(beta, __fsqrt_rn(node_var)));
  float q[J];
  float lo = INFINITY, hi = -INFINITY;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    q[j] = __fadd_rn(e.rew[j], __fmul_rn(e.dis[j], e.val[j]));
    if (use_beta) {
      const float qv = __fadd_rn(0.0f, __fmul_rn(__fmul_rn(e.dis[j], e.dis[j]), e.vvar[j]));
      q[j] = __fadd_rn(q[j], __fmul_rn(beta, __fsqrt_rn(qv)));
    }
    const float safe = e.vis[j] > 0 ? q[j] : node_value;
    if (valid[j]) { lo = fminf(lo, safe); hi = fmaxf(hi, safe); }
  }
  const float mn = eaz_min(node_value, group_min<G>(lo)), mx = eaz_max(node_value, group_max<G>(hi));
  const float den = eaz_max(__fsub_rn(mx, mn), sp.epsilon);
  const float nv = (float)node_visits;
  const float pb_c = __fadd_rn(sp.pb_c_init, eaz_log(__fdiv_rn(__fadd_rn(__fadd_rn(nv, sp.pb_c_base), 1.0f), sp.pb_c_base)));
  const float explore = __fmul_rn(__fsqrt_rn(nv), pb_c);
  float p[J];
  group_softmax<G, J>(e.pl, valid, p);
  float best = -INFINITY;
  int besti = 1 << 30;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int a = gl + G * j;
    float s = -INFINITY;
    if (valid[j]) {
      const float value_score = __fdiv_rn(__fsub_rn(e.vis[j] > 0 ? q[j] : mn, mn), den);
      const float policy_score = __fdiv_rn(__fmul_rn(explore, p[j]), __fadd_rn((float)e.vis[j], 1.0f));
      const float noise = __fmul_rn(1e-7f, tie_noise(sp.noise_seed, b, node, (uint32_t)node_visits, (uint32_t)a));
      s = __fadd_rn(__fadd_rn(value_score, policy_score), noise);
      if (inval[j]) s = -INFINITY;
    }
    const int ia = valid[j] ? a : (1 << 30);
    if (s > best || (s == best && ia < besti)) { best = s; besti = ia; }
  }
  return group_argmax<G>(best, besti);
}

#define EAZ_GROUP_PROLOGUE()                                               \
  const int lane = threadIdx.x & 31;                                       \
  const int gl = lane & (G - 1);                                           \
  const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;    \
  const int b = warp_global * (32 / G) + (lane / G);                       \
  const bool in_range = b < t.B;                                           \
  bool valid[J];                                                           \
  _Pragma("unroll") for (int j = 0; j < J; ++j) valid[j] = (gl + G * j) < t.A;

// In-kernel standard Gumbel noise: a counter-based stream keyed by (noise_seed, draw counter of the workspace, tree, action), with one
// more round by kSampleSalt for the noise of the action draw (EAZ_ACTION_*): u in (0, 1) with 24 bits, g = -log(-log(u))
constexpr uint32_t kSampleSalt = 0x53414D50u;
__device__ __forceinline__ float stream_gumbel(uint32_t seed, uint32_t ctr, uint32_t tree, uint32_t a, bool sample) {
  uint32_t h = seed + EAZ_XX_P1;
  h = xx_round(h, ctr);
  h = xx_round(h, tree);
  h = xx_round(h, a);
  if (sample) h = xx_round(h, kSampleSalt);
  h ^= h >> 15; h *= EAZ_XX_P2; h ^= h >> 13; h *= EAZ_XX_P3; h ^= h >> 16;
  const float u = __fmul_rn(__fadd_rn((float)(h >> 8), 0.5f), 5.9604644775390625e-08f);
  return -eaz_log(-eaz_log(u));
}

// ------------------------------------------------------------------ root initialisation (A.1 steps 1-2, A.2)
// prior_logits == NULL: the uniform root prior (EAZ_ROOT_PRIOR_UNIFORM), every logit 0 before the masking.  keep_draw_ctr: copy the
// draw counter to draw_ctr[1], where finalize_kernel reads it for the noise of the action draw while it advances draw_ctr[0].
template <int G, int J>
__global__ void __launch_bounds__(128) root_init_kernel(Tree t, SearchParams sp, const float* __restrict__ prior_logits,
                                                         const float* __restrict__ value, const float* __restrict__ var,
                                                         const float* __restrict__ gumbel, const uint8_t* __restrict__ invalid,
                                                         float* __restrict__ out_value, float* __restrict__ out_ube, int batch_offset,
                                                         int keep_draw_ctr) {
  EAZ_GROUP_PROLOGUE();
  float lg[J];
  float m = -INFINITY;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    lg[j] = (in_range && valid[j] && prior_logits) ? prior_logits[(size_t)b * t.A + gl + G * j] : 0.0f;
    if (valid[j]) m = fmaxf(m, lg[j]);
  }
  m = group_max<G>(m);
  if (!in_range) return;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    if (!valid[j]) continue;
    const int a = gl + G * j;
    const bool inv = invalid && invalid[(size_t)b * t.A + a];
    t.edges[(size_t)b * t.A + a].pl = inv ? EAZ_F32_MIN : __fsub_rn(lg[j], m);  // _mask_invalid_actions (reanalyze.py:16-29)
    // jax.random.gumbel(gumbel_rng) of mctx policies.py: pre-drawn by the caller, or (gumbel == NULL) drawn here
    const float g = gumbel ? gumbel[(size_t)b * t.A + a] : stream_gumbel(sp.noise_seed, t.draw_ctr[0], (uint32_t)(batch_offset + b), (uint32_t)a, false);
    t.gumbel[(size_t)b * t.A + a] = __fmul_rn(sp.gumbel_scale, g);
  }
  if (gl == 0) {
    NodeRec r;
    r.visits = 1; r.val = value[b]; r.var = var[b]; r.pad0 = 0;
    r.raw = r.val; r.rawvar = r.var; r.parent1 = 0; r.action1 = 0;
    t.nodes[b] = r;
    if (out_value) out_value[b] = r.val;  // selfplay.py:139-140 value_prediction / ube_prediction
    if (out_ube) out_ube[b] = r.var;
    if (keep_draw_ctr && b == 0) t.draw_ctr[1] = t.draw_ctr[0];
  }
}

}  // namespace eaz
#include "tree_step.cuh"
#include "psearch.cuh"
namespace eaz {

// ------------------------------------------------------------------ persistent search (psearch.cuh): eligibility, output table, launch
static unsigned long long* g_ps_trace = nullptr;  // eaz_debug_set_ps_trace
static bool persistent_eligible(int B, int N, int A, int flags, const EnvDesc& env, int mlp_mode, int* ncap_out) {
  static const bool disabled = getenv("EAZ_NO_PERSISTENT") != nullptr;  // measurement knob: the per-simulation launch chain instead
  static const int tile_flags = getenv("EAZ_TILE_FLAGS") ? atoi(getenv("EAZ_TILE_FLAGS")) : 0;
  if (disabled || tile_flags > 0) return false;
  if (env.kind != EAZ_ENV_DEEPSEA || mlp_mode != EAZ_MLP_TENSOR || A > ps::kG) return false;
  if (flags & EAZ_FLAG_PUCT) return false;  // PUCT selection has no staged form: DIRECT chain
  if (N > 16383) return false;              // 16-bit cached selections
  const int ncap = (N + 1) & ~1;
  int dev = 0, max_optin = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 32 ||
      cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
    return false;
  const size_t smem = ps::smem_bytes(ncap, env.size);
  if (smem > (size_t)max_optin) return false;  // trees too large for the shared-memory caches
  // At most two waves of CTAs: a CTA's chain of simulations is latency-bound, so every further wave adds a whole search time, while the
  // per-simulation launch chain fills the machine with every kernel.  Measured at DeepSea-100 x 8192 trees x 128 simulations (C4), with
  // the network still evaluated inside the kernel: two waves 3.99 ms persistent vs 4.6 - 4.9 ms chain.  Larger batches stay on the chain
  // (unmeasured beyond).
  static bool attr_set[32] = {false};  // per device (idempotent; a race only repeats the call)
  if (!attr_set[dev]) {
    if (cudaFuncSetAttribute(ps::ds_search_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin) != cudaSuccess) {
      cudaGetLastError();
      return false;
    }
    attr_set[dev] = true;
  }
  int per_sm = 0;  // co-resident CTAs per SM at this shape's shared memory
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ps::ds_search_kernel, ps::kThreads, smem) != cudaSuccess || per_sm < 1) {
    cudaGetLastError();
    return false;
  }
  static const bool any_waves = getenv("EAZ_PERSISTENT_WAVES") != nullptr;  // measurement knob: allow more CTAs than two waves
  if (!any_waves && ceil_div(B, ps::kSlots) > 2 * per_sm * sms) return false;
  if (ncap_out) *ncap_out = ncap;
  return true;
}

// bytes of the per-cell output table the persistent search reads (DeepSea, tensor mode)
static size_t ds_out_bytes(int mlp_mode, const EnvDesc& env) {
  return (mlp_mode == EAZ_MLP_TENSOR && env.kind == EAZ_ENV_DEEPSEA) ? (size_t)env.obs_dim * sizeof(float4) : 0;
}

// per-model table of the three head outputs of every DeepSea cell (after launch_deepsea_seen_table and prepare_tensor_weights)
static int launch_output_table(const Tree& t, const EnvDesc& env, const NetDesc& net, const TensorWeights& tw, int lhead, cudaStream_t st) {
  ps::TableArgs a{};
  const int heads[ps::kHeads] = {EAZ_HEAD_VALUE, EAZ_HEAD_UBE, lhead};
  for (int r = 0; r < ps::kHeads; ++r) {
    const int h = heads[r];
    a.w2img[r] = (const uint8_t*)tw.w2_ck16[h];
    a.h1[r] = (const uint8_t*)tw.h1[h];
    a.b2[r] = net.b[h][1];
    a.w3[r] = net.w[h][2];
    a.b3[r] = net.b[h][2];
    a.nout[r] = h >= EAZ_HEAD_EXPLOIT ? net.A : 1;
    a.head_id[r] = h;
  }
  a.wscale = tw.wscale;
  a.ds_seen = t.ds_seen;
  a.max_u = net.max_u;
  a.novelty_scale = net.novelty_scale;
  a.cells = env.obs_dim;
  a.out = t.ds_out;
  static bool attr_set = false;  // idempotent; a race only repeats the call
  if (!attr_set) {
    if (cudaError_t e = cudaFuncSetAttribute(ps::ds_output_table_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ps::kTableSmem);
        e != cudaSuccess)
      return cuda_fail(e, "cudaFuncSetAttribute(ds_output_table_kernel)");
    attr_set = true;
  }
  ps::ds_output_table_kernel<<<dim3(ceil_div(env.obs_dim, ps::kRows), ps::kHeads), ps::kTableThreads, ps::kTableSmem, st>>>(a);
  EAZ_CHECK_LAUNCH("ds_output_table_kernel");
  return 0;
}

static int launch_persistent(const Tree& t, const SearchParams& sp, const EnvDesc& env, const eaz_search_inputs* in, int ncap, cudaStream_t st) {
  ps::Args a{};
  a.t = t;
  a.sp = sp;
  a.env = env;
  a.beta = in->beta;
  a.invalid = in->invalid_actions;
  a.ds_out = t.ds_out;
  a.ncap = ncap;
  a.trace = g_ps_trace;
  // (cudaFuncAttributeMaxDynamicSharedMemorySize was raised to the largest eligible size by persistent_eligible)
  ps::ds_search_kernel<<<ceil_div(t.B, ps::kSlots), ps::kThreads, ps::smem_bytes(ncap, env.size), st>>>(a);
  EAZ_CHECK_LAUNCH("ds_search_kernel");
  return 0;
}

// ------------------------------------------------------------------ Subleq transition on tree states (context.py:127)
__global__ void __launch_bounds__(3 * EAZ_SQ_EPB) subleq_tree_step_kernel(Tree t, EnvDesc env) {
  __shared__ SqShared sh;
  extern __shared__ __align__(16) uint8_t sq_dyn[];  // per-(env, test) memory images + cycle-detector snapshots
  __shared__ int kind[EAZ_SQ_EPB];  // 0 absorbing, 1 terminate now, 2 execute
  __shared__ __align__(8) uint8_t hdr[EAZ_SQ_EPB][EAZ_SQ_HDR];
  const int ws = env.ws, S = t.S;
  const int e = threadIdx.x / 3, k = threadIdx.x % 3;
  const int b = blockIdx.x * EAZ_SQ_EPB + e;
  if (k == 0) {
    int kd = -1, run = 0;
    if (b < t.B) {
      const uint8_t* ps = t.states + ((size_t)t.parent[b] * t.B + b) * S;
      for (int i = 0; i < EAZ_SQ_HDR / 8; ++i) reinterpret_cast<uint2*>(hdr[e])[i] = reinterpret_cast<const uint2*>(ps)[i];
      for (int i = 0; i < S - EAZ_SQ_HDR; i += 8) *reinterpret_cast<uint2*>(&sh.base[e][i]) = *reinterpret_cast<const uint2*>(ps + EAZ_SQ_HDR + i);
      uint16_t* h = reinterpret_cast<uint16_t*>(hdr[e]);
      const int flags = hdr[e][35];
      if (flags & (EAZ_SQ_FLAG_TERM | EAZ_SQ_FLAG_TRUNC)) {
        kd = 0;
      } else {
        const int step = h[16] + 1;  // _step_count incremented before _step
        h[16] = (uint16_t)step;
        if (step >= ws - 3 || (flags & EAZ_SQ_FLAG_SOLVED)) {  // subleq.py:671-673
          kd = 1;
          hdr[e][35] = (uint8_t)(flags | EAZ_SQ_FLAG_TERM);
        } else {
          sh.base[e][step - 1] = (uint8_t)t.action[b];  // :654
          sh.trow[e] = sq_task_row(hdr[e][34]);
          kd = 2;
          run = 1;
        }
      }
    }
    kind[e] = kd;
    sh.run[e] = run;
  }
  __syncthreads();
  sq_run_tests_block(sh, sq_dyn, ws);
  if (k != 0 || b >= t.B) return;
  float reward = 0.0f;
  if (kind[e] == 2) {
    const int solved = sh.correct[e][0] & sh.correct[e][1] & sh.correct[e][2];
    const int bytes = max(sh.bytes[e][0], max(sh.bytes[e][1], sh.bytes[e][2]));
    reward = subleq_reward(env.reward_fn, solved, bytes);
    uint16_t* h = reinterpret_cast<uint16_t*>(hdr[e]);
    for (int i = 0; i < 8; ++i) {
      h[i] = (uint16_t)sh.in_after[e][i];
      h[8 + i] = (uint16_t)sh.out_after[e][i];
    }
    hdr[e][35] = (uint8_t)((hdr[e][35] & ~EAZ_SQ_FLAG_SOLVED) | (solved ? EAZ_SQ_FLAG_SOLVED : 0));
  }
  uint8_t* cs = t.states + ((size_t)t.leaf[b] * t.B + b) * S;
  for (int i = 0; i < EAZ_SQ_HDR / 8; ++i) reinterpret_cast<uint2*>(cs)[i] = reinterpret_cast<const uint2*>(hdr[e])[i];
  for (int i = 0; i < S - EAZ_SQ_HDR; i += 8) *reinterpret_cast<uint2*>(cs + EAZ_SQ_HDR + i) = *reinterpret_cast<const uint2*>(&sh.base[e][i]);
  t.reward[b] = reward;
}

// The same transition for word size 16 (C3 / C5 above kSqFusedMaxTrees): the machine runs in registers (common.cuh: subleq_simulate16), so a
// block needs neither the 264-byte program rows nor the per-test images -- 8 KB of shared memory for 64 envs instead of 38 KB for 32, and
// ten 192-thread blocks per SM instead of six 96-thread ones (the dense kernel above ran at 7-8 % of the SM's warp slots).
constexpr int kSq16Epb = 64;
__global__ void __launch_bounds__(3 * kSq16Epb) subleq16_tree_step_kernel(Tree t, EnvDesc env) {
  constexpr int kRec = EAZ_SQ_HDR + 16;  // compact state record: header + 16 memory bytes
  __shared__ __align__(8) uint8_t rec[kSq16Epb][kRec];
  __shared__ unsigned long long s_mem[kSq16Epb];
  __shared__ int kind[kSq16Epb], trow[kSq16Epb];  // kind: 0 absorbing, 1 terminate now, 2 execute
  __shared__ int correct[kSq16Epb][3], bytes_used[kSq16Epb][3];
  __shared__ int16_t in_after[kSq16Epb][8], out_after[kSq16Epb][8];
  const int e = threadIdx.x / 3, k = threadIdx.x % 3;
  const int b = blockIdx.x * kSq16Epb + e;
  if (k == 0) {
    int kd = -1;
    if (b < t.B) {
      const uint2* ps = reinterpret_cast<const uint2*>(t.states + ((size_t)t.parent[b] * t.B + b) * kRec);
#pragma unroll
      for (int i = 0; i < kRec / 8; ++i) reinterpret_cast<uint2*>(rec[e])[i] = ps[i];
      uint16_t* h = reinterpret_cast<uint16_t*>(rec[e]);
      const int flags = rec[e][35];
      if (flags & (EAZ_SQ_FLAG_TERM | EAZ_SQ_FLAG_TRUNC)) {
        kd = 0;
      } else {
        const int step = h[16] + 1;  // _step_count incremented before _step
        h[16] = (uint16_t)step;
        if (step >= 16 - 3 || (flags & EAZ_SQ_FLAG_SOLVED)) {  // subleq.py:671-673
          kd = 1;
          rec[e][35] = (uint8_t)(flags | EAZ_SQ_FLAG_TERM);
        } else {
          rec[e][EAZ_SQ_HDR + step - 1] = (uint8_t)t.action[b];  // :654
          trow[e] = sq_task_row(rec[e][34]);
          s_mem[e] = sq_pack_nibbles16(reinterpret_cast<const uint32_t*>(rec[e] + EAZ_SQ_HDR));
          kd = 2;
        }
      }
    }
    kind[e] = kd;
  }
  __syncthreads();
  if (kind[e] == 2) {  // run_tests (subleq.py:504-532): thread k interprets test case k
    SubleqSim r;
    subleq_simulate16<true>(s_mem[e], trow[e], k, r);
    correct[e][k] = r.correct;
    bytes_used[e][k] = r.bytes_used;
    if (k == 0) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        in_after[e][i] = (int16_t)r.in[i];
        out_after[e][i] = (int16_t)r.out[i];
      }
    }
  }
  __syncthreads();
  if (k != 0 || b >= t.B) return;
  float reward = 0.0f;
  if (kind[e] == 2) {
    const int solved = correct[e][0] & correct[e][1] & correct[e][2];
    const int bytes = max(bytes_used[e][0], max(bytes_used[e][1], bytes_used[e][2]));
    reward = subleq_reward(env.reward_fn, solved, bytes);
    uint16_t* h = reinterpret_cast<uint16_t*>(rec[e]);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      h[i] = (uint16_t)in_after[e][i];
      h[8 + i] = (uint16_t)out_after[e][i];
    }
    rec[e][35] = (uint8_t)((rec[e][35] & ~EAZ_SQ_FLAG_SOLVED) | (solved ? EAZ_SQ_FLAG_SOLVED : 0));
  }
  uint2* cs = reinterpret_cast<uint2*>(t.states + ((size_t)t.leaf[b] * t.B + b) * kRec);
#pragma unroll
  for (int i = 0; i < kRec / 8; ++i) cs[i] = reinterpret_cast<const uint2*>(rec[e])[i];
  t.reward[b] = reward;
}

// categorical draw as Gumbel-max (mctx policies.py: _get_logits_from_probs + _apply_temperature + categorical): the argmax over valid,
// not excluded actions of (x - max x) / max(tiny, temperature) + g with x = log(max(w, tiny)); ties go to the lowest index, and a row
// with every action excluded gets the lowest valid one
template <int G, int J>
__device__ __forceinline__ int gumbel_max_draw(const float (&w)[J], const bool (&valid)[J], const bool (&excluded)[J], const float (&g)[J],
                                               float temperature, int gl) {
  float x[J];
  float m = -INFINITY;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    x[j] = eaz_log(eaz_max(w[j], EAZ_F32_TINY));
    if (valid[j]) m = fmaxf(m, x[j]);
  }
  m = group_max<G>(m);
  const float tdiv = eaz_max(EAZ_F32_TINY, temperature);
  float best = -INFINITY;
  int besti = 1 << 30;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const float s = (valid[j] && !excluded[j]) ? __fadd_rn(__fdiv_rn(__fsub_rn(x[j], m), tdiv), g[j]) : -INFINITY;
    const int ia = valid[j] ? gl + G * j : (1 << 30);
    if (s > best || (s == best && ia < besti)) { best = s; besti = ia; }
  }
  return group_argmax<G>(best, besti);
}

// ------------------------------------------------------------------ policy output (A.1 step 4) + epistemic_summary (A.7)
struct SummaryOut {
  int32_t* action;
  float *action_weights, *value, *value_std, *visit_counts, *visit_probs, *qvalues, *qvalues_var;
};

// sampling (EAZ_ACTION_*): the played action is drawn from the visit probabilities or action_weights with the noise sample_gumbel, or
// (sample_gumbel == NULL) with the in-kernel stream at the draw counter root_init_kernel kept in draw_ctr[1]
template <int G, int J>
__global__ void __launch_bounds__(128) finalize_kernel(Tree t, SearchParams sp, const float* __restrict__ beta_in,
                                                        const uint8_t* __restrict__ invalid, SummaryOut out, int bump_draw_ctr,
                                                        int sampling, const float* __restrict__ sample_gumbel, int batch_offset) {
  EAZ_GROUP_PROLOGUE();
  const float beta = (in_range && beta_in) ? beta_in[b] : 0.0f;
  float gum[J];
  bool inval[J];
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int a = gl + G * j;
    gum[j] = (in_range && valid[j]) ? t.gumbel[(size_t)b * t.A + a] : 0.0f;
    inval[j] = (in_range && valid[j] && invalid) ? (invalid[(size_t)b * t.A + a] != 0) : false;
  }
  Edge<G, J> e;
  load_edges<G, J>(t, (unsigned)(in_range ? b : 0), gl, in_range, e);
  float raw, raw_var;
  load_node_raw(t, (unsigned)(in_range ? b : 0), in_range, raw, raw_var);
  float cq[J];
  int sumN, maxN;
  qtransform<G, J>(sp, e, valid, raw, raw_var, beta, (sp.flags & EAZ_FLAG_BETA_FINAL) != 0, cq, sumN, maxN);
  int act;
  float x[J], p[J];
  if (sp.flags & EAZ_FLAG_PUCT) {
    // mctx policies.muzero_policy: action_weights = visit_probs; action ~ categorical(log(visit_probs) / temperature) = Gumbel-max
    bool none[J];
#pragma unroll
    for (int j = 0; j < J; ++j) {
      p[j] = sumN > 0 ? __fdiv_rn((float)e.vis[j], eaz_max((float)sumN, 1.0f)) : __fdiv_rn(1.0f, (float)t.A);
      none[j] = false;
    }
    act = gumbel_max_draw<G, J>(p, valid, none, gum, sp.temperature, gl);
  } else {
    act = root_argmax<G, J>(e, valid, gum, inval, cq, maxN, gl);  // considered_visit = max visit count
    // action_weights = softmax(mask_invalid(root_logits + completed_q))
    float m = -INFINITY;
#pragma unroll
    for (int j = 0; j < J; ++j) {
      x[j] = __fadd_rn(e.pl[j], cq[j]);
      if (valid[j]) m = fmaxf(m, x[j]);
    }
    m = group_max<G>(m);
#pragma unroll
    for (int j = 0; j < J; ++j) x[j] = inval[j] ? EAZ_F32_MIN : __fsub_rn(x[j], m);
    group_softmax<G, J>(x, valid, p);
    if (sampling) {  // selfplay.py:125-134: the played action ~ visit counts / improved policy instead of the policy's action
      float w[J], sg[J];
#pragma unroll
      for (int j = 0; j < J; ++j) {
        const int a = gl + G * j;
        w[j] = sampling == EAZ_ACTION_IMPROVED ? p[j]
                                               : (sumN > 0 ? __fdiv_rn((float)e.vis[j], eaz_max((float)sumN, 1.0f)) : __fdiv_rn(1.0f, (float)t.A));
        sg[j] = !(in_range && valid[j]) ? 0.0f
                : sample_gumbel        ? sample_gumbel[(size_t)b * t.A + a]
                                       : stream_gumbel(sp.noise_seed, t.draw_ctr[1], (uint32_t)(batch_offset + b), (uint32_t)a, true);
      }
      act = gumbel_max_draw<G, J>(w, valid, inval, sg, sp.temperature, gl);
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && bump_draw_ctr) t.draw_ctr[0] += 1u;  // (root_init of this search has long finished)
  if (!in_range) return;
  if (gl == 0) {
    out.action[b] = act;
    if (out.value) out.value[b] = t.nodes[b].val;
    if (out.value_std) out.value_std[b] = __fsqrt_rn(t.nodes[b].var);
  }
#pragma unroll
  for (int j = 0; j < J; ++j) {
    if (!valid[j]) continue;
    const size_t o = (size_t)b * t.A + gl + G * j;
    const float vc = (float)e.vis[j];
    if (out.action_weights) out.action_weights[o] = p[j];
    if (out.visit_counts) out.visit_counts[o] = vc;
    if (out.visit_probs) out.visit_probs[o] = sumN > 0 ? __fdiv_rn(vc, eaz_max((float)sumN, 1.0f)) : __fdiv_rn(1.0f, (float)t.A);
    if (out.qvalues) out.qvalues[o] = __fadd_rn(e.rew[j], __fmul_rn(e.dis[j], e.val[j]));
    if (out.qvalues_var) out.qvalues_var[o] = __fadd_rn(0.0f, __fmul_rn(__fmul_rn(e.dis[j], e.dis[j]), e.vvar[j]));
  }
}

// ------------------------------------------------------------------ reanalyze targets (reanalyze.py:86-129)
struct ReanalyzeArgs {
  const int32_t* action;
  const float *qvalues, *qvar, *visit_counts, *value, *value_std, *next_value, *next_rewards;
  const uint8_t *next_terminated, *terminated, *invalid;
  float *value_target, *ube_target, *policy_target;
};

template <int G, int J>
__global__ void __launch_bounds__(128) reanalyze_targets_kernel(eaz_reanalyze_config cfg, int B, int A, ReanalyzeArgs r) {
  const int lane = threadIdx.x & 31;
  const int gl = lane & (G - 1);
  const int b = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * (32 / G) + (lane / G);
  const bool in_range = b < B;
  const size_t row = (size_t)(in_range ? b : 0) * A;
  bool valid[J];
  float q[J], qv[J], x[J], p[J];
  const int act = in_range ? r.action[b] : 0;
  const float vfill = in_range ? __fadd_rn(r.value[b], __fmul_rn(cfg.exploration_beta, r.value_std[b])) : 0.0f;  // :116
  float qmax = -INFINITY, m = -INFINITY, q_act = 0.0f, qv_act = 0.0f;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int a = gl + G * j;
    valid[j] = a < A;
    q[j] = (in_range && valid[j]) ? r.qvalues[row + a] : 0.0f;
    qv[j] = (in_range && valid[j]) ? r.qvar[row + a] : 0.0f;
    const float vc = (in_range && valid[j]) ? r.visit_counts[row + a] : 0.0f;
    const float qs = __fadd_rn(q[j], __fmul_rn(cfg.exploration_beta, __fsqrt_rn(qv[j])));  // :114
    x[j] = vc > 0.0f ? qs : vfill;                                                            // complete_qs :32-40
    if (valid[j]) {
      qmax = fmaxf(qmax, qv[j]);
      m = fmaxf(m, x[j]);
    }
  }
  qmax = group_max<G>(qmax);
  m = group_max<G>(m);
  {  // broadcast the chosen action's entries from their owner (lane act % G, slot act / G) -- bit-exact, unlike a sum with zeros
    float qa = 0.0f, qva = 0.0f;
#pragma unroll
    for (int j = 0; j < J; ++j)
      if (j == act / G) { qa = q[j]; qva = qv[j]; }
    const int owner = (lane & ~(G - 1)) + (act & (G - 1));
    q_act = __shfl_sync(0xffffffffu, qa, owner);
    qv_act = __shfl_sync(0xffffffffu, qva, owner);
  }
#pragma unroll
  for (int j = 0; j < J; ++j) {  // mask_invalid_actions :16-29, then the temperature :121
    const bool inv = in_range && valid[j] && r.invalid && r.invalid[row + gl + G * j] != 0;
    x[j] = __fmul_rn(inv ? EAZ_F32_MIN : __fsub_rn(x[j], m), cfg.exploration_policy_target_temperature);
  }
  group_softmax<G, J>(x, valid, p);  // :120
  if (!in_range) return;
#pragma unroll
  for (int j = 0; j < J; ++j)
    if (valid[j]) r.policy_target[row + gl + G * j] = p[j];
  if (gl == 0) {
    const float not_term_next = r.next_terminated[b] ? 0.0f : 1.0f, not_term = r.terminated[b] ? 0.0f : 1.0f;
    const float from_td = __fadd_rn(r.next_rewards[b], __fmul_rn(__fmul_rn(cfg.discount, r.next_value[b]), not_term_next));  // :94-95
    const float vt = eaz_max(q_act, from_td);                                                                                 // :101
    const float ut = cfg.exploration_ube_target ? qmax : qv_act;                                                              // :102-106
    r.value_target[b] = __fmul_rn(vt, not_term);                                                                              // :109-110
    r.ube_target[b] = __fmul_rn(ut, not_term);
  }
}

// ------------------------------------------------------------------ optional tree export: node-major -> emctx [B,N,...]
struct TreeOut {
  int32_t *node_visits, *parents, *action_from_parent, *children_index, *children_visits;
  float *raw_values, *node_values, *raw_var, *node_var;
  float *prior, *rewards, *discounts, *values, *rewards_var, *values_var;
  uint8_t* embeddings;
};

__global__ void export_tree_kernel(Tree t, TreeOut o) {
  const size_t nb = (size_t)t.N * t.B, nba = nb * t.A;
  const size_t stride = (size_t)gridDim.x * blockDim.x, tid0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (size_t i = tid0; i < nb; i += stride) {  // i indexes the OUTPUT [B][N]
    const size_t b = i / t.N, n = i % t.N, s = n * t.B + b;
    const NodeRec r = t.nodes[s];
    if (o.node_visits) o.node_visits[i] = r.visits;
    if (o.raw_values) o.raw_values[i] = r.raw;
    if (o.node_values) o.node_values[i] = r.val;
    if (o.raw_var) o.raw_var[i] = r.rawvar;
    if (o.node_var) o.node_var[i] = r.var;
    if (o.parents) o.parents[i] = r.parent1 - 1;
    if (o.action_from_parent) o.action_from_parent[i] = r.action1 - 1;
    if (o.embeddings) {
      const bool live = r.visits > 0;
      for (int k = 0; k < t.S; ++k) o.embeddings[i * t.S + k] = live ? t.states[s * t.S + k] : 0;
    }
  }
  for (size_t i = tid0; i < nba; i += stride) {  // output [B][N][A]
    const size_t a = i % t.A, bn = i / t.A, b = bn / t.N, n = bn % t.N, s = (n * t.B + b) * t.A + a;
    const EdgeRec e = t.edges[s];
    if (o.children_index) o.children_index[i] = e.ci1 - 1;
    if (o.children_visits) o.children_visits[i] = e.vis;
    if (o.prior) o.prior[i] = e.pl;
    if (o.rewards) o.rewards[i] = e.rew;
    if (o.discounts) o.discounts[i] = e.dis;
    if (o.values) o.values[i] = e.val;
    if (o.rewards_var) o.rewards_var[i] = 0.0f;  // context.py:149
    if (o.values_var) o.values_var[i] = e.vvar;
  }
}

// ------------------------------------------------------------------ host side
template <int G, int J>
static int run_search(const Tree& t, const SearchParams& sp, const EnvDesc& env, const NetDesc& net, const eaz_search_inputs* in,
                      const SummaryOut& so, int mlp_mode, int exploration, const TensorWeights* tw, float* root_out_value, float* root_out_ube,
                      int batch_offset, int root_prior, int sampling, cudaStream_t st) {
  const int envs_per_block = 4 * (32 / G);
  const int grid = ceil_div(t.B, envs_per_block);
  const int lhead = exploration ? EAZ_HEAD_EXPLORE : EAZ_HEAD_EXPLOIT;  // context.py:132
  const int mask = (1 << EAZ_HEAD_VALUE) | (1 << EAZ_HEAD_UBE) | (1 << lhead);
  MlpSource src{nullptr, t.states, t.leaf, env.kind == EAZ_ENV_DEEPSEA ? t.ds_seen : nullptr, env.kind == EAZ_ENV_DEEPSEA ? t.cell : nullptr};
  src.many_trees = (sp.flags & kFlagManyTrees) ? 1 : 0;
  MlpOutputs mo{{nullptr, nullptr}, t.net_value, t.net_ube, nullptr};
  mo.logits[lhead - EAZ_HEAD_EXPLOIT] = t.net_logits;
  const float *root_logits = in->prior_logits, *root_value = in->value, *root_var = in->value_epistemic_variance;
  // Tile flags (common.cuh) between the tree kernel and the one-hot network kernel: each 128-tree tile hands over to its 3
  // head CTAs (and back) as soon as IT is done, instead of every kernel waiting for the whole previous grid.  Measured on
  // B200 at C2 (profiles/r1_summary.md section 9): 1.435 ms / step with flags both ways vs 1.453 ms with grid-wide PDL waits --
  // inside the run-to-run noise, the fence + poll hand-over costs what the PDL release does.  OFF by default; EAZ_TILE_FLAGS=1
  // (tree -> network only) or 2 (both ways) enables the protocol for experiments (tests/test_gpu_parity.py runs mode 2).
  static const int flag_mode = getenv("EAZ_TILE_FLAGS") ? atoi(getenv("EAZ_TILE_FLAGS")) : 0;
  const bool flags = flag_mode > 0 && mlp_mode == EAZ_MLP_TENSOR && env.kind == EAZ_ENV_DEEPSEA && t.A <= 4 && tl_prof == nullptr;
  const int tiles = ceil_div(t.B, kTileRows), nheads = 3;
  int* tile_done = flags ? t.tile_ctr : nullptr;
  int* mlp_done = flags ? t.tile_ctr + tiles : nullptr;
  int mlp_launches = 0;
  if (flags) {
    if (cudaError_t me = cudaMemsetAsync(t.tile_ctr, 0, (size_t)2 * tiles * sizeof(int), st); me != cudaSuccess) return cuda_fail(me, "tile counter memset");
    src.tile_done = tile_done;
    src.mlp_done = mlp_done;
  }
  if (!root_logits) {  // fused root: forward.apply on the root states (node 0 = the first B compact states), selfplay.py:89
    ProfScope ps(CLS_MLP, st);
    MlpSource rsrc{nullptr, t.states, nullptr, src.ds_seen, nullptr, nullptr, 0, mlp_done};
    ++mlp_launches;
    if (int rc = launch_mlp(net, env, rsrc, t.B, mask, mo, mlp_mode, st, tw)) return rc;
    root_logits = t.net_logits;
    root_value = t.net_value;
    root_var = t.net_ube;
  }
  // the draw counter advances once per search that draws noise itself: root noise (gumbel == NULL) and / or the noise of the action draw
  const bool draw_sample = sampling != EAZ_ACTION_SEARCH && !in->sample_gumbel;
  const int bump_draw_ctr = (int)(in->gumbel == nullptr || draw_sample);
  {
    ProfScope ps(CLS_INIT, st);
    root_init_kernel<G, J><<<grid, 128, 0, st>>>(t, sp, root_prior == EAZ_ROOT_PRIOR_UNIFORM ? nullptr : root_logits, root_value, root_var, in->gumbel,
                                                  in->invalid_actions, root_out_value, root_out_ube, batch_offset, (int)draw_sample);
  }
  EAZ_CHECK_LAUNCH("root_init_kernel");
  if constexpr (G == ps::kG && J == 1) {
    int ncap = 0;
    if (!flags && tw && tw->w2_ck16[0] && persistent_eligible(t.B, t.N, t.A, sp.flags, env, mlp_mode, &ncap)) {  // ONE launch runs all sp.n simulations
      {
        ProfScope ps_scope(CLS_SELECT, st);
        if (int rc = launch_persistent(t, sp, env, in, ncap, st)) return rc;
      }
      ProfScope pf(CLS_FINAL, st);
      finalize_kernel<G, J><<<grid, 128, 0, st>>>(t, sp, in->beta, in->invalid_actions, so, bump_draw_ctr, sampling, in->sample_gumbel, batch_offset);
      EAZ_CHECK_LAUNCH("finalize_kernel");
      return 0;
    }
  }
  // staging area of tree_step_kernel (tree_step.cuh): per warp, sized for the cached selections + states of all N nodes
  static const bool no_staging = getenv("EAZ_NO_STAGING") != nullptr;  // measurement knob: force the DIRECT path
  const int chase_cap = (J == 1 && t.N <= 512 && !no_staging) ? ((t.N + 2 + 7) & ~7) : 0;
  const size_t stage_bytes = chase_cap ? (size_t)4 * Stage<G>::words(chase_cap) * sizeof(uint32_t) : 0;
  static const bool one_per_warp = getenv("EAZ_ONE_TREE_PER_WARP") != nullptr;  // measurement knob
  bool two_per_warp = false;
  size_t stage2_bytes = 0;
  if constexpr (G <= 4 && J == 1) {
    stage2_bytes = (size_t)8 * Stage2<G>::words(chase_cap) * sizeof(uint32_t);
    // issue-bound regime only (measured: C2 = 4096 trees is 3 % faster with one tree per warp, 8192 trees 4 % and 65536 trees 12 %
    // faster with two): the caller-visible batch decides, not the sub-batch of one stream
    two_per_warp = !one_per_warp && (sp.flags & kFlagManyTrees) && chase_cap > 0 && stage2_bytes <= 48 * 1024 && !flags &&
                   !(sp.flags & EAZ_FLAG_PUCT);  // (the PUCT selection is staged in the one-tree-per-warp kernel)
  }
  // Subleq: the transition of the pending expansion runs inside the tree kernel (tree_step.cuh: subleq_expand_fused) for batches up to
  // kSqFusedMaxTrees, as the separate subleq_tree_step_kernel launch above that
  const bool sq_fused = env.kind == EAZ_ENV_SUBLEQ && (sp.flags & kFlagSqFused);
  const size_t sq_bytes = sq_fused ? (size_t)4 * sq_warp_scratch_bytes(env.ws) : 0;
  for (int sim = 0; sim <= sp.n; ++sim) {
    {  // backward of simulation sim-1 fused with the descent of simulation sim
      ProfScope ps(sim < sp.n ? CLS_SELECT : CLS_EXPAND, st);
      cudaError_t le;
      if constexpr (G <= 4 && J == 1) {
        if (two_per_warp)  // 16 lanes per tree (tree_step.cuh: tree_step2_kernel)
          le = launch_pdl(tree_step2_kernel<G>, dim3(ceil_div(t.B, 8)), dim3(128), stage2_bytes, st, t, sp, env, sim, (int)(sim > 0), (int)(sim < sp.n),
                          in->beta, in->invalid_actions, g_timeline, g_tree_trace, chase_cap);
      }
      if (!two_per_warp)
      le = launch_pdl(tree_step_kernel<G, J>, dim3(ceil_div(t.B, 4)), dim3(128), stage_bytes + sq_bytes, st,  // one warp per tree
                                  t, sp, env, sim, (int)(sim > 0), (int)(sim < sp.n), in->beta, in->invalid_actions, g_timeline, g_tree_trace,
                                  chase_cap, tile_done, (const int*)mlp_done, (sim > 0 && flag_mode > 1) ? nheads * mlp_launches : 0, (int)sq_fused);
      if (le != cudaSuccess) return cuda_fail(le, "tree_step_kernel launch");
    }
    EAZ_CHECK_LAUNCH("tree_step_kernel");
    if (sim == sp.n) break;
    if (env.kind == EAZ_ENV_SUBLEQ && !sq_fused) {
      ProfScope ps(CLS_ENV, st);
      static const bool generic_sq = getenv("EAZ_SUBLEQ_GENERIC") != nullptr;  // measurement knob: the any-word-size kernel for ws = 16 too
      if (env.ws == 16 && t.S == EAZ_SQ_HDR + 16 && !generic_sq) {
        subleq16_tree_step_kernel<<<ceil_div(t.B, kSq16Epb), 3 * kSq16Epb, 0, st>>>(t, env);
      } else {
        size_t dyn = 0;
        if (cudaError_t e = sq_prepare_launch(subleq_tree_step_kernel, env.ws, &dyn); e != cudaSuccess) return cuda_fail(e, "subleq_tree_step_kernel attribute");
        subleq_tree_step_kernel<<<ceil_div(t.B, EAZ_SQ_EPB), 3 * EAZ_SQ_EPB, dyn, st>>>(t, env);
      }
      EAZ_CHECK_LAUNCH("subleq_tree_step_kernel");
    }
    {
      ProfScope ps(CLS_MLP, st);
      src.tree_epoch = flags ? sim + 1 : 0;  // tree launches so far
      ++mlp_launches;
      if (int rc = launch_mlp(net, env, src, t.B, mask, mo, mlp_mode, st, tw)) return rc;
    }
  }
  {
    ProfScope ps(CLS_FINAL, st);
    finalize_kernel<G, J><<<grid, 128, 0, st>>>(t, sp, in->beta, in->invalid_actions, so, bump_draw_ctr, sampling, in->sample_gumbel, batch_offset);
  }
  EAZ_CHECK_LAUNCH("finalize_kernel");
  return 0;
}

static size_t wimg_bytes_for(int mlp_mode, const EnvDesc& env) {
  if (mlp_mode != EAZ_MLP_TENSOR) return 0;
  NetDesc nd{};
  nd.D = env.obs_dim;
  nd.H = EAZ_FC_HIDDEN_MAX;
  nd.A = env.num_actions;
  return tensor_weights_bytes(nd, env);
}

static int check_search(const eaz_search_config* cfg, const eaz_search_inputs* in, const eaz_search_outputs* out, EnvDesc* env, NetDesc* net) {
  EAZ_CHECK_ARG(cfg && in && out, "search: NULL config / inputs / outputs");
  EAZ_CHECK_ARG(cfg->batch >= 1, "batch must be >= 1");
  EAZ_CHECK_ARG(cfg->num_simulations >= 1 && cfg->num_simulations <= 4094, "num_simulations %d outside [1,4094]", cfg->num_simulations);
  EAZ_CHECK_ARG(cfg->max_num_considered_actions >= 1 && cfg->max_num_considered_actions <= 256, "max_num_considered_actions outside [1,256]");
  EAZ_CHECK_ARG(cfg->max_depth >= 0, "max_depth must be >= 0 (0 = None)");
  if (int rc = make_env_desc(in->env, env)) return rc;
  if (int rc = make_net_desc(in->net, env, net)) return rc;
  EAZ_CHECK_ARG(in->embedding != nullptr, "search inputs: embedding must be non-NULL");
  const bool fused_root = !in->prior_logits && !in->value && !in->value_epistemic_variance;
  EAZ_CHECK_ARG(fused_root || (in->prior_logits && in->value && in->value_epistemic_variance),
                "search inputs: prior_logits / value / value_epistemic_variance must be all non-NULL, or all NULL (fused root)");
  EAZ_CHECK_ARG(out->action != nullptr, "search outputs: action must be non-NULL");
  EAZ_CHECK_ARG(cfg->root_prior == EAZ_ROOT_PRIOR_GIVEN || cfg->root_prior == EAZ_ROOT_PRIOR_UNIFORM, "root_prior %d is not an EAZ_ROOT_PRIOR_*",
                cfg->root_prior);
  EAZ_CHECK_ARG(cfg->action_sampling >= EAZ_ACTION_SEARCH && cfg->action_sampling <= EAZ_ACTION_IMPROVED, "action_sampling %d is not an EAZ_ACTION_*",
                cfg->action_sampling);
  EAZ_CHECK_ARG(!(cfg->flags & EAZ_FLAG_PUCT) || (cfg->root_prior == EAZ_ROOT_PRIOR_GIVEN && cfg->action_sampling == EAZ_ACTION_SEARCH),
                "root_prior / action_sampling are options of the Gumbel policy: not with EAZ_FLAG_PUCT");
  EAZ_CHECK_ARG(cfg->action_sampling == EAZ_ACTION_SEARCH || (isfinite(cfg->temperature) && cfg->temperature > 0.0f),
                "action_sampling needs a finite temperature > 0 (got %g)", (double)cfg->temperature);
  if ((size_t)(cfg->num_simulations + 1) * cfg->batch * env->num_actions >= ((size_t)1 << 31)) {
    set_error("tree of %d nodes x %d envs x %d actions exceeds 2^31 edges: shard the batch", cfg->num_simulations + 1, cfg->batch, env->num_actions);
    return EAZ_ERR_UNSUPPORTED;
  }
  return 0;
}

}  // namespace eaz

using namespace eaz;

extern "C" {

int eaz_env_compact(const eaz_env* env, const eaz_state* state, uint8_t* out, int32_t B, void* stream) {
  EnvDesc d;
  if (int rc = make_env_desc(env, &d)) return rc;
  EAZ_CHECK_ARG(state && out && B >= 0, "eaz_env_compact: bad arguments");
  if (B == 0) return 0;
  pack_states_kernel<<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(d, soa_of(state), out, B);
  EAZ_CHECK_LAUNCH("pack_states_kernel");
  return 0;
}

int eaz_env_uncompact(const eaz_env* env, const uint8_t* compact, const float* rewards, eaz_state* out, int32_t B, void* stream) {
  EnvDesc d;
  if (int rc = make_env_desc(env, &d)) return rc;
  EAZ_CHECK_ARG(compact && out && B >= 0, "eaz_env_uncompact: bad arguments");
  EAZ_CHECK_ARG(out->step_count && out->rewards && out->terminated, "eaz_env_uncompact: step_count / rewards / terminated must be non-NULL");
  if (d.kind == EAZ_ENV_DEEPSEA) EAZ_CHECK_ARG(out->col != nullptr, "eaz_env_uncompact: col is NULL");
  else EAZ_CHECK_ARG(out->memory && out->task && out->solved && out->input_after && out->output_after, "eaz_env_uncompact: NULL Subleq leaf");
  if (B == 0) return 0;
  unpack_states_kernel<<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(d, compact, rewards, soa_of(out), B);
  EAZ_CHECK_LAUNCH("unpack_states_kernel");
  if (out->observation) return eaz_env_observe(env, out, out->observation, B, stream);
  return 0;
}

int eaz_mlp_forward_states(const eaz_fc_params* net, const eaz_env* env, const eaz_state* state, int32_t B, float* exploit_logits,
                           float* explore_logits, float* value, float* ube, float* novelty, void* workspace, size_t workspace_bytes,
                           void* stream) {
  EnvDesc ed;
  if (int rc = make_env_desc(env, &ed)) return rc;
  NetDesc nd;
  if (int rc = make_net_desc(net, &ed, &nd)) return rc;
  EAZ_CHECK_ARG(state && B >= 0, "eaz_mlp_forward_states: bad arguments");
  if (!workspace || workspace_bytes < (size_t)B * ed.compact_bytes || ((uintptr_t)workspace & 15)) {
    set_error("eaz_mlp_forward_states: workspace must be >= B*compact_bytes = %zu bytes, 16-byte aligned", (size_t)B * ed.compact_bytes);
    return EAZ_ERR_WORKSPACE;
  }
  if (B == 0) return 0;
  if (int rc = eaz_env_compact(env, state, (uint8_t*)workspace, B, stream)) return rc;
  MlpSource src{nullptr, (const uint8_t*)workspace, nullptr, nullptr, nullptr};
  MlpOutputs out{{exploit_logits, explore_logits}, value, ube, novelty};
  int mask = 0;
  if (value) mask |= 1 << EAZ_HEAD_VALUE;
  if (ube || novelty) mask |= 1 << EAZ_HEAD_UBE;
  if (exploit_logits) mask |= 1 << EAZ_HEAD_EXPLOIT;
  if (explore_logits) mask |= 1 << EAZ_HEAD_EXPLORE;
  return launch_mlp(nd, ed, src, B, mask, out, EAZ_MLP_EXACT, (cudaStream_t)stream);
}

static size_t layout_bytes(const eaz_search_config* cfg, const EnvDesc& d, int batch) {
  Layout L;
  make_layout(batch, cfg->num_simulations + 1, d.num_actions, d.compact_bytes, (cfg->max_num_considered_actions + 1) * cfg->num_simulations,
              d.obs_dim, wimg_bytes_for(cfg->mlp_mode, d), ds_out_bytes(cfg->mlp_mode, d), cfg->max_depth > 0 ? cfg->max_depth : cfg->num_simulations, &L);
  return L.total;
}
// EAZ_FLAG_STREAMS(k): the batch is cut into up to k sub-batches of whole 128-tree tiles; returns their sizes (count in *parts)
static void sub_batches(const eaz_search_config* cfg, int* sizes, int* parts) {
  int k = (cfg->flags >> EAZ_FLAG_STREAMS_SHIFT) & 0xF;
  if (k > 8) k = 8;
  const int tiles = ceil_div(cfg->batch, kTileRows);
  if (k < 1) k = 1;
  if (k > tiles) k = tiles;
  const int per = ceil_div(tiles, k) * kTileRows;
  int left = cfg->batch, p = 0;
  while (left > 0) {
    sizes[p] = left < per ? left : per;
    left -= sizes[p++];
  }
  *parts = p;
}

size_t eaz_search_workspace_bytes(const eaz_search_config* cfg, const eaz_env* env) {
  EnvDesc d;
  if (!cfg || make_env_desc(env, &d) || cfg->batch < 1 || cfg->num_simulations < 1) return 0;
  int sizes[8], parts;
  sub_batches(cfg, sizes, &parts);
  size_t total = 0;
  for (int p = 0; p < parts; ++p) total += layout_bytes(cfg, d, sizes[p]);  // every sub-batch owns a complete layout
  const size_t whole = layout_bytes(cfg, d, cfg->batch);                    // (the profiled variant runs unsplit)
  return total > whole ? total : whole;
}

int32_t eaz_search_num_launches(const eaz_search_config* cfg, const eaz_env* env) {
  EnvDesc d;
  if (!cfg || make_env_desc(env, &d)) return -1;
  const int per_sim = 1 + ((d.kind == EAZ_ENV_SUBLEQ && !subleq_fused_for(cfg->batch)) ? 1 : 0) + mlp_num_launches(cfg->mlp_mode);
  const bool build_tables = (cfg->flags & EAZ_FLAG_REUSE_PREPARED) == 0;
  const int prep = (cfg->mlp_mode == EAZ_MLP_TENSOR ? 3 * (d.kind == EAZ_ENV_DEEPSEA ? 4 : 3) : 0) + 1 + (d.kind == EAZ_ENV_DEEPSEA ? 1 : 0);  // weight images, seq-halving + seen tables
  // 1 memset + pack + root init + [tables] + per simulation + last tree step + finalize  (+1 network launch with a fused root)
  int sizes[8], parts = 1;
  if (cfg->batch >= 1) sub_batches(cfg, sizes, &parts);  // EAZ_FLAG_STREAMS: every sub-batch launches its own sequence
  if (cfg->batch >= 1 && persistent_eligible(cfg->batch, cfg->num_simulations + 1, d.num_actions, cfg->flags, d, cfg->mlp_mode, nullptr))
    return 1 + 2 + (build_tables ? prep + 1 : 0) + 1 + 1;  // memset + pack + root init + [tables + output table] + ONE persistent kernel + finalize (+1 with a fused root)
  return parts * (1 + 2 + (build_tables ? prep : 0) + per_sim * cfg->num_simulations + 1 + 1);
}

// one search over the whole batch of `cfg` on one stream
static int search_one(const eaz_search_config* cfg, const eaz_search_inputs* in, eaz_search_outputs* out, void* workspace,
                      size_t workspace_bytes, void* stream, int batch_offset = 0) {
  EnvDesc env;
  NetDesc net;
  if (int rc = check_search(cfg, in, out, &env, &net)) return rc;
  const int B = cfg->batch, n = cfg->num_simulations, N = n + 1, A = env.num_actions, S = env.compact_bytes;
  Layout L;
  make_layout(B, N, A, S, (cfg->max_num_considered_actions + 1) * n, env.obs_dim, wimg_bytes_for(cfg->mlp_mode, env), ds_out_bytes(cfg->mlp_mode, env),
              cfg->max_depth > 0 ? cfg->max_depth : n, &L);
  if (!workspace || workspace_bytes < L.total || ((uintptr_t)workspace & 255)) {
    set_error("search workspace must be >= %zu bytes and 256-byte aligned (got %zu)", L.total, workspace_bytes);
    return EAZ_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  Tree t = make_tree(workspace, L, B, N, A, S);
  SearchParams sp{n, cfg->max_depth > 0 ? cfg->max_depth : n, cfg->max_num_considered_actions, cfg->gumbel_scale, cfg->discount,
                  cfg->value_scale, cfg->maxvisit_init, cfg->epsilon, cfg->two_players_game, cfg->rescale_values, cfg->use_mixed_value,
                  cfg->flags, cfg->pb_c_init, cfg->pb_c_base, cfg->temperature, cfg->noise_seed};
  TensorWeights tw{};
  {
  ProfScope init_scope(CLS_INIT, st);  // (a stack object: closed on every return path)
  cudaError_t e = cudaMemsetAsync((uint8_t*)workspace + L.zero_begin, 0, L.zero_end - L.zero_begin, st);
  if (e != cudaSuccess) return cuda_fail(e, "search memset");
  const bool build_tables = (cfg->flags & EAZ_FLAG_REUSE_PREPARED) == 0;  // parameter-derived tables: once per model, not per search
  if (build_tables) {
    seq_halving_table_kernel<<<ceil_div(cfg->max_num_considered_actions + 1, 32), 32, 0, st>>>(cfg->max_num_considered_actions, n, t.table);
    EAZ_CHECK_LAUNCH("seq_halving_table_kernel");
  }
  if (int rc = eaz_env_compact(in->env, in->embedding, t.states, B, stream)) return rc;  // node 0 = roots
  if (env.kind == EAZ_ENV_DEEPSEA && build_tables)
    if (int rc = launch_deepsea_seen_table(net, env, t.ds_seen, st)) return rc;
  if (cfg->mlp_mode == EAZ_MLP_TENSOR) {
    const int lhead = cfg->exploration ? EAZ_HEAD_EXPLORE : EAZ_HEAD_EXPLOIT;
    if (int rc = prepare_tensor_weights(net, env, (1 << EAZ_HEAD_VALUE) | (1 << EAZ_HEAD_UBE) | (1 << lhead), t.wimg, &tw, st, build_tables)) return rc;
    if (build_tables && persistent_eligible(B, N, A, cfg->flags, env, cfg->mlp_mode, nullptr))
      if (int rc = launch_output_table(t, env, net, tw, lhead, st)) return rc;
  }
  }

  SummaryOut so{out->action, out->action_weights, out->value, out->value_epistemic_std, out->visit_counts, out->visit_probs,
                out->qvalues, out->qvalues_epistemic_variance};
  int rc;
#define EAZ_RUN(G, J) rc = run_search<G, J>(t, sp, env, net, in, so, cfg->mlp_mode, cfg->exploration, cfg->mlp_mode == EAZ_MLP_TENSOR ? &tw : nullptr, out->root_value, out->root_ube, batch_offset, cfg->root_prior, cfg->action_sampling, st)
  if (A <= 2) EAZ_RUN(2, 1);
  else if (A <= 4) EAZ_RUN(4, 1);
  else if (A <= 8) EAZ_RUN(8, 1);
  else if (A <= 16) EAZ_RUN(16, 1);
  else if (A <= 32) EAZ_RUN(32, 1);
  else if (A <= 64) EAZ_RUN(32, 2);
  else if (A <= 128) EAZ_RUN(32, 4);
  else EAZ_RUN(32, 8);
#undef EAZ_RUN
  if (rc) return rc;

  const bool want_tree = out->node_visits || out->raw_values || out->node_values || out->raw_values_epistemic_variance ||
                         out->node_values_epistemic_variance || out->parents || out->action_from_parent || out->children_index ||
                         out->children_prior_logits || out->children_visits || out->children_rewards || out->children_discounts ||
                         out->children_values || out->children_rewards_epistemic_variance || out->children_values_epistemic_variance ||
                         out->embeddings;
  if (want_tree) {
    TreeOut to{out->node_visits, out->parents, out->action_from_parent, out->children_index, out->children_visits,
               out->raw_values, out->node_values, out->raw_values_epistemic_variance, out->node_values_epistemic_variance,
               out->children_prior_logits, out->children_rewards, out->children_discounts, out->children_values,
               out->children_rewards_epistemic_variance, out->children_values_epistemic_variance, out->embeddings};
    ProfScope ps(CLS_EXPORT, st);
    export_tree_kernel<<<148 * 8, 256, 0, st>>>(t, to);
    EAZ_CHECK_LAUNCH("export_tree_kernel");
  }
  return 0;
}

// Auxiliary streams / events for EAZ_FLAG_STREAMS: one set PER WORKSPACE (the workspace already identifies one search at a
// time -- two searches must not share one), so concurrent callers -- host threads, plans on different user streams -- never
// re-record each other's fork / join events or interleave on each other's streams.  Sets are created on first use, kept in a
// small per-process table (never destroyed: they may be baked into captured graphs) and, should a process ever cycle
// through more than kAuxSets workspaces, shared by hashing -- which only costs false serialisation, because a set is locked
// for the whole enqueue.
struct AuxStreams {
  cudaStream_t s[8];
  cudaEvent_t fork, join[8];
  std::mutex enqueue;  // held from the fork record to the last join wait
  const void* owner = nullptr;
  int device = -1;
  bool ready = false;
};
constexpr int kAuxSets = 64;
static AuxStreams* aux_streams(const void* workspace) {
  static AuxStreams table[kAuxSets];
  static std::mutex mu;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
  std::lock_guard<std::mutex> lock(mu);
  AuxStreams* pick = nullptr;
  for (int i = 0; i < kAuxSets && !pick; ++i)
    if (table[i].ready && table[i].owner == workspace && table[i].device == dev) pick = &table[i];
  for (int i = 0; i < kAuxSets && !pick; ++i)
    if (!table[i].ready) {
      AuxStreams* a = &table[i];
      for (int k = 0; k < 8; ++k) {
        if (cudaStreamCreateWithFlags(&a->s[k], cudaStreamNonBlocking) != cudaSuccess) return nullptr;
        if (cudaEventCreateWithFlags(&a->join[k], cudaEventDisableTiming) != cudaSuccess) return nullptr;
      }
      if (cudaEventCreateWithFlags(&a->fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
      a->owner = workspace;
      a->device = dev;
      a->ready = true;
      pick = a;
    }
  if (!pick) {  // table full: share a set of the same device (serialised by its enqueue mutex)
    const size_t h = ((uintptr_t)workspace >> 8) * 0x9E3779B97F4A7C15ull >> 32;
    for (int k = 0; k < kAuxSets && !pick; ++k) {
      AuxStreams* a = &table[(h + k) % kAuxSets];
      if (a->device == dev) pick = a;
    }
  }
  return pick;
}

int eaz_search_gumbel(const eaz_search_config* cfg, const eaz_search_inputs* in, eaz_search_outputs* out, void* workspace,
                      size_t workspace_bytes, void* stream) {
  EAZ_CHECK_ARG(cfg && in && out, "search: NULL config / inputs / outputs");
  int sizes[8], parts = 1;
  if (cfg->batch >= 1) sub_batches(cfg, sizes, &parts);
  bool persistent = false;
  {
    EnvDesc d;
    if (cfg->batch >= 1 && in->env && make_env_desc(in->env, &d) == 0)
      persistent = persistent_eligible(cfg->batch, cfg->num_simulations + 1, d.num_actions, cfg->flags, d, cfg->mlp_mode, nullptr);
  }
  if (parts <= 1 || tl_prof != nullptr || persistent) {  // (the persistent kernel's CTAs are independent chains already: nothing to split)
    eaz_search_config c = *cfg;
    c.flags = (c.flags & ~(kFlagManyTrees | kFlagSqFused)) | (cfg->batch >= kManyTrees ? kFlagManyTrees : 0) | (subleq_fused_for(cfg->batch) ? kFlagSqFused : 0);
    return search_one(&c, in, out, workspace, workspace_bytes, stream);
  }
  // ---- EAZ_FLAG_STREAMS: independent sub-batches (trees never interact) searched concurrently on auxiliary streams, so that
  // one sub-batch's tree kernel (issue-bound) overlaps another's network kernel (tensor / L2-bound) and env step (latency-bound)
  EnvDesc env;
  NetDesc net;
  if (int rc = check_search(cfg, in, out, &env, &net)) return rc;
  AuxStreams* aux = aux_streams(workspace);
  if (!aux) {
    set_error("could not create the auxiliary streams for EAZ_FLAG_STREAMS");
    return EAZ_ERR_CUDA;
  }
  std::lock_guard<std::mutex> enqueue_lock(aux->enqueue);
  const size_t A = env.num_actions, N = cfg->num_simulations + 1, S = env.compact_bytes, D = env.obs_dim, W = env.ws;
  size_t need = 0;
  for (int p = 0; p < parts; ++p) need += layout_bytes(cfg, env, sizes[p]);
  if (!workspace || workspace_bytes < need || ((uintptr_t)workspace & 255)) {
    set_error("search workspace must be >= %zu bytes and 256-byte aligned (got %zu)", need, workspace_bytes);
    return EAZ_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaError_t e = cudaEventRecord(aux->fork, st); e != cudaSuccess) return cuda_fail(e, "fork event");
  size_t b0 = 0, ws_off = 0;
  int rc_all = 0;
  for (int p = 0; p < parts; ++p) {
    eaz_search_config c = *cfg;
    c.batch = sizes[p];
    c.flags &= ~(0xF << EAZ_FLAG_STREAMS_SHIFT);
    c.flags = (c.flags & ~(kFlagManyTrees | kFlagSqFused)) | (cfg->batch >= kManyTrees ? kFlagManyTrees : 0) | (subleq_fused_for(cfg->batch) ? kFlagSqFused : 0);
    auto offf = [&](const float* q, size_t per) { return q ? q + b0 * per : nullptr; };
    auto offu = [&](const uint8_t* q, size_t per) { return q ? q + b0 * per : nullptr; };
    auto offi = [&](const int32_t* q, size_t per) { return q ? q + b0 * per : nullptr; };
    const eaz_state* e0 = in->embedding;
    eaz_state es{};
    if (e0) {
      es.step_count = (int32_t*)offi(e0->step_count, 1);
      es.rewards = (float*)offf(e0->rewards, 1);
      es.terminated = (uint8_t*)offu(e0->terminated, 1);
      es.truncated = (uint8_t*)offu(e0->truncated, 1);
      es.observation = (uint8_t*)offu(e0->observation, D);
      es.col = (int32_t*)offi(e0->col, 1);
      es.memory = (int32_t*)offi(e0->memory, W);
      es.task = (int32_t*)offi(e0->task, 1);
      es.solved = (uint8_t*)offu(e0->solved, 1);
      es.input_after = (int32_t*)offi(e0->input_after, 8);
      es.output_after = (int32_t*)offi(e0->output_after, 8);
    }
    eaz_search_inputs si = *in;
    si.prior_logits = offf(in->prior_logits, A);
    si.value = offf(in->value, 1);
    si.value_epistemic_variance = offf(in->value_epistemic_variance, 1);
    si.beta = offf(in->beta, 1);
    si.embedding = e0 ? &es : nullptr;
    si.invalid_actions = offu(in->invalid_actions, A);
    si.gumbel = offf(in->gumbel, A);
    si.sample_gumbel = offf(in->sample_gumbel, A);
    eaz_search_outputs so = *out;
    so.action = (int32_t*)offi(out->action, 1);
    so.action_weights = (float*)offf(out->action_weights, A);
    so.value = (float*)offf(out->value, 1);
    so.value_epistemic_std = (float*)offf(out->value_epistemic_std, 1);
    so.visit_counts = (float*)offf(out->visit_counts, A);
    so.visit_probs = (float*)offf(out->visit_probs, A);
    so.qvalues = (float*)offf(out->qvalues, A);
    so.qvalues_epistemic_variance = (float*)offf(out->qvalues_epistemic_variance, A);
    so.node_visits = (int32_t*)offi(out->node_visits, N);
    so.raw_values = (float*)offf(out->raw_values, N);
    so.node_values = (float*)offf(out->node_values, N);
    so.raw_values_epistemic_variance = (float*)offf(out->raw_values_epistemic_variance, N);
    so.node_values_epistemic_variance = (float*)offf(out->node_values_epistemic_variance, N);
    so.parents = (int32_t*)offi(out->parents, N);
    so.action_from_parent = (int32_t*)offi(out->action_from_parent, N);
    so.children_index = (int32_t*)offi(out->children_index, N * A);
    so.children_prior_logits = (float*)offf(out->children_prior_logits, N * A);
    so.children_visits = (int32_t*)offi(out->children_visits, N * A);
    so.children_rewards = (float*)offf(out->children_rewards, N * A);
    so.children_discounts = (float*)offf(out->children_discounts, N * A);
    so.children_values = (float*)offf(out->children_values, N * A);
    so.children_rewards_epistemic_variance = (float*)offf(out->children_rewards_epistemic_variance, N * A);
    so.children_values_epistemic_variance = (float*)offf(out->children_values_epistemic_variance, N * A);
    so.embeddings = (uint8_t*)offu(out->embeddings, N * S);
    so.root_value = (float*)offf(out->root_value, 1);
    so.root_ube = (float*)offf(out->root_ube, 1);
    const size_t bytes = layout_bytes(cfg, env, sizes[p]);
    cudaStream_t sp = aux->s[p];
    if (cudaError_t e = cudaStreamWaitEvent(sp, aux->fork, 0); e != cudaSuccess) return cuda_fail(e, "fork wait");
    const int rc = search_one(&c, &si, &so, (uint8_t*)workspace + ws_off, bytes, sp, (int)b0);
    if (rc && !rc_all) rc_all = rc;
    // always rejoin, also after an error: a forked stream must not be left dangling inside a stream capture
    if (cudaError_t e = cudaEventRecord(aux->join[p], sp); e != cudaSuccess) return cuda_fail(e, "join event");
    if (cudaError_t e = cudaStreamWaitEvent(st, aux->join[p], 0); e != cudaSuccess) return cuda_fail(e, "join wait");
    b0 += sizes[p];
    ws_off += bytes;
  }
  return rc_all;
}

int eaz_search_numeric_status(const eaz_search_config* cfg, const eaz_env* env_in, const void* workspace, size_t workspace_bytes, void* stream,
                              int32_t* flags_out) {
  EAZ_CHECK_ARG(cfg && workspace, "numeric status: NULL config / workspace");
  EnvDesc env;
  if (int rc = make_env_desc(env_in, &env)) return rc;
  if (flags_out) *flags_out = 0;
  if (cfg->mlp_mode != EAZ_MLP_TENSOR || cfg->batch < 1) return 0;  // the fp32 FMA path has no scaled split
  int sizes[8], parts = 1;
  sub_batches(cfg, sizes, &parts);
  if (persistent_eligible(cfg->batch, cfg->num_simulations + 1, env.num_actions, cfg->flags, env, cfg->mlp_mode, nullptr)) parts = 1;
  if (parts == 1) sizes[0] = cfg->batch;
  if (cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream); e != cudaSuccess) return cuda_fail(e, "numeric status sync");
  const size_t wbytes = wimg_bytes_for(cfg->mlp_mode, env);
  uint32_t flags = 0;
  size_t ws_off = 0;
  for (int p = 0; p < parts; ++p) {
    Layout L;
    make_layout(sizes[p], cfg->num_simulations + 1, env.num_actions, env.compact_bytes, (cfg->max_num_considered_actions + 1) * cfg->num_simulations,
                env.obs_dim, wbytes, ds_out_bytes(cfg->mlp_mode, env), cfg->max_depth > 0 ? cfg->max_depth : cfg->num_simulations, &L);
    if (ws_off + L.total > workspace_bytes) break;
    const uint8_t* ns = (const uint8_t*)workspace + ws_off + L.off[24] + wbytes - 256;
    uint32_t f = 0;
    if (cudaError_t e = cudaMemcpy(&f, ns + offsetof(NumStatus, flags), sizeof(f), cudaMemcpyDeviceToHost); e != cudaSuccess) return cuda_fail(e, "numeric status read");
    flags |= f;
    ws_off += L.total;
  }
  if (flags_out) *flags_out = (int32_t)flags;
  if (flags == 0) return 0;
  set_error("tensor-core network path out of range:%s%s -- use mlp_mode EXACT for this model",
            (flags & kNumWeightsNonFinite) ? " a weight matrix holds inf / nan or |w| > 2^20;" : "",
            (flags & kNumActSaturated) ? " a hidden activation exceeded 4094 (fp16 range of the 16x-scaled split) and was clamped;" : "");
  return EAZ_ERR_UNSUPPORTED;
}

int eaz_reanalyze_targets(const eaz_reanalyze_config* cfg, int32_t B, int32_t A, const int32_t* action, const float* qvalues,
                          const float* qvalues_epistemic_variance, const float* visit_counts, const float* value,
                          const float* value_epistemic_std, const float* next_state_value, const float* next_rewards,
                          const uint8_t* next_terminated, const uint8_t* terminated, const uint8_t* invalid_actions,
                          float* value_target, float* ube_target, float* exploration_policy_target, void* stream) {
  EAZ_CHECK_ARG(cfg != nullptr && B >= 0 && A >= 1 && A <= 256, "eaz_reanalyze_targets: bad cfg / B / A (1 <= A <= 256)");
  EAZ_CHECK_ARG(action && qvalues && qvalues_epistemic_variance && visit_counts && value && value_epistemic_std && next_state_value &&
                    next_rewards && next_terminated && terminated && value_target && ube_target && exploration_policy_target,
                "eaz_reanalyze_targets: NULL array");
  if (B == 0) return 0;
  ReanalyzeArgs r{action, qvalues, qvalues_epistemic_variance, visit_counts, value, value_epistemic_std, next_state_value, next_rewards,
                  next_terminated, terminated, invalid_actions, value_target, ube_target, exploration_policy_target};
  cudaStream_t st = (cudaStream_t)stream;
#define EAZ_RUN(G, J) reanalyze_targets_kernel<G, J><<<ceil_div(B, 4 * (32 / G)), 128, 0, st>>>(*cfg, B, A, r)
  if (A <= 2) EAZ_RUN(2, 1);
  else if (A <= 4) EAZ_RUN(4, 1);
  else if (A <= 8) EAZ_RUN(8, 1);
  else if (A <= 16) EAZ_RUN(16, 1);
  else if (A <= 32) EAZ_RUN(32, 1);
  else if (A <= 64) EAZ_RUN(32, 2);
  else if (A <= 128) EAZ_RUN(32, 4);
  else EAZ_RUN(32, 8);
#undef EAZ_RUN
  EAZ_CHECK_LAUNCH("reanalyze_targets_kernel");
  return 0;
}

int eaz_search_gumbel_profiled(const eaz_search_config* cfg, const eaz_search_inputs* in, eaz_search_outputs* out, void* workspace,
                               size_t workspace_bytes, void* stream, float* ms_by_class, int32_t* launches_by_class) {
  EAZ_CHECK_ARG(ms_by_class && launches_by_class, "profiled search: NULL result arrays");
  Prof prof;
  tl_prof = &prof;
  const int rc = eaz_search_gumbel(cfg, in, out, workspace, workspace_bytes, stream);
  tl_prof = nullptr;
  cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
  for (int c = 0; c < EAZ_PROFILE_CLASSES; ++c) { ms_by_class[c] = 0.0f; launches_by_class[c] = 0; }
  for (size_t i = 0; i < prof.cls.size(); ++i) {
    float ms = 0.0f;
    if (e == cudaSuccess && rc == 0) cudaEventElapsedTime(&ms, prof.ev[2 * i], prof.ev[2 * i + 1]);
    ms_by_class[prof.cls[i]] += ms;
    launches_by_class[prof.cls[i]] += 1;
    cudaEventDestroy(prof.ev[2 * i]);
    cudaEventDestroy(prof.ev[2 * i + 1]);
  }
  if (e != cudaSuccess) return cuda_fail(e, "profiled search sync");
  return rc;
}

// Debug hook (not in the public header): device buffer of num_simulations * 128 u64 receiving the per-simulation milestones of the
// tree warps of CTA 0 of the persistent search kernel (psearch.cuh: Trace).
void eaz_debug_set_ps_trace(unsigned long long* device_buffer) { eaz::g_ps_trace = device_buffer; }

// Debug hook (not in the public header): device buffer of (n+1)*B*8 int64 receiving per-tree section stamps of tree_step_kernel.
void eaz_debug_set_tree_trace(long long* device_buffer) { eaz::g_tree_trace = device_buffer; }

}  // extern "C"
