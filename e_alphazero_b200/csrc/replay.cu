// replay.cu -- prioritised replay sampling on the device (SURVEY 8f-3): the sum tree behind the reference's flashbax
// prioritised flat buffer (main.py:217-225 priority_exponent, main.py:413-414 sample / batch.indices, main.py:454
// set_priorities), over the slots of a compact replay ring [T slots, B envs].
//
// THE CONTRACT (oracle: tests/priority_oracle.c states the same rules; both must change together)
//
//   Items.  Item i = t * B + b is the pair (slot t, slot (t + 1) % T) of env b.  t is the PHYSICAL ring slot, so an index
//     is an opaque handle, as flashbax's are.  An item is VALID only when both of its slots hold data and slot t + 1 is not
//     the slot written next (slot s holds data iff (cursor - 1 - s) mod T < length).  An invalid item has weight 0.
//   Weights.  w(p) = eaz_exp(eaz_mul(alpha, eaz_log(p))) for 0 < p <= FLT_MAX, w = 0 for p == 0 (also at alpha = 0).
//     A negative or non-finite p is stored as 0 and sets EAZ_PRIORITY_BAD_PRIORITY.
//   Buffer (eaz_priority_tree_bytes).  [0, 32): header {float alpha; uint32 seed; uint32 draw_ctr; uint32 status;
//     int32 cursor; int32 length; float max_priority (raw p, starts at 1); uint32 0}; [256, ...): int32 tag[N] (-1 between
//     calls: the duplicate resolution of eaz_priority_set), then the fp32 levels, leaves first: n_0 = N = T * B,
//     n_{l+1} = ceil(n_l / 32) down to n_{L-1} = 1.  Every region starts at a multiple of 128 bytes and each level is
//     padded with zeros to a multiple of 32 floats.
//   Node sums.  Node j of level l + 1 = orc_tree_sum of the 32 children 32 j .. 32 j + 31 of level l (child c in lane c,
//     xor-butterfly with strides 1, 2, 4, 8, 16; a missing child is 0).  A node is always recomputed from its children,
//     never updated by a delta, so the tree is a pure function of the leaves.
//   add_step(c).  If c == cursor: cursor = (c + 1) % T, length = min(length + 1, T); if c == cursor - 1 (the newest slot
//     was rewritten) cursor and length stay; any other c sets EAZ_PRIORITY_BAD_ADD and changes nothing.  Then the items of
//     row c - 1 get w(max_priority) if length >= 2 (else 0) and the items of row c get 0.
//   set(indices[K], priorities[K]).  An index outside [0, N) sets EAZ_PRIORITY_BAD_INDEX and is skipped.  For a duplicated
//     index the LAST occurrence in the batch wins.  The leaf becomes w(p) if the item is valid, else 0.  max_priority =
//     max(max_priority, p of every in-range entry).
//   sample(K).  total = the root.  Sample k: r_k = 24 bits of h * 2^-24 with h = seed + 0x9E3779B1; h = xx_round(h,
//     draw_ctr); h = xx_round(h, k); then the xxhash avalanche (>>15, *P2, >>13, *P3, >>16), r_k = (h >> 8) * 2^-24;
//     u = eaz_mul(eaz_div(eaz_add((float)k, r_k), (float)K), total).  Descent from the root: over the 32 children w_0..w_31
//     of the current node, prefix_c = ((0 + w_0) + w_1) + ... + w_c (serial, ascending); pick the first c with prefix_c > u
//     and w_c > 0; if none, the last c with w_c > 0; then u = eaz_sub(u, prefix_{c-1}) (0 for c = 0).  At the leaf:
//     index i, probability = eaz_div(w_i, total).  The draw counter advances once per call.  total == 0 (or not finite)
//     sets EAZ_PRIORITY_EMPTY and every sample is index 0, probability 0.
//
// A keyed sample (eaz_priority_sample_keyed) is sample(K) with (seed, draw_ctr) := (key[0], key[1]) that writes nothing into
// the buffer: no counter advance, no status bit.  eaz_replay_add's add_step is add_step(c) with c = the header's cursor.
//
// add_sequence(n) (eaz_replay_add_sequence) IS n calls of add_step(cursor), in every byte of the buffer; it is not a second rule.
//   Derivation, with c, len, m = the header's cursor, length, max_priority before the call and w = w(m): call k (0 <= k < n) is
//   add_step(c + k), which sets length min(len + k + 1, T), so it writes row c + k - 1 := w if len + k >= 1 (else 0), then row
//   c + k := 0.  Call k only writes logical rows c + k - 1 and c + k, so a physical row ends with the value of the LAST logical
//   row j == it (mod T) in c - 1 .. c + n - 1: logical row c + n - 1 ends at 0, logical row c + k - 1 (k < n) at w if
//   len + k >= 1, else 0.  The touched physical rows are the last min(n + 1, T) of those logical rows.  The header ends with
//   cursor (c + n) % T and length min(len + n, T); max_priority, alpha, status and the tags are not written by add_step(cursor).
//   The levels being a pure function of the leaves, setting the touched leaves to their final values and recomputing their
//   ancestors gives the bytes of the n sequential calls, for any n (n > T included) and any starting ring.
//
// Kernels: add_step is one CTA (two rows of B leaves, then their ancestors level by level); set is a tag pass (atomicMax
// of k per leaf: last occurrence wins), a leaf pass, and one launch per level above the leaves; sample is one warp per
// sample (descent + gather of both slots' compact records and rewards) and, unless keyed, a one-thread counter bump.
// eaz_replay_add is a compaction kernel that writes ring row `cursor` (read from the header) followed by add_step with the
// slot taken from the header, so the cursor never leaves the device.  eaz_replay_add_sequence is a row-copy kernel (the last
// min(n, T) rows into their slots), a leaf pass over the touched rows and one launch per level above the leaves, the root's
// launch also writing the header: L + 1 launches whatever n.  All latency-bound.
#include "common.cuh"

#include <float.h>

namespace eaz {

struct PrioHeader {
  float alpha;
  uint32_t seed;
  uint32_t draw_ctr;
  uint32_t status;
  int32_t cursor;
  int32_t length;
  float max_priority;
  uint32_t reserved;
};
static_assert(sizeof(PrioHeader) == 32, "header layout is part of the oracle contract");

constexpr int kPrioMaxLevels = 8;  // N < 2^31 = 32^6 * 32: at most 8 levels

struct PrioTree {
  PrioHeader* hdr;
  int32_t* tag;
  float* lvl[kPrioMaxLevels];
  float* root;  // lvl[L - 1]
  int L, T, B, N;
};

struct PrioGeom {
  int L, n[kPrioMaxLevels];
  size_t tag_off, lvl_off[kPrioMaxLevels], bytes;
};

static inline size_t align128(size_t x) { return (x + 127) / 128 * 128; }

static int prio_geom(int32_t T, int32_t B, PrioGeom* g, const char* who) {
  EAZ_CHECK_ARG(T >= 2 && B >= 1, "%s: need T >= 2 time slots and B >= 1 envs (got T=%d, B=%d)", who, T, B);
  EAZ_CHECK_ARG((int64_t)T * B < ((int64_t)1 << 31), "%s: T * B = %lld items must be below 2^31", who, (long long)T * B);
  const int N = T * B;
  g->tag_off = 256;
  size_t off = align128(g->tag_off + (size_t)N * 4);
  int n = N, L = 0;
  while (true) {
    g->n[L] = n;
    g->lvl_off[L] = off;
    off += align128((size_t)(n + 31) / 32 * 32 * 4);
    ++L;
    if (n == 1) break;
    n = (n + 31) / 32;
  }
  g->L = L;
  g->bytes = off;
  return 0;
}

static int prio_view(void* tree, size_t tree_bytes, int32_t T, int32_t B, PrioTree* tr, const char* who) {
  PrioGeom g;
  if (int rc = prio_geom(T, B, &g, who)) return rc;
  EAZ_CHECK_ARG(tree != nullptr && ((uintptr_t)tree % 128) == 0, "%s: tree must be a 128-byte aligned device buffer", who);
  EAZ_CHECK_ARG(tree_bytes >= g.bytes, "%s: tree buffer of %zu bytes, eaz_priority_tree_bytes(%d, %d) = %zu", who, tree_bytes, T, B, g.bytes);
  uint8_t* p = (uint8_t*)tree;
  tr->hdr = (PrioHeader*)p;
  tr->tag = (int32_t*)(p + g.tag_off);
  for (int l = 0; l < kPrioMaxLevels; ++l) tr->lvl[l] = l < g.L ? (float*)(p + g.lvl_off[l]) : nullptr;
  tr->root = tr->lvl[g.L - 1];
  tr->L = g.L, tr->T = T, tr->B = B, tr->N = T * B;
  return 0;
}

__device__ __forceinline__ float prio_weight(float p, float alpha) { return p > 0.0f ? eaz_exp(eaz_mul(alpha, eaz_log(p))) : 0.0f; }
__device__ __forceinline__ bool prio_bad(float p) { return !(p >= 0.0f && p <= FLT_MAX); }
__device__ __forceinline__ float prio_clean(float p) { return (p > 0.0f && p <= FLT_MAX) ? p : 0.0f; }

__device__ __forceinline__ bool prio_filled(int s, int T, int cursor, int length) {
  int a = cursor - 1 - s;
  if (a < 0) a += T;
  return a < length;
}
__device__ __forceinline__ bool prio_valid(int t, int T, int cursor, int length) {
  const int t1 = t + 1 == T ? 0 : t + 1;
  return t1 != cursor && prio_filled(t, T, cursor, length) && prio_filled(t1, T, cursor, length);
}

// node j of level l (>= 1) from its 32 children, by one whole warp (the orc_tree_sum order)
__device__ __forceinline__ void prio_recompute(const float* child, float* node, int j, int lane) {
  const float v = group_sum<32>(child[32 * j + lane]);
  if (lane == 0) node[j] = v;
}

__global__ void prio_init_kernel(PrioTree tr, float alpha, uint32_t seed) {
  PrioHeader h;
  h.alpha = alpha, h.seed = seed, h.draw_ctr = 0u, h.status = 0u, h.cursor = 0, h.length = 0, h.max_priority = 1.0f, h.reserved = 0u;
  *tr.hdr = h;
}

// c < 0: the slot is the header's cursor (eaz_replay_add: no host copy of the cursor exists)
__global__ void __launch_bounds__(1024) prio_add_step_kernel(PrioTree tr, int c) {
  __shared__ int s_ok, s_c;
  __shared__ float s_w;
  const int T = tr.T, B = tr.B;
  if (threadIdx.x == 0) {
    const PrioHeader h = *tr.hdr;
    if (c < 0) c = h.cursor;
    s_c = c;
    int ok = 1, cur = h.cursor, len = h.length;
    if (c == h.cursor) {
      cur = c + 1 == T ? 0 : c + 1;
      len = min(len + 1, T);
    } else if (c != (h.cursor == 0 ? T - 1 : h.cursor - 1)) {
      ok = 0;
      tr.hdr->status = h.status | EAZ_PRIORITY_BAD_ADD;
    }
    if (ok) tr.hdr->cursor = cur, tr.hdr->length = len;
    s_ok = ok;
    s_w = len >= 2 ? prio_weight(h.max_priority, h.alpha) : 0.0f;
  }
  __syncthreads();
  if (!s_ok) return;
  c = s_c;
  const int rp = c == 0 ? T - 1 : c - 1;
  const float w = s_w;
  for (int j = threadIdx.x; j < 2 * B; j += blockDim.x) {
    if (j < B) tr.lvl[0][(size_t)rp * B + j] = w;
    else tr.lvl[0][(size_t)c * B + (j - B)] = 0.0f;
  }
  __syncthreads();
  int lo0 = rp * B, hi0 = rp * B + B - 1, lo1 = c * B, hi1 = c * B + B - 1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
#pragma unroll
  for (int l = 1; l < kPrioMaxLevels; ++l) {  // unrolled: tr.lvl[] is indexed by constants (no local-memory copy of the struct)
    if (l >= tr.L) break;
    lo0 >>= 5, hi0 >>= 5, lo1 >>= 5, hi1 >>= 5;
    int n0 = hi0 - lo0 + 1, n1 = hi1 - lo1 + 1;
    if (lo1 <= hi0 + 1 && lo0 <= hi1 + 1) {  // overlapping or adjacent ranges: one range, no node twice
      const int lo = min(lo0, lo1), hi = max(hi0, hi1);
      n0 = hi - lo + 1, lo0 = lo, n1 = 0;
    }
    for (int q = warp; q < n0 + n1; q += nwarps) prio_recompute(tr.lvl[l - 1], tr.lvl[l], q < n0 ? lo0 + q : lo1 + (q - n0), lane);
    __syncthreads();
  }
}

__global__ void prio_set_tag_kernel(PrioTree tr, const int32_t* __restrict__ idx, const float* __restrict__ pri, int K) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  const int i = idx[k];
  const float p = pri[k];
  if (prio_bad(p)) atomicOr(&tr.hdr->status, (uint32_t)EAZ_PRIORITY_BAD_PRIORITY);
  if (i < 0 || i >= tr.N) {
    atomicOr(&tr.hdr->status, (uint32_t)EAZ_PRIORITY_BAD_INDEX);
    return;
  }
  atomicMax(&tr.tag[i], k);
  atomicMax((unsigned int*)&tr.hdr->max_priority, __float_as_uint(prio_clean(p)));  // non-negative floats order as their bits
}

__global__ void prio_set_leaf_kernel(PrioTree tr, const int32_t* __restrict__ idx, const float* __restrict__ pri, int K) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  const int i = idx[k];
  if (i < 0 || i >= tr.N || tr.tag[i] != k) return;  // the last occurrence of a duplicated index writes
  const int cursor = tr.hdr->cursor, length = tr.hdr->length;
  tr.lvl[0][i] = prio_valid(i / tr.B, tr.T, cursor, length) ? prio_weight(prio_clean(pri[k]), tr.hdr->alpha) : 0.0f;
}

// one warp per entry recomputes the entry's ancestor at level l; the level-1 pass also clears the tags the tag pass set
__global__ void prio_set_level_kernel(const float* child, float* node, int32_t* tag, const int32_t* __restrict__ idx, int K, int N, int l) {
  const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (k >= K) return;
  const int i = idx[k];
  if (i < 0 || i >= N) return;
  prio_recompute(child, node, i >> (5 * l), lane);
  if (l == 1 && lane == 0) tag[i] = -1;
}

__device__ __forceinline__ float prio_uniform(uint32_t seed, uint32_t ctr, uint32_t k) {
  uint32_t h = seed + EAZ_XX_P1;
  h = xx_round(h, ctr);
  h = xx_round(h, k);
  h ^= h >> 15; h *= EAZ_XX_P2; h ^= h >> 13; h *= EAZ_XX_P3; h ^= h >> 16;
  return __fmul_rn((float)(h >> 8), 5.9604644775390625e-08f);  // 24 random bits * 2^-24: exact
}

// key == nullptr: (seed, draw_ctr) from the header, an empty tree sets EAZ_PRIORITY_EMPTY (the caller bumps the counter).
// key != nullptr (keyed sampling): (seed, draw_ctr) = (key[0], key[1]) and the tree is only read.
__global__ void __launch_bounds__(256) prio_sample_kernel(PrioTree tr, int K, const uint32_t* __restrict__ key,
                                                          const uint8_t* __restrict__ states, const float* __restrict__ rewards, int S,
                                                          int32_t* __restrict__ out_idx, float* __restrict__ out_prob,
                                                          uint8_t* __restrict__ first, float* __restrict__ first_r,
                                                          uint8_t* __restrict__ second, float* __restrict__ second_r) {
  const int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (k >= K) return;
  const float* node = tr.root;
  const float total = node[0];
  int i = 0;
  float prob = 0.0f;
  if (!(total > 0.0f && total <= FLT_MAX)) {
    if (lane == 0 && key == nullptr) atomicOr(&tr.hdr->status, (uint32_t)EAZ_PRIORITY_EMPTY);
  } else {
    const uint32_t seed = key ? key[0] : tr.hdr->seed, ctr = key ? key[1] : tr.hdr->draw_ctr;
    float u = eaz_mul(eaz_div(eaz_add((float)k, prio_uniform(seed, ctr, (uint32_t)k)), (float)K), total);
    int j = 0;
    float wc = 0.0f;
    for (int l = tr.L - 1; l >= 1; --l) {
      // level l-1 fills the 32 * n_l floats right below level l, n_l = ceil(N / 32^l) (no indexing of tr.lvl[]: that would
      // copy the struct to local memory)
      node -= (size_t)32 * (size_t)((((int64_t)tr.N - 1) >> (5 * l)) + 1);
      const float w = node[32 * j + lane];
      float pre = 0.0f;
#pragma unroll
      for (int q = 0; q < 32; ++q) {
        const float x = __shfl_sync(0xffffffffu, w, q);
        if (q <= lane) pre = __fadd_rn(pre, x);
      }
      const uint32_t hit = __ballot_sync(0xffffffffu, pre > u && w > 0.0f);
      const uint32_t nz = __ballot_sync(0xffffffffu, w > 0.0f);
      const int c = hit ? __ffs(hit) - 1 : (nz ? 31 - __clz(nz) : 0);
      const float excl = __shfl_sync(0xffffffffu, pre, (c + 31) & 31);
      wc = __shfl_sync(0xffffffffu, w, c);
      u = __fsub_rn(u, c == 0 ? 0.0f : excl);
      j = 32 * j + c;
    }
    i = j;
    prob = __fdiv_rn(wc, total);
  }
  if (lane == 0) out_idx[k] = i, out_prob[k] = prob;
  if (states == nullptr) return;
  const int t = i / tr.B, b = i - t * tr.B, t1 = t + 1 == tr.T ? 0 : t + 1;
  const size_t r0 = (size_t)t * tr.B + b, r1 = (size_t)t1 * tr.B + b;
  for (int q = lane; q < S; q += 32) {
    first[(size_t)k * S + q] = states[r0 * S + q];
    second[(size_t)k * S + q] = states[r1 * S + q];
  }
  if (lane == 0 && rewards != nullptr) first_r[k] = rewards[r0], second_r[k] = rewards[r1];
}

__global__ void prio_bump_kernel(PrioHeader* hdr) { hdr->draw_ctr += 1u; }

// eaz_replay_add, first launch: the B states into ring row `cursor` (read on the device; prio_add_step_kernel advances it after)
__global__ void replay_compact_kernel(EnvDesc env, StateSoA s, const PrioHeader* __restrict__ hdr, uint8_t* __restrict__ ring_states,
                                      float* __restrict__ ring_rewards, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const size_t slot = (size_t)hdr->cursor;
  pack_state(env, s, b, ring_states + slot * B * env.compact_bytes);
  ring_rewards[slot * B + b] = s.rewards[b];
}

// ---- eaz_replay_add_sequence (add_sequence(n) of the contract).  `keep` = min(n, T) rows are written, `rows` = min(n + 1, T) leaf
// rows are touched.  Every kernel reads the cursor c from the header; only the root's level pass, the last launch, writes it.

// physical slot of the first of the last `count` logical slots c .. c + n - 1 (ring rows: (c, n); leaf rows: (c - 1, n + 1))
__device__ __forceinline__ int seq_first_slot(int c, int n, int count, int T) { return (int)(((int64_t)c + n - count + T) % T); }

// ring rows j = n - keep .. n - 1 of the sequence into slots (c + j) % T; V: the widest word dividing a row of B records
template <typename V>
__global__ void __launch_bounds__(256) replay_seq_copy_kernel(const PrioHeader* __restrict__ hdr, const V* __restrict__ src, V* __restrict__ dst,
                                                              int64_t row_words, const float* __restrict__ rewards, float* __restrict__ ring_rewards,
                                                              int B, int T, int n, int keep) {
  const int s0 = seq_first_slot(hdr->cursor, n, keep, T);
  const int64_t j0 = n - keep, stride = (int64_t)gridDim.x * blockDim.x, first = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (int64_t e = first; e < keep * row_words; e += stride) {
    const int64_t q = e / row_words, o = e - q * row_words;
    const int64_t slot = s0 + q < T ? s0 + q : s0 + q - T;
    dst[slot * row_words + o] = src[(j0 + q) * row_words + o];
  }
  for (int64_t e = first; e < (int64_t)keep * B; e += stride) {
    const int64_t q = e / B, b = e - q * B;
    const int64_t slot = s0 + q < T ? s0 + q : s0 + q - T;
    ring_rewards[slot * B + b] = rewards[(j0 + q) * B + b];
  }
}

// the leaves of the touched rows: logical row c - 1 + k (k = n + 1 - rows + q) gets w if len + k >= 1, the last (k = n) gets 0
__global__ void __launch_bounds__(256) prio_seq_leaf_kernel(PrioTree tr, int n, int rows) {
  const PrioHeader h = *tr.hdr;
  const int T = tr.T, B = tr.B, p0 = seq_first_slot(h.cursor - 1, n + 1, rows, T);
  const float w = prio_weight(h.max_priority, h.alpha);
  const int stride = gridDim.x * blockDim.x;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < rows * B; e += stride) {
    const int q = e / B, b = e - q * B, k = n + 1 - rows + q;
    const int p = p0 + q < T ? p0 + q : p0 + q - T;
    tr.lvl[0][(size_t)p * B + b] = q == rows - 1 ? 0.0f : (h.length > 0 || k > 0) ? w : 0.0f;
  }
}

// one warp per ancestor at level l (>= 1) of the touched leaves: every node of the level when rows == T, else the nodes over the
// touched leaf range, which wraps past slot T - 1 into at most two ranges (merged where they meet, so no node is computed twice).
// The root's pass (n_nodes == 1, one warp) then writes the header: cursor (c + n) % T, length min(length + n, T).
__global__ void __launch_bounds__(256) prio_seq_level_kernel(PrioHeader* hdr, const float* child, float* node, int l, int n_nodes, int T, int B,
                                                             int n, int rows) {
  const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  const int c = hdr->cursor;
  int lo0 = 0, n0 = n_nodes, lo1 = 0, n1 = 0;
  if (rows < T) {
    const int p0 = seq_first_slot(c - 1, n + 1, rows, T), p1 = p0 + rows;
    lo0 = p0 * B;
    int hi0 = min(p1, T) * B - 1, hi1 = -1;
    if (p1 > T) hi1 = (p1 - T) * B - 1;
    lo0 >>= 5 * l, hi0 >>= 5 * l;
    n0 = hi0 - lo0 + 1;
    if (hi1 >= 0) {
      hi1 >>= 5 * l;
      if (lo1 <= hi0 + 1 && lo0 <= hi1 + 1) {
        const int lo = min(lo0, lo1), hi = max(hi0, hi1);
        lo0 = lo, n0 = hi - lo + 1;
      } else {
        n1 = hi1 - lo1 + 1;
      }
    }
  }
  if (q < n0 + n1) prio_recompute(child, node, q < n0 ? lo0 + q : lo1 + (q - n0), lane);
  if (n_nodes == 1 && q == 0) {
    __syncwarp();  // every lane has read the cursor
    if (lane == 0) {
      hdr->cursor = (int)(((int64_t)c + n) % T);
      hdr->length = (int)min((int64_t)hdr->length + n, (int64_t)T);
    }
  }
}

static int prio_sample_launch(void* tree, size_t tree_bytes, int32_t T, int32_t B, int32_t K, const uint32_t* key, const uint8_t* states,
                              const float* rewards, int32_t S, int32_t* indices, float* probabilities, uint8_t* first, float* first_rewards,
                              uint8_t* second, float* second_rewards, cudaStream_t s, const char* who) {
  PrioTree tr;
  if (int rc = prio_view(tree, tree_bytes, T, B, &tr, who)) return rc;
  EAZ_CHECK_ARG(K >= 1 && K <= (1 << 24), "%s: K = %d outside [1, 2^24]", who, K);
  EAZ_CHECK_ARG(indices && probabilities, "%s: NULL indices / probabilities", who);
  if (states) {
    EAZ_CHECK_ARG(S >= 1 && first && second, "%s: gathering needs S >= 1 and first / second buffers", who);
    EAZ_CHECK_ARG(!rewards || (first_rewards && second_rewards), "%s: rewards given without first / second reward buffers", who);
  }
  prio_sample_kernel<<<ceil_div(K, 8), 256, 0, s>>>(tr, K, key, states, rewards, S, indices, probabilities, first, first_rewards, second,
                                                    second_rewards);
  EAZ_CHECK_LAUNCH("prio_sample_kernel");
  return 0;
}

}  // namespace eaz

using namespace eaz;

extern "C" {

size_t eaz_priority_tree_bytes(int32_t T, int32_t B) {
  PrioGeom g;
  return prio_geom(T, B, &g, "eaz_priority_tree_bytes") ? 0 : g.bytes;
}

int eaz_priority_init(void* tree, size_t tree_bytes, int32_t T, int32_t B, float priority_exponent, uint32_t seed, void* stream) {
  PrioTree tr;
  if (int rc = prio_view(tree, tree_bytes, T, B, &tr, "eaz_priority_init")) return rc;
  EAZ_CHECK_ARG(priority_exponent >= 0.0f && priority_exponent <= 1.0f, "eaz_priority_init: priority_exponent must lie in [0, 1]");
  PrioGeom g;
  prio_geom(T, B, &g, "eaz_priority_init");
  cudaStream_t s = (cudaStream_t)stream;
  if (cudaError_t e = cudaMemsetAsync(tree, 0, g.bytes, s); e != cudaSuccess) return cuda_fail(e, "eaz_priority_init memset");
  if (cudaError_t e = cudaMemsetAsync(tr.tag, 0xff, (size_t)tr.N * 4, s); e != cudaSuccess) return cuda_fail(e, "eaz_priority_init memset");
  prio_init_kernel<<<1, 1, 0, s>>>(tr, priority_exponent, seed);
  EAZ_CHECK_LAUNCH("prio_init_kernel");
  return 0;
}

int eaz_priority_add_step(void* tree, size_t tree_bytes, int32_t T, int32_t B, int32_t slot, void* stream) {
  PrioTree tr;
  if (int rc = prio_view(tree, tree_bytes, T, B, &tr, "eaz_priority_add_step")) return rc;
  EAZ_CHECK_ARG(slot >= 0 && slot < T, "eaz_priority_add_step: slot %d outside [0, %d)", slot, T);
  prio_add_step_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(tr, slot);
  EAZ_CHECK_LAUNCH("prio_add_step_kernel");
  return 0;
}

int eaz_priority_set(void* tree, size_t tree_bytes, int32_t T, int32_t B, const int32_t* indices, const float* priorities, int32_t K,
                     void* stream) {
  PrioTree tr;
  if (int rc = prio_view(tree, tree_bytes, T, B, &tr, "eaz_priority_set")) return rc;
  EAZ_CHECK_ARG(K >= 0, "eaz_priority_set: K = %d < 0", K);
  if (K == 0) return 0;
  EAZ_CHECK_ARG(indices && priorities, "eaz_priority_set: NULL indices / priorities");
  cudaStream_t s = (cudaStream_t)stream;
  prio_set_tag_kernel<<<ceil_div(K, 256), 256, 0, s>>>(tr, indices, priorities, K);
  EAZ_CHECK_LAUNCH("prio_set_tag_kernel");
  prio_set_leaf_kernel<<<ceil_div(K, 256), 256, 0, s>>>(tr, indices, priorities, K);
  EAZ_CHECK_LAUNCH("prio_set_leaf_kernel");
  for (int l = 1; l < tr.L; ++l) {
    prio_set_level_kernel<<<ceil_div(K, 8), 256, 0, s>>>(tr.lvl[l - 1], tr.lvl[l], tr.tag, indices, K, tr.N, l);
    EAZ_CHECK_LAUNCH("prio_set_level_kernel");
  }
  return 0;
}

int eaz_priority_sample(void* tree, size_t tree_bytes, int32_t T, int32_t B, int32_t K, const uint8_t* states, const float* rewards, int32_t S,
                        int32_t* indices, float* probabilities, uint8_t* first, float* first_rewards, uint8_t* second,
                        float* second_rewards, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (int rc = prio_sample_launch(tree, tree_bytes, T, B, K, nullptr, states, rewards, S, indices, probabilities, first, first_rewards, second,
                                  second_rewards, s, "eaz_priority_sample"))
    return rc;
  prio_bump_kernel<<<1, 1, 0, s>>>((PrioHeader*)tree);
  EAZ_CHECK_LAUNCH("prio_bump_kernel");
  return 0;
}

int eaz_priority_sample_keyed(const void* tree, size_t tree_bytes, int32_t T, int32_t B, int32_t K, const uint32_t* key, const uint8_t* states,
                              const float* rewards, int32_t S, int32_t* indices, float* probabilities, uint8_t* first, float* first_rewards,
                              uint8_t* second, float* second_rewards, void* stream) {
  EAZ_CHECK_ARG(key != nullptr, "eaz_priority_sample_keyed: NULL key (a device uint32[2])");
  return prio_sample_launch(const_cast<void*>(tree), tree_bytes, T, B, K, key, states, rewards, S, indices, probabilities, first, first_rewards,
                            second, second_rewards, (cudaStream_t)stream, "eaz_priority_sample_keyed");
}

int eaz_replay_add(const eaz_env* env, const eaz_state* state, uint8_t* ring_states, float* ring_rewards, void* tree, size_t tree_bytes,
                   int32_t T, int32_t B, void* stream) {
  EnvDesc d;
  if (int rc = make_env_desc(env, &d)) return rc;
  PrioTree tr;
  if (int rc = prio_view(tree, tree_bytes, T, B, &tr, "eaz_replay_add")) return rc;
  EAZ_CHECK_ARG(state && state->step_count && state->rewards && state->terminated, "eaz_replay_add: NULL state / step_count / rewards / terminated");
  if (d.kind == EAZ_ENV_DEEPSEA) EAZ_CHECK_ARG(state->col != nullptr, "eaz_replay_add: col is NULL");
  else EAZ_CHECK_ARG(state->memory && state->task && state->solved && state->input_after && state->output_after, "eaz_replay_add: NULL Subleq leaf");
  EAZ_CHECK_ARG(ring_states && ring_rewards, "eaz_replay_add: NULL ring_states / ring_rewards");
  cudaStream_t s = (cudaStream_t)stream;
  replay_compact_kernel<<<ceil_div(B, 128), 128, 0, s>>>(d, soa_of(state), tr.hdr, ring_states, ring_rewards, B);
  EAZ_CHECK_LAUNCH("replay_compact_kernel");
  prio_add_step_kernel<<<1, 1024, 0, s>>>(tr, -1);
  EAZ_CHECK_LAUNCH("prio_add_step_kernel");
  return 0;
}

int eaz_replay_add_sequence(const eaz_env* env, const uint8_t* compact, const float* rewards, int32_t steps, uint8_t* ring_states,
                            float* ring_rewards, void* tree, size_t tree_bytes, int32_t T, int32_t B, int32_t S, void* stream) {
  EnvDesc d;
  if (int rc = make_env_desc(env, &d)) return rc;
  PrioTree tr;
  if (int rc = prio_view(tree, tree_bytes, T, B, &tr, "eaz_replay_add_sequence")) return rc;
  EAZ_CHECK_ARG(steps >= 0 && steps < INT32_MAX, "eaz_replay_add_sequence: steps = %d outside [0, 2^31 - 1)", steps);
  EAZ_CHECK_ARG(S == d.compact_bytes, "eaz_replay_add_sequence: S = %d, eaz_env_compact_bytes(env) = %d", S, d.compact_bytes);
  EAZ_CHECK_ARG(ring_states && ring_rewards, "eaz_replay_add_sequence: NULL ring_states / ring_rewards");
  EAZ_CHECK_ARG(steps == 0 || (compact && rewards), "eaz_replay_add_sequence: NULL compact / rewards");
  if (steps == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  const int keep = min(steps, T), rows = steps < T ? steps + 1 : T;
  const size_t row_bytes = (size_t)B * S;
  const int64_t copy_elems = (int64_t)keep * (int64_t)row_bytes;
  const int copy_blocks = (int)std::min<int64_t>((copy_elems + 255) / 256, 4096);
  const bool a16 = row_bytes % 16 == 0 && (uintptr_t)compact % 16 == 0 && (uintptr_t)ring_states % 16 == 0;
  const bool a4 = row_bytes % 4 == 0 && (uintptr_t)compact % 4 == 0 && (uintptr_t)ring_states % 4 == 0;
  if (a16)
    replay_seq_copy_kernel<uint4><<<copy_blocks, 256, 0, s>>>(tr.hdr, (const uint4*)compact, (uint4*)ring_states, (int64_t)(row_bytes / 16), rewards,
                                                              ring_rewards, B, T, steps, keep);
  else if (a4)
    replay_seq_copy_kernel<uint32_t><<<copy_blocks, 256, 0, s>>>(tr.hdr, (const uint32_t*)compact, (uint32_t*)ring_states, (int64_t)(row_bytes / 4),
                                                                 rewards, ring_rewards, B, T, steps, keep);
  else
    replay_seq_copy_kernel<uint8_t><<<copy_blocks, 256, 0, s>>>(tr.hdr, compact, ring_states, (int64_t)row_bytes, rewards, ring_rewards, B, T,
                                                                steps, keep);
  EAZ_CHECK_LAUNCH("replay_seq_copy_kernel");
  prio_seq_leaf_kernel<<<(int)std::min<int64_t>(((int64_t)rows * B + 255) / 256, 4096), 256, 0, s>>>(tr, steps, rows);
  EAZ_CHECK_LAUNCH("prio_seq_leaf_kernel");
  for (int l = 1; l < tr.L; ++l) {
    const int n_nodes = (int)((((int64_t)tr.N - 1) >> (5 * l)) + 1);
    // the host does not know the cursor: it launches enough warps for the widest placement of the touched leaves (two ranges
    // of rows * B leaves in all cover at most rows * B / 32^l + 4 nodes)
    const int warps = rows == T ? n_nodes : (int)std::min<int64_t>(n_nodes, ((int64_t)rows * B >> (5 * l)) + 4);
    const int wpb = std::min(warps, 8);  // warps per block
    prio_seq_level_kernel<<<ceil_div(warps, wpb), 32 * wpb, 0, s>>>(tr.hdr, tr.lvl[l - 1], tr.lvl[l], l, n_nodes, T, B, steps, rows);
    EAZ_CHECK_LAUNCH("prio_seq_level_kernel");
  }
  return 0;
}

int eaz_priority_status_async(const void* tree, size_t tree_bytes, int32_t* flags_dev, void* stream) {
  EAZ_CHECK_ARG(tree && tree_bytes >= sizeof(PrioHeader), "eaz_priority_status_async: NULL / short tree buffer");
  EAZ_CHECK_ARG(flags_dev != nullptr, "eaz_priority_status_async: NULL flags");
  if (cudaError_t e = cudaMemcpyAsync(flags_dev, (const uint8_t*)tree + offsetof(PrioHeader, status), sizeof(int32_t), cudaMemcpyDeviceToDevice,
                                      (cudaStream_t)stream);
      e != cudaSuccess)
    return cuda_fail(e, "eaz_priority_status_async copy");
  return 0;
}

int eaz_priority_status(const void* tree, size_t tree_bytes, void* stream, int32_t* flags_out) {
  EAZ_CHECK_ARG(tree && tree_bytes >= sizeof(PrioHeader), "eaz_priority_status: NULL / short tree buffer");
  if (flags_out) *flags_out = 0;
  if (cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream); e != cudaSuccess) return cuda_fail(e, "eaz_priority_status sync");
  uint32_t f = 0;
  if (cudaError_t e = cudaMemcpy(&f, (const uint8_t*)tree + offsetof(PrioHeader, status), sizeof(f), cudaMemcpyDeviceToHost); e != cudaSuccess)
    return cuda_fail(e, "eaz_priority_status read");
  if (flags_out) *flags_out = (int32_t)f;
  if (f) {
    set_error("eaz_priority_status: flags 0x%x (%s%s%s%s)", f, (f & EAZ_PRIORITY_BAD_PRIORITY) ? "negative / non-finite priority stored as 0; " : "",
              (f & EAZ_PRIORITY_BAD_INDEX) ? "out-of-range index skipped; " : "", (f & EAZ_PRIORITY_EMPTY) ? "sampled an empty tree; " : "",
              (f & EAZ_PRIORITY_BAD_ADD) ? "add_step slot out of order" : "");
    return EAZ_ERR_UNSUPPORTED;
  }
  return 0;
}

}  // extern "C"
