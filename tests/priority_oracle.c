/*
 * priority_oracle.c -- CPU ORACLE of the prioritised replay sum tree (TEST INFRASTRUCTURE, NOT PRODUCT CODE).
 *
 * A plain-C restatement of e_alphazero_b200/csrc/replay.cu in the same operation order, checked bit for bit against it by
 * tests/test_gpu_replay_priority.py.  It is one translation unit with the search oracle (oracle/eaz_oracle.c is included
 * below) so that the node sums are orc_tree_sum and the random stream is orc_xx_round, the very functions the search oracle
 * uses.  The buffer has the byte layout of the device buffer, so tests compare the two whole buffers.
 *
 * THE CONTRACT (the same text heads csrc/replay.cu; both must change together)
 *
 *   Items.  Item i = t * B + b is the pair (slot t, slot (t + 1) % T) of env b.  t is the PHYSICAL ring slot, so an index
 *     is an opaque handle, as flashbax's are.  An item is VALID only when both of its slots hold data and slot t + 1 is not
 *     the slot written next (slot s holds data iff (cursor - 1 - s) mod T < length).  An invalid item has weight 0.
 *   Weights.  w(p) = eaz_exp(eaz_mul(alpha, eaz_log(p))) for 0 < p <= FLT_MAX, w = 0 for p == 0 (also at alpha = 0).
 *     A negative or non-finite p is stored as 0 and sets EAZ_PRIORITY_BAD_PRIORITY.
 *   Buffer (eaz_priority_tree_bytes).  [0, 32): header {float alpha; uint32 seed; uint32 draw_ctr; uint32 status;
 *     int32 cursor; int32 length; float max_priority (raw p, starts at 1); uint32 0}; [256, ...): int32 tag[N] (-1 between
 *     calls: the duplicate resolution of eaz_priority_set), then the fp32 levels, leaves first: n_0 = N = T * B,
 *     n_{l+1} = ceil(n_l / 32) down to n_{L-1} = 1.  Every region starts at a multiple of 128 bytes and each level is
 *     padded with zeros to a multiple of 32 floats.
 *   Node sums.  Node j of level l + 1 = orc_tree_sum of the 32 children 32 j .. 32 j + 31 of level l (child c in lane c,
 *     xor-butterfly with strides 1, 2, 4, 8, 16; a missing child is 0).  A node is always recomputed from its children,
 *     never updated by a delta, so the tree is a pure function of the leaves.
 *   add_step(c).  If c == cursor: cursor = (c + 1) % T, length = min(length + 1, T); if c == cursor - 1 (the newest slot
 *     was rewritten) cursor and length stay; any other c sets EAZ_PRIORITY_BAD_ADD and changes nothing.  Then the items of
 *     row c - 1 get w(max_priority) if length >= 2 (else 0) and the items of row c get 0.
 *   set(indices[K], priorities[K]).  An index outside [0, N) sets EAZ_PRIORITY_BAD_INDEX and is skipped.  For a duplicated
 *     index the LAST occurrence in the batch wins.  The leaf becomes w(p) if the item is valid, else 0.  max_priority =
 *     max(max_priority, p of every in-range entry).
 *   sample(K).  total = the root.  Sample k: r_k = 24 bits of h * 2^-24 with h = seed + 0x9E3779B1; h = xx_round(h,
 *     draw_ctr); h = xx_round(h, k); then the xxhash avalanche (>>15, *P2, >>13, *P3, >>16), r_k = (h >> 8) * 2^-24;
 *     u = eaz_mul(eaz_div(eaz_add((float)k, r_k), (float)K), total).  Descent from the root: over the 32 children w_0..w_31
 *     of the current node, prefix_c = ((0 + w_0) + w_1) + ... + w_c (serial, ascending); pick the first c with prefix_c > u
 *     and w_c > 0; if none, the last c with w_c > 0; then u = eaz_sub(u, prefix_{c-1}) (0 for c = 0).  At the leaf:
 *     index i, probability = eaz_div(w_i, total).  The draw counter advances once per call.  total == 0 (or not finite)
 *     sets EAZ_PRIORITY_EMPTY and every sample is index 0, probability 0.
 */
#include "../oracle/eaz_oracle.c"

#include <float.h>

typedef struct {
  float alpha;
  uint32_t seed;
  uint32_t draw_ctr;
  uint32_t status;
  int32_t cursor;
  int32_t length;
  float max_priority;
  uint32_t reserved;
} prio_header;

#define PRIO_MAX_LEVELS 8

typedef struct {
  prio_header* hdr;
  int32_t* tag;
  float* lvl[PRIO_MAX_LEVELS];
  int n[PRIO_MAX_LEVELS];
  int L, T, B, N;
  size_t bytes;
} prio_tree;

static size_t prio_align128(size_t x) { return (x + 127) / 128 * 128; }

/* layout only (buf may be NULL): returns the byte size, 0 for invalid T, B */
static size_t prio_layout(uint8_t* buf, int T, int B, prio_tree* tr) {
  if (T < 2 || B < 1 || (int64_t)T * B >= ((int64_t)1 << 31)) return 0;
  tr->T = T, tr->B = B, tr->N = T * B;
  tr->hdr = (prio_header*)buf;
  tr->tag = (int32_t*)(buf ? buf + 256 : NULL);
  size_t off = prio_align128(256 + (size_t)tr->N * 4);
  int n = tr->N, L = 0;
  for (;;) {
    tr->n[L] = n;
    tr->lvl[L] = buf ? (float*)(buf + off) : NULL;
    off += prio_align128((size_t)(n + 31) / 32 * 32 * 4);
    ++L;
    if (n == 1) break;
    n = (n + 31) / 32;
  }
  tr->L = L;
  tr->bytes = off;
  return off;
}

static float prio_weight(float p, float alpha) { return p > 0.0f ? eaz_exp(eaz_mul(alpha, eaz_log(p))) : 0.0f; }
static int prio_bad(float p) { return !(p >= 0.0f && p <= FLT_MAX); }
static float prio_clean(float p) { return (p > 0.0f && p <= FLT_MAX) ? p : 0.0f; }

static int prio_filled(int s, int T, int cursor, int length) {
  int a = cursor - 1 - s;
  if (a < 0) a += T;
  return a < length;
}
static int prio_valid(int t, int T, int cursor, int length) {
  const int t1 = t + 1 == T ? 0 : t + 1;
  return t1 != cursor && prio_filled(t, T, cursor, length) && prio_filled(t1, T, cursor, length);
}

/* every inner node from its children (the tree is a pure function of the leaves, so this equals recomputing the touched
 * ancestors only) */
static void prio_rebuild(prio_tree* tr) {
  for (int l = 1; l < tr->L; ++l)
    for (int j = 0; j < tr->n[l]; ++j) tr->lvl[l][j] = orc_tree_sum(tr->lvl[l - 1] + (size_t)32 * j, 32); /* pads are 0 */
}

size_t orc_priority_tree_bytes(int32_t T, int32_t B) {
  prio_tree tr;
  return prio_layout(NULL, T, B, &tr);
}

int orc_priority_init(uint8_t* buf, int32_t T, int32_t B, float alpha, uint32_t seed) {
  prio_tree tr;
  const size_t bytes = prio_layout(buf, T, B, &tr);
  if (!bytes || !(alpha >= 0.0f && alpha <= 1.0f)) return EAZ_ERR_INVALID_ARG;
  memset(buf, 0, bytes);
  memset(tr.tag, 0xff, (size_t)tr.N * 4);
  prio_header h = {alpha, seed, 0u, 0u, 0, 0, 1.0f, 0u};
  *tr.hdr = h;
  return 0;
}

int orc_priority_add_step(uint8_t* buf, int32_t T, int32_t B, int32_t c) {
  prio_tree tr;
  if (!prio_layout(buf, T, B, &tr) || c < 0 || c >= T) return EAZ_ERR_INVALID_ARG;
  prio_header* h = tr.hdr;
  if (c == h->cursor) {
    h->cursor = c + 1 == T ? 0 : c + 1;
    h->length = h->length + 1 < T ? h->length + 1 : T;
  } else if (c != (h->cursor == 0 ? T - 1 : h->cursor - 1)) {
    h->status |= EAZ_PRIORITY_BAD_ADD;
    return 0;
  }
  const float w = h->length >= 2 ? prio_weight(h->max_priority, h->alpha) : 0.0f;
  const int rp = c == 0 ? T - 1 : c - 1;
  for (int b = 0; b < B; ++b) {
    tr.lvl[0][(size_t)rp * B + b] = w;
    tr.lvl[0][(size_t)c * B + b] = 0.0f;
  }
  prio_rebuild(&tr);
  return 0;
}

int orc_priority_set(uint8_t* buf, int32_t T, int32_t B, const int32_t* idx, const float* pri, int32_t K) {
  prio_tree tr;
  if (!prio_layout(buf, T, B, &tr) || K < 0) return EAZ_ERR_INVALID_ARG;
  prio_header* h = tr.hdr;
  for (int k = 0; k < K; ++k) { /* ascending k: the last occurrence of an index is written last */
    const int i = idx[k];
    if (prio_bad(pri[k])) h->status |= EAZ_PRIORITY_BAD_PRIORITY;
    if (i < 0 || i >= tr.N) {
      h->status |= EAZ_PRIORITY_BAD_INDEX;
      continue;
    }
    const float p = prio_clean(pri[k]);
    if (p > h->max_priority) h->max_priority = p;
    tr.lvl[0][i] = prio_valid(i / B, T, h->cursor, h->length) ? prio_weight(p, h->alpha) : 0.0f;
  }
  prio_rebuild(&tr);
  return 0;
}

static float prio_uniform(uint32_t seed, uint32_t ctr, uint32_t k) {
  uint32_t h = seed + 0x9E3779B1u;
  h = orc_xx_round(h, ctr);
  h = orc_xx_round(h, k);
  h ^= h >> 15; h *= 0x85EBCA77u; h ^= h >> 13; h *= 0xC2B2AE3Du; h ^= h >> 16;
  return eaz_mul((float)(h >> 8), 5.9604644775390625e-08f);
}

/* the descent of one sample from u (exported for the boundary tests); returns the leaf index, or -1 on an empty tree */
int orc_priority_descend(const uint8_t* buf, int32_t T, int32_t B, float u) {
  prio_tree tr;
  if (!prio_layout((uint8_t*)buf, T, B, &tr)) return EAZ_ERR_INVALID_ARG;
  const float total = tr.lvl[tr.L - 1][0];
  if (!(total > 0.0f && total <= FLT_MAX)) return -1;
  int j = 0;
  for (int l = tr.L - 1; l >= 1; --l) {
    const float* w = tr.lvl[l - 1] + (size_t)32 * j;
    float pre[32], acc = 0.0f;
    for (int c = 0; c < 32; ++c) pre[c] = acc = eaz_add(acc, w[c]);
    int pick = -1, last = 0;
    for (int c = 0; c < 32; ++c) {
      if (w[c] > 0.0f) last = c;
      if (pick < 0 && pre[c] > u && w[c] > 0.0f) pick = c;
    }
    if (pick < 0) pick = last;
    u = eaz_sub(u, pick == 0 ? 0.0f : pre[pick - 1]);
    j = 32 * j + pick;
  }
  return j;
}

int orc_priority_sample(uint8_t* buf, int32_t T, int32_t B, int32_t K, const uint8_t* states, const float* rewards, int32_t S,
                        int32_t* indices, float* probabilities, uint8_t* first, float* first_r, uint8_t* second, float* second_r) {
  prio_tree tr;
  if (!prio_layout(buf, T, B, &tr) || K < 1 || K > (1 << 24)) return EAZ_ERR_INVALID_ARG;
  prio_header* h = tr.hdr;
  const float total = tr.lvl[tr.L - 1][0];
  const int empty = !(total > 0.0f && total <= FLT_MAX);
  if (empty) h->status |= EAZ_PRIORITY_EMPTY;
  for (int k = 0; k < K; ++k) {
    int i = 0;
    float prob = 0.0f;
    if (!empty) {
      const float u = eaz_mul(eaz_div(eaz_add((float)k, prio_uniform(h->seed, h->draw_ctr, (uint32_t)k)), (float)K), total);
      i = orc_priority_descend(buf, T, B, u);
      prob = eaz_div(tr.lvl[0][i], total);
    }
    indices[k] = i;
    probabilities[k] = prob;
    if (states) {
      const int t = i / B, b = i - t * B, t1 = t + 1 == T ? 0 : t + 1;
      const size_t r0 = (size_t)t * B + b, r1 = (size_t)t1 * B + b;
      memcpy(first + (size_t)k * S, states + r0 * S, (size_t)S);
      memcpy(second + (size_t)k * S, states + r1 * S, (size_t)S);
      if (rewards) first_r[k] = rewards[r0], second_r[k] = rewards[r1];
    }
  }
  h->draw_ctr += 1u;
  return 0;
}
