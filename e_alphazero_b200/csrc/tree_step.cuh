// tree_step.cuh -- the per-simulation tree kernel of the search (included by search.cu after the
// lane-group helpers).  ONE WARP PER TREE.  One launch does, for its tree:
//   1. expand  (mctx search.py expand / update_tree_node + the glue of context.py:132-154) for the leaf chosen
//              by the previous launch, using the network outputs;
//   2. backward (A.5) along the recorded path: lane l owns level l; the value / variance recurrences run as a
//              short uniform loop over levels (exact op order), the per-level running means (the divisions)
//              are computed by all levels in parallel;
//   3. action refresh: every node whose statistics just changed (the path + the new leaf) gets its NEXT action
//              selection recomputed NOW -- qtransform + seq-halving root score / interior score (A.3, A.6, A.7) --
//              32/G nodes at a time, G lanes per node, and cached in the node record together with the child it
//              leads to.  This is the same arithmetic on the same inputs the descent would evaluate, but all
//              levels are independent here, so they run in parallel instead of one after the other;
//   4. simulate (A.3) for the next simulation: a pure pointer chase over the cached (action, child) pairs,
//              recording the path;  [+ the DeepSea transition, context.py:127].
//
// Two code paths with identical arithmetic:
//   * STAGED (the common case, A <= 32): the kernel is launched programmatically (PDL) while the network kernel of
//     this simulation is still running.  Everything the steps above read EXCEPT the network outputs was written by
//     earlier tree / env kernels, which are complete by then (the network kernel triggers its dependents only
//     after its own grid-dependency wait).  So BEFORE griddepcontrol.wait the warp stages all of it -- path, node
//     and edge records of the path nodes, cached selections and compact states of every node -- in its slice of
//     shared memory (the wait invalidates L1, so an L1 prefetch would not survive: profiles/micro/pdl_l1.cu).
//     After the wait the only global loads on the critical path are the network outputs; the backward's edge
//     updates are patched into the staged copies in registers instead of being re-read from memory.
//   * DIRECT: load-as-you-go, used for A > 32, for the first launch of a search, and for paths longer than the
//     staging area.
#pragma once

namespace eaz {

// cached selection in NodeRec.pad0: bits 0..7 action, bits 8.. child index + 1 (0 = unvisited)
__device__ __forceinline__ int pack_next(int action, int child) { return action | ((child + 1) << 8); }
__device__ __forceinline__ uint32_t pack_next16(int packed) {  // NodeRec.pad0 (action | child + 1 << 8) -> 16 bits (action | child + 1 << 2), A <= 4
  return (uint32_t)(packed & 3) | ((uint32_t)(packed >> 8) << 2);
}

// gumbel_muzero_root_action_selection / gumbel_muzero_interior_action_selection for the lane group's node
// (mctx action_selection.py; SURVEY A.3, A.6, A.7).  Returns the selected action; *child = children_index[node, act].
template <int G, int J>
__device__ __forceinline__ int select_action(const Tree& t, const SearchParams& sp, const Edge<G, J>& e, const bool (&valid)[J], float raw,
                                             float raw_var, float beta, bool is_root, unsigned ub, unsigned uA,
                                             const uint8_t* __restrict__ invalid, int lane, int gl, int* child) {
  float cq[J];
  int sumN, maxN, act = 0;
  const bool use_beta = is_root || (sp.flags & EAZ_FLAG_BETA_INTERIOR) != 0;
  qtransform<G, J>(sp, e, valid, raw, raw_var, beta, use_beta, cq, sumN, maxN);
  if (__any_sync(0xffffffffu, is_root)) {  // gumbel_muzero_root_action_selection (node 0 is level 0 of round 0)
    float gum[J];
    bool inval[J];
    int num_valid = 0;
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const int a = gl + G * j;
      gum[j] = (is_root && valid[j]) ? t.gumbel[ub * uA + a] : 0.0f;
      inval[j] = (is_root && valid[j] && invalid) ? (invalid[ub * uA + a] != 0) : false;
      num_valid += (valid[j] && !inval[j]) ? 1 : 0;
    }
    num_valid = group_sum_i<G>(num_valid);
    const int num_considered = min(sp.max_considered, num_valid);
    const int considered_visit = is_root ? t.table[num_considered * sp.n + min(sumN, sp.n - 1)] : 0;
    act = root_argmax<G, J>(e, valid, gum, inval, cq, considered_visit, gl);
  }
  int act_i;
  {  // gumbel_muzero_interior_action_selection
    float x[J], p[J];
#pragma unroll
    for (int j = 0; j < J; ++j) x[j] = __fadd_rn(e.pl[j], cq[j]);
    group_softmax<G, J>(x, valid, p);
    const float den = (float)(1 + sumN);
    float best = -INFINITY;
    int besti = 1 << 30;
#pragma unroll
    for (int j = 0; j < J; ++j) {
      const float s = valid[j] ? __fsub_rn(p[j], __fdiv_rn((float)e.vis[j], den)) : -INFINITY;
      const int ia = valid[j] ? gl + G * j : (1 << 30);
      if (s > best || (s == best && ia < besti)) { best = s; besti = ia; }
    }
    act_i = group_argmax<G>(best, besti);
  }
  if (!is_root) act = act_i;
  // children_index[node, act]: owned by lane act % G of the group, slot act / G
  int ci_sel = -1;
#pragma unroll
  for (int j = 0; j < J; ++j)
    if (j == act / G) ci_sel = e.ci[j];
  *child = __shfl_sync(0xffffffffu, ci_sel, (lane & ~(G - 1)) + (act & (G - 1)));
  return act;
}

// STAGED path: the same selection with everything that does not depend on this simulation's network output precomputed
// before the grid-dependency wait: p = max(tiny, softmax(prior logits)) of the node (the priors of an expanded node never
// change) and, for the root, g2 = gumbel + (logit - max logit), the invalid flags and the considered-visit count.
// Identical operations in identical order to qtransform / root_argmax / select_action above (J == 1).
template <int G>
__device__ __forceinline__ int select_action_staged(const SearchParams& sp, const Edge<G, 1>& e, bool valid, float raw, float raw_var, float p,
                                                    float beta, bool is_root, float g2, bool inval, int considered_visit, int lane, int gl, int* child) {
  const bool use_beta = is_root || (sp.flags & EAZ_FLAG_BETA_INTERIOR) != 0;
  float q = __fadd_rn(e.rew[0], __fmul_rn(e.dis[0], e.val[0]));
  if (use_beta) {
    const float qv = __fadd_rn(0.0f, __fmul_rn(__fmul_rn(e.dis[0], e.dis[0]), e.vvar[0]));  // reward variance == 0 (context.py:149)
    q = __fadd_rn(q, __fmul_rn(beta, __fsqrt_rn(qv)));
  }
  const int sumN = group_sum_i<G>(valid ? e.vis[0] : 0);
  const int maxN = group_max_i<G>(valid ? e.vis[0] : 0);
  if (use_beta && (sp.flags & EAZ_FLAG_BETA_RAW)) raw = __fadd_rn(raw, __fmul_rn(beta, __fsqrt_rn(raw_var)));
  float value = raw;
  if (sp.mixed) {  // _compute_mixed_value with the staged prior probabilities
    const bool vis_on = valid && e.vis[0] > 0;
    const float sP = group_sum<G>(__fadd_rn(0.0f, vis_on ? p : 0.0f));
    const float wq = group_sum<G>(__fadd_rn(0.0f, vis_on ? __fdiv_rn(__fmul_rn(p, q), sP) : 0.0f));
    value = __fdiv_rn(__fadd_rn(raw, __fmul_rn((float)sumN, wq)), (float)(sumN + 1));
  }
  float c = e.vis[0] > 0 ? q : value;  // _complete_qvalues (reanalyze.py:32-40)
  if (sp.rescale) {                     // _rescale_qvalues
    const float lo = group_min<G>(valid ? c : INFINITY), hi = group_max<G>(valid ? c : -INFINITY);
    c = __fdiv_rn(__fsub_rn(c, lo), eaz_max(__fsub_rn(hi, lo), sp.epsilon));
  }
  const float cq = __fmul_rn(__fmul_rn(__fadd_rn(sp.maxvisit_init, (float)maxN), sp.value_scale), c);
  int act = 0;
  if (__any_sync(0xffffffffu, is_root)) {  // seq_halving.score_considered + masked_argmax on the staged root terms
    float sc = -INFINITY;
    if (is_root && valid) {
      sc = eaz_max(-1e9f, __fadd_rn(g2, cq));
      sc = __fadd_rn(sc, e.vis[0] == considered_visit ? 0.0f : -INFINITY);
      if (inval) sc = -INFINITY;
    }
    const int ia = valid ? gl : (1 << 30);
    float best = -INFINITY;
    int besti = 1 << 30;
    if (sc > best || (sc == best && ia < besti)) { best = sc; besti = ia; }
    act = group_argmax<G>(best, besti);
  }
  int act_i;
  {  // gumbel_muzero_interior_action_selection
    const float x = __fadd_rn(e.pl[0], cq);
    const float m = group_max<G>(valid ? x : -INFINITY);
    const float ex = valid ? eaz_exp(__fsub_rn(x, m)) : 0.0f;
    const float sm = group_sum<G>(__fadd_rn(0.0f, ex));
    const float pr = __fdiv_rn(ex, sm);
    const float sc = valid ? __fsub_rn(pr, __fdiv_rn((float)e.vis[0], (float)(1 + sumN))) : -INFINITY;
    const int ia = valid ? gl : (1 << 30);
    float best = -INFINITY;
    int besti = 1 << 30;
    if (sc > best || (sc == best && ia < besti)) { best = sc; besti = ia; }
    act_i = group_argmax<G>(best, besti);
  }
  if (!is_root) act = act_i;
  *child = __shfl_sync(0xffffffffu, e.ci[0], (lane & ~(G - 1)) + (act & (G - 1)));
  return act;
}

// DIRECT path: one warp, one tree, everything loaded as it is needed (also the reference implementation of the arithmetic that
// the STAGED paths reproduce from staged copies).
// ---------------------------------------------------------------------------------------------------------------------
// Subleq transition of the pending expansion, FUSED into the tree step (context.py:127 env.step -> subleq.py:648-677 -> run_tests
// :504-532 -> simulate :156-395): the warp that has just finished a tree's descent copies the parent's compact state into its
// scratch, writes the action into the program, lanes 0..2 interpret the three test cases (common.cuh: subleq_simulate with the exact
// loop shortcut), and the child state + reward go straight into the tree's workspace -- no separate launch, no second pass over
// the states.  Same steps as subleq_tree_step_kernel (search.cu), which stays as a measurement knob.
// scratch (per warp, 16-byte aligned): [state S bytes | 3 images | 3 snapshots | results]
__host__ __device__ inline int sq_warp_scratch_bytes(int ws) {
  const int S = EAZ_SQ_HDR + ((ws + 7) & ~7);
  return ((S + 15) & ~15) + ((6 * sq_img_stride(ws) + 15) & ~15) + 32;
}
__device__ __forceinline__ void subleq_expand_fused(const Tree& t, const EnvDesc& env, int b, int lane, int node, int action, int new_leaf,
                                                    uint8_t* scratch) {
  const int ws = env.ws, S = t.S;
  uint8_t* const st = scratch;                                // the state record being stepped
  uint8_t* const imgs = scratch + ((S + 15) & ~15);           // images 0..2, snapshots 3..5
  int* const res = reinterpret_cast<int*>(imgs + ((6 * sq_img_stride(ws) + 15) & ~15));  // [0..2] correct, [3..5] bytes used
  const uint8_t* ps = t.states + ((size_t)node * t.B + b) * S;
  for (int i = lane; i < S / 8; i += 32) reinterpret_cast<uint2*>(st)[i] = reinterpret_cast<const uint2*>(ps)[i];
  __syncwarp();
  int kd = 0;  // 0 absorbing, 1 terminate now, 2 execute
  if (lane == 0) {
    uint16_t* h = reinterpret_cast<uint16_t*>(st);
    const int flags = st[35];
    if (!(flags & (EAZ_SQ_FLAG_TERM | EAZ_SQ_FLAG_TRUNC))) {
      const int step = h[16] + 1;  // _step_count incremented before _step
      h[16] = (uint16_t)step;
      if (step >= ws - 3 || (flags & EAZ_SQ_FLAG_SOLVED)) {  // subleq.py:671-673
        kd = 1;
        st[35] = (uint8_t)(flags | EAZ_SQ_FLAG_TERM);
      } else {
        st[EAZ_SQ_HDR + step - 1] = (uint8_t)action;  // :654
        kd = 2;
      }
    }
  }
  kd = __shfl_sync(0xffffffffu, kd, 0);
  float reward = 0.0f;
  if (kd == 2) {  // (warp-uniform)
    __syncwarp();
    SubleqSim r;
    if (lane < 3) {
      const uint32_t* base = reinterpret_cast<const uint32_t*>(st + EAZ_SQ_HDR);
      if (ws == 16) {  // register-resident machine (common.cuh)
        subleq_simulate16<true>(sq_pack_nibbles16(base), sq_task_row(st[34]), lane, r);
      } else {
        const int stride = sq_img_stride(ws);
        uint8_t* img = imgs + lane * stride;
        uint8_t* snap = imgs + (3 + lane) * stride;
        for (int i = 0; i < (ws + 3) >> 2; ++i) {
          const uint32_t w = base[i];
          reinterpret_cast<uint32_t*>(img)[i] = w;
          reinterpret_cast<uint32_t*>(snap)[i] = w;
        }
        subleq_simulate<true>(ws, img, snap, sq_task_row(st[34]), lane, r);
      }
      res[lane] = r.correct;
      res[3 + lane] = r.bytes_used;
    }
    __syncwarp();
    if (lane == 0) {
      const int solved = res[0] & res[1] & res[2];
      const int bytes = max(res[3], max(res[4], res[5]));
      reward = subleq_reward(env.reward_fn, solved, bytes);
      uint16_t* h = reinterpret_cast<uint16_t*>(st);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        h[i] = (uint16_t)r.in[i];
        h[8 + i] = (uint16_t)r.out[i];
      }
      st[35] = (uint8_t)((st[35] & ~EAZ_SQ_FLAG_SOLVED) | (solved ? EAZ_SQ_FLAG_SOLVED : 0));
    }
  }
  __syncwarp();
  uint8_t* cs = t.states + ((size_t)new_leaf * t.B + b) * S;
  for (int i = lane; i < S / 8; i += 32) reinterpret_cast<uint2*>(cs)[i] = reinterpret_cast<const uint2*>(st)[i];
  if (lane == 0) t.reward[b] = reward;
  __syncwarp();
}

template <int G, int J>
__device__ __forceinline__ void tree_step_direct(const Tree& t, const SearchParams& sp, const EnvDesc& env, int sim, int do_backward, int do_select,
                                                 float beta, const uint8_t* __restrict__ invalid, int b, int lane, long long* trc,
                                                 uint8_t* sq_scratch = nullptr) {
  const unsigned uB = (unsigned)t.B, uA = (unsigned)t.A, ub = (unsigned)b;
  constexpr int kLevelsPerRound = 32 / G;
  const int gl = lane & (G - 1), glev = lane / G;
  bool valid[J];
#pragma unroll
  for (int j = 0; j < J; ++j) valid[j] = (gl + G * j) < t.A;
  int L = 0, leaf = 0;
  if (do_backward) {
    // ------------------------------------------------------------------ 1. expand
    leaf = t.leaf[b];
    L = t.path_len[b];
    const unsigned lslot = (unsigned)leaf * uB + ub;
    float m = -INFINITY;
    for (int a = lane; a < t.A; a += 32) m = fmaxf(m, t.net_logits[ub * uA + a]);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, s));  // context.py:135
    for (int a = lane; a < t.A; a += 32)
      t.edges[(size_t)(lslot * uA + a)].pl = __fsub_rn(t.net_logits[ub * uA + a], m);  // legal_action_mask is all True (:137)
    int term;
    if (env.kind == EAZ_ENV_DEEPSEA) term = EAZ_DS_TERM(reinterpret_cast<const uint32_t*>(t.states)[lslot]);
    else term = t.states[(size_t)lslot * t.S + 35] & EAZ_SQ_FLAG_TERM;
    const float value = term ? 0.0f : t.net_value[b];  // :140
    const float var = term ? 0.0f : t.net_ube[b];      // :141
    float disc = sp.discount;
    if (sp.two_players) disc = __fmul_rn(disc, -1.0f);  // :142-143
    if (term) disc = 0.0f;                              // :144
    const int2 last = t.path[(unsigned)(L - 1) * uB + ub];
    EdgeRec* pe0 = t.edges + (size_t)(((unsigned)last.x * uB + ub) * uA + (unsigned)last.y);
    if (lane == 0) {
      // update_tree_node: the leaf's record (visits + 1: a leaf can be re-expanded under a max_depth cut-off)
      uint4* ln = reinterpret_cast<uint4*>(t.nodes + lslot);
      const int old_visits = (int)ln[0].x;
      ln[0] = make_uint4((unsigned)(old_visits + 1), __float_as_uint(value), __float_as_uint(var), 0u);
      ln[1] = make_uint4(__float_as_uint(value), __float_as_uint(var), (unsigned)(last.x + 1), (unsigned)(last.y + 1));
      pe0->ci1 = leaf + 1;
      pe0->rew = t.reward[b];  // :139
      pe0->dis = disc;
    }
    __syncwarp();
    if (trc) trc[1] = clock64();

    // ------------------------------------------------------------------ 2. backward (levels L-1 .. 0)
    const bool std_backup = (sp.flags & EAZ_FLAG_BACKUP_STD) != 0;
    float lv = value, lvar = std_backup ? __fsqrt_rn(var) : var;  // running leaf_value / leaf variance (or std)
    float below_val = value, below_var = var;                     // updated mean / variance of the node one level deeper
    for (int hi = L; hi > 0; hi -= 32) {                          // rounds of 32 levels, deepest first
      const int lo = max(hi - 32, 0), cnt = hi - lo;
      const int lev = lo + lane;                                  // this lane's level
      const bool have = lane < cnt;
      int2 pa = make_int2(0, 0);
      uint4 nrec = make_uint4(0u, 0u, 0u, 0u);
      float rr = 0.0f, dd = 0.0f;
      int cvis = 0;
      unsigned pslot = 0;
      EdgeRec* pe = nullptr;
      if (have) {
        pa = t.path[(unsigned)lev * uB + ub];
        pslot = (unsigned)pa.x * uB + ub;
        pe = t.edges + (size_t)(pslot * uA + (unsigned)pa.y);
        nrec = reinterpret_cast<const uint4*>(t.nodes + pslot)[0];
        cvis = pe->vis;
        rr = pe->rew;
        dd = pe->dis;
      }
      // the recurrences: a uniform loop over this round's levels, deepest first, in the reference's op order
      float my_lv = 0.0f, my_lvar = 0.0f;
      for (int i = cnt - 1; i >= 0; --i) {
        const float r = __shfl_sync(0xffffffffu, rr, i), d = __shfl_sync(0xffffffffu, dd, i);
        lv = __fadd_rn(r, __fmul_rn(d, lv));
        lvar = std_backup ? __fadd_rn(0.0f, __fmul_rn(fabsf(d), lvar)) : __fadd_rn(0.0f, __fmul_rn(__fmul_rn(d, d), lvar));
        if (lane == i) { my_lv = lv; my_lvar = lvar; }
      }
      // running means, all levels in parallel
      const int nvis = (int)nrec.x;
      const float nval = __uint_as_float(nrec.y), nvar = __uint_as_float(nrec.z);
      const float count = (float)nvis;
      const float pv = __fdiv_rn(__fadd_rn(__fmul_rn(nval, count), my_lv), __fadd_rn(count, 1.0f));
      float pvar;
      if (std_backup) {
        const float ps = __fdiv_rn(__fadd_rn(__fmul_rn(__fsqrt_rn(nvar), count), my_lvar), __fadd_rn(count, 1.0f));
        pvar = __fmul_rn(ps, ps);
      } else {
        pvar = __fdiv_rn(__fadd_rn(__fmul_rn(nvar, count), my_lvar), __fadd_rn(count, 1.0f));
      }
      // children_values[parent, a] = the child's CURRENT (already updated) mean: one level deeper
      float cval = __shfl_down_sync(0xffffffffu, pv, 1), cvarr = __shfl_down_sync(0xffffffffu, pvar, 1);
      if (lane == cnt - 1) { cval = below_val; cvarr = below_var; }
      if (have) {
        reinterpret_cast<uint4*>(t.nodes + pslot)[0] = make_uint4((unsigned)(nvis + 1), __float_as_uint(pv), __float_as_uint(pvar), 0u);
        pe->vis = cvis + 1;
        *reinterpret_cast<float2*>(&pe->val) = make_float2(cval, cvarr);
      }
      below_val = __shfl_sync(0xffffffffu, pv, 0);
      below_var = __shfl_sync(0xffffffffu, pvar, 0);
    }
    __syncwarp();
    if (trc) { trc[2] = clock64(); trc[6] = L; }
  }
  if (!do_select) return;

  // -------------------------------------------------------------------- 3. refresh the cached selections
  // nodes: path levels 0..L-1 and the new leaf (index L); before the first simulation only the root.
  {
    const int nrefresh = do_backward ? L + 1 : 1;
    for (int base = 0; base < nrefresh; base += kLevelsPerRound) {
      const int lev = base + glev;
      const bool act_on = lev < nrefresh;
      int node = 0;
      if (act_on && do_backward) node = lev < L ? t.path[(unsigned)lev * uB + ub].x : leaf;
      const unsigned slot = (unsigned)node * uB + ub;
      Edge<G, J> e;
      float raw, raw_var;
      load_edges<G, J>(t, slot, gl, act_on, e);
      load_node_raw(t, slot, act_on, raw, raw_var);
      int child, act;
      if (sp.flags & EAZ_FLAG_PUCT) {  // muzero_action_selection at every depth (warp-uniform switch)
        const bool is_root = act_on && node == 0;
        uint4 h0 = make_uint4(0u, 0u, 0u, 0u);
        if (act_on) h0 = reinterpret_cast<const uint4*>(t.nodes + slot)[0];  // node_visits, node value, node variance
        bool inval[J];
#pragma unroll
        for (int j = 0; j < J; ++j) inval[j] = (is_root && valid[j] && invalid) ? (invalid[ub * uA + gl + G * j] != 0) : false;
        act = puct_select<G, J>(sp, e, valid, (int)h0.x, __uint_as_float(h0.y), __uint_as_float(h0.z), beta,
                                is_root || (sp.flags & EAZ_FLAG_BETA_INTERIOR) != 0, ub, (unsigned)node, inval, gl);
        int ci_sel = -1;
#pragma unroll
        for (int j = 0; j < J; ++j)
          if (j == act / G) ci_sel = e.ci[j];
        child = __shfl_sync(0xffffffffu, ci_sel, (lane & ~(G - 1)) + (act & (G - 1)));
      } else {
        act = select_action<G, J>(t, sp, e, valid, raw, raw_var, beta, act_on && node == 0, ub, uA, invalid, lane, gl, &child);
      }
      if (act_on && gl == 0) t.nodes[slot].pad0 = pack_next(act, child);
    }
    __syncwarp();
    if (trc) trc[3] = clock64();
  }

  // -------------------------------------------------------------------- 4. simulate: follow the cached selections
  // Nodes 0..sim exist.  For trees of up to 32*kChaseSlots nodes every cached (action, child) word is fetched once
  // (independent loads, lane i holds nodes i, i+32, ...) and the chase itself runs over registers with warp
  // shuffles; larger trees chase through memory, one dependent 16-byte load per level.
  constexpr int kChaseSlots = 9;
  int node = 0, depth = 0, action = 0, child = -1;
  if (sim < 32 * kChaseSlots) {
    int nxw[kChaseSlots];
#pragma unroll
    for (int s = 0; s < kChaseSlots; ++s) {
      const int nd = lane + 32 * s;
      nxw[s] = (32 * s <= sim && nd <= sim) ? t.nodes[(unsigned)nd * uB + ub].pad0 : 0;
    }
    while (true) {
      const int slot = node >> 5;
      int v = 0;
#pragma unroll
      for (int s = 0; s < kChaseSlots; ++s)
        if (s == slot) v = nxw[s];
      const int nx = __shfl_sync(0xffffffffu, v, node & 31);
      action = nx & 0xff;
      child = (nx >> 8) - 1;
      if (lane == 0) t.path[(unsigned)depth * uB + ub] = make_int2(node, action);
      depth += 1;
      if (child < 0 || depth >= sp.max_depth) break;
      node = child;
    }
  } else {
    while (true) {
      const int nx = t.nodes[(unsigned)node * uB + ub].pad0;
      action = nx & 0xff;
      child = (nx >> 8) - 1;
      if (lane == 0) t.path[(unsigned)depth * uB + ub] = make_int2(node, action);
      depth += 1;
      if (child < 0 || depth >= sp.max_depth) break;
      node = child;
    }
  }
  if (trc) { trc[4] = clock64(); trc[5] = depth; }
  if (lane == 0) {
    const int new_leaf = child < 0 ? sim + 1 : child;  // search.py: node first expanded on simulation i gets index i+1
    t.path_len[b] = depth;
    t.parent[b] = node;
    t.action[b] = action;
    t.leaf[b] = new_leaf;
    if (env.kind == EAZ_ENV_DEEPSEA) {  // context.py:127 env.step fused here
      uint32_t* st = reinterpret_cast<uint32_t*>(t.states);
      float reward;
      const uint32_t ns = deepsea_step(st[(unsigned)node * uB + ub], action, env.size, env.action_map, &reward);
      st[(unsigned)new_leaf * uB + ub] = ns;
      t.reward[b] = reward;
      t.cell[b] = deepsea_obs_index(ns, env.size);
    }
  }
  if (env.kind == EAZ_ENV_SUBLEQ && sq_scratch) subleq_expand_fused(t, env, b, lane, node, action, child < 0 ? sim + 1 : child, sq_scratch);
}

// Staging area of one warp (uint32 words); kRounds refresh rounds = kNodes nodes (path + leaf) fit.
template <int G>
struct Stage {
  static constexpr int kRounds = G == 2 ? 2 : 4;
  static constexpr int kNodes = kRounds * (32 / G);
  static constexpr int kLaneWords = 10;                 // ci1, vis, pl, rew, val, vvar, dis, raw, rawvar, prior probability
  static constexpr int kEdgeWords = kRounds * kLaneWords * 32;  // [round][word][lane]
  static constexpr int kBackWords = 4 * 32;            // [node | action << 16, visits, value, variance][level]
  static constexpr int kRootWords = 2 * 32;            // lanes 0..G-1: gumbel + (logit - max logit), invalid flag
  static constexpr int kMiscWords = 8;                  // term flag of the leaf, reward bits, root considered-visit
  static __host__ __device__ constexpr int words(int chase_cap) { return kEdgeWords + kBackWords + kRootWords + kMiscWords + 2 * chase_cap; }
};

template <int G, int J>
__global__ void __launch_bounds__(128, (G == 16 && J == 1) ? 8 : 1) tree_step_kernel(Tree t, SearchParams sp, EnvDesc env, int sim, int do_backward, int do_select,
                                                         const float* __restrict__ beta_in, const uint8_t* __restrict__ invalid,
                                                         unsigned long long* tl, long long* trace, int chase_cap, int* tile_done,
                                                         const int* mlp_done, int mlp_target, int sq_fused) {
  extern __shared__ __align__(16) uint32_t stage_smem[];
  // (Subleq, fused transition: per-warp interpreter scratch behind the four staging areas)
  uint8_t* const sq_scratch = sq_fused ? reinterpret_cast<uint8_t*>(stage_smem) + (chase_cap ? (size_t)4 * Stage<G>::words(chase_cap) * sizeof(uint32_t) : 0) +
                                             (size_t)(threadIdx.x >> 5) * sq_warp_scratch_bytes(env.ws)
                                       : nullptr;
  unsigned long long t_entry = 0;
  if (tl && blockIdx.x == 0 && threadIdx.x == 0) t_entry = globaltimer_ns();
  const int lane = threadIdx.x & 31;
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // one warp per tree
  const bool in_batch = b < t.B;                               // warp-uniform
  const unsigned uB = (unsigned)t.B, uA = (unsigned)t.A, ub = (unsigned)(in_batch ? b : 0);
  constexpr int kLevelsPerRound = 32 / G;
  const int gl = lane & (G - 1), glev = lane / G;
  bool valid[J];
#pragma unroll
  for (int j = 0; j < J; ++j) valid[j] = (gl + G * j) < t.A;

  // ==================================================================== staging (before the grid-dependency wait)
  using SG = Stage<G>;
  bool staged = false;
  int L = 0, leaf = 0;
  uint32_t* const sw = stage_smem + (threadIdx.x >> 5) * SG::words(chase_cap);
  uint32_t* const s_edge = sw;
  uint32_t* const s_back = sw + SG::kEdgeWords;
  uint32_t* const s_root = s_back + SG::kBackWords;
  uint32_t* const s_misc = s_root + SG::kRootWords;
  uint32_t* const s_next = s_misc + SG::kMiscWords;  // cached selection per node
  uint32_t* const s_state = s_next + chase_cap;      // DeepSea: compact state per node
  if constexpr (J == 1) {
    // Gumbel and PUCT selection alike refresh from the staged records; PUCT only for small action counts: its trees are deep, and with
    // 16 lanes per node the staging area holds 8 nodes -- most Subleq steps then fall back to DIRECT after paying for the staging
    // (measured, 4096 x 64 DeepSea-30: 1.29 ms staged vs 1.45 DIRECT; 8192 x 64 Subleq-16: 7.60 vs 6.34)
    if (in_batch && do_backward && chase_cap > sim + 1 && (!(sp.flags & EAZ_FLAG_PUCT) || G <= 4)) {
      leaf = t.leaf[b];
      L = t.path_len[b];
      const unsigned lslot = (unsigned)leaf * uB + ub;
      // (a leaf that already has visits is being re-expanded under a max_depth cut-off: its priors change -> DIRECT path)
      if (L + 1 <= SG::kNodes && L <= 32 && reinterpret_cast<const uint4*>(t.nodes + lslot)[0].x == 0u) {
        staged = true;
        int2 pa = make_int2(0, 0);  // backward operands, lane = level
        if (lane < L) pa = t.path[(unsigned)lane * uB + ub];
        if (lane < L) {
          const uint4 nrec = reinterpret_cast<const uint4*>(t.nodes + ((unsigned)pa.x * uB + ub))[0];
          s_back[0 * 32 + lane] = (uint32_t)pa.x | ((uint32_t)pa.y << 16);
          s_back[1 * 32 + lane] = nrec.x;
          s_back[2 * 32 + lane] = nrec.y;
          s_back[3 * 32 + lane] = nrec.z;
        }
        // refresh operands: group glev of round r holds entry r * kLevelsPerRound + glev of (path nodes..., leaf)
#pragma unroll
        for (int r = 0; r < SG::kRounds; ++r) {
          const int lev = r * kLevelsPerRound + glev;
          if (r * kLevelsPerRound <= L) {  // warp-uniform
            const int node = __shfl_sync(0xffffffffu, pa.x, lev & 31);
            const bool on = lev <= L && gl < t.A;
            uint4 h0 = make_uint4(0u, 0u, 0u, 0u), h1 = h0, n1 = h0;
            if (on) {
              const unsigned slot = (unsigned)(lev < L ? node : leaf) * uB + ub;
              const uint4* p = reinterpret_cast<const uint4*>(t.edges + (size_t)(slot * uA + (unsigned)gl));
              h0 = p[0];
              h1 = p[1];
              n1 = reinterpret_cast<const uint4*>(t.nodes + slot)[1];
            }
            // p = max(tiny, softmax(prior logits)) of _compute_mixed_value (the priors of an expanded node never change)
            const float xl[1] = {__uint_as_float(h0.z)};
            float pr[1];
            group_softmax<G, 1>(xl, valid, pr);
            if (on) {
              uint32_t* se = s_edge + r * SG::kLaneWords * 32 + lane;
              se[0 * 32] = h0.x; se[1 * 32] = h0.y; se[2 * 32] = h0.z; se[3 * 32] = h0.w;
              se[4 * 32] = h1.x; se[5 * 32] = h1.y; se[6 * 32] = h1.z;
              se[7 * 32] = n1.x; se[8 * 32] = n1.y;
              se[9 * 32] = __float_as_uint(eaz_max(EAZ_F32_TINY, pr[0]));
            }
            if (r == 0) {  // the root is level 0 of every path: its seq-halving score terms (mctx seq_halving.score_considered)
              const bool rt = glev == 0 && gl < t.A;
              const float gum = rt ? t.gumbel[ub * uA + gl] : 0.0f;
              const bool inval = rt && invalid && invalid[ub * uA + gl] != 0;
              const float m = group_max<G>(gl < t.A ? xl[0] : -INFINITY);
              const int num_valid = group_sum_i<G>((gl < t.A && !inval) ? 1 : 0);
              if (rt) {
                s_root[lane] = __float_as_uint(__fadd_rn(gum, __fsub_rn(xl[0], m)));
                s_root[32 + lane] = inval ? 1u : 0u;
              }
              if (lane == 0) s_misc[5] = (uint32_t)t.table[min(sp.max_considered, num_valid) * sp.n + min(sim, sp.n - 1)];
            }
          }
        }
        if (lane == 0) {
          s_misc[2] = env.kind == EAZ_ENV_DEEPSEA ? (uint32_t)EAZ_DS_TERM(reinterpret_cast<const uint32_t*>(t.states)[lslot])
                                                   : (uint32_t)(t.states[(size_t)lslot * t.S + 35] & EAZ_SQ_FLAG_TERM);
          s_misc[4] = __float_as_uint(t.reward[b]);
        }
        if (do_select) {  // every existing node's cached selection (and DeepSea state) for the descent
          for (int nd = lane; nd <= sim; nd += 32) {
            s_next[nd] = (uint32_t)t.nodes[(unsigned)nd * uB + ub].pad0;
            if (env.kind == EAZ_ENV_DEEPSEA) s_state[nd] = reinterpret_cast<const uint32_t*>(t.states)[(unsigned)nd * uB + ub];
          }
        }
      }
    }
    __syncwarp();
  }

  // the network outputs of this simulation: per-tile counters (the 3 head CTAs of this tree's tile) or the grid-wide PDL wait
  if (mlp_done && mlp_target > 0) {
    // (the 4 trees of a CTA belong to one tile: one polling thread per CTA)
    if (threadIdx.x == 0) wait_counter(mlp_done + (blockIdx.x * (blockDim.x >> 5)) / kTileRows, mlp_target);
    __syncthreads();
  } else {
    pdl_wait();
  }
  pdl_trigger();  // the next kernel (Subleq step / network) may begin its prologue now
  unsigned long long t_wait = 0;
  if (tl && blockIdx.x == 0 && threadIdx.x == 0) t_wait = globaltimer_ns();
  struct TlExit {  // records at every exit path of the first warp
    unsigned long long *tl, a, b;
    __device__ ~TlExit() {
      if (tl && blockIdx.x == 0 && threadIdx.x == 0) {
        const unsigned long long i = atomicAdd(tl, 1ull);
        if (i < 2000) { tl[8 + 4 * i] = a; tl[9 + 4 * i] = b; tl[10 + 4 * i] = globaltimer_ns(); tl[11 + 4 * i] = 0; }
      }
    }
  } tl_exit{tl, t_entry, t_wait};
  if (!in_batch) return;
  struct TileSignal {  // at every exit of the warp: results visible, then the tile's counter moves (consumed by the network kernel)
    int* ctr;
    int lane;
    __device__ ~TileSignal() {
      if (ctr) {
        __syncwarp();  // every lane's stores are ordered before lane 0's release fence (cumulative)
        if (lane == 0) signal_counter(ctr);
      }
    }
  } tile_signal{tile_done ? tile_done + b / kTileRows : nullptr, lane};
  // optional per-tree section stamps (eaz_debug_set_tree_trace): [sim][b][8] = start, expand, backward, refresh, chase, depth, L, staged
  long long* trc = (trace && lane == 0) ? trace + ((size_t)sim * t.B + b) * 8 : nullptr;
  if (trc) { trc[0] = clock64(); trc[7] = staged; }
  const float beta = beta_in ? beta_in[b] : 0.0f;

  if constexpr (J == 1) {
    if (staged) {
      // ================================================================ STAGED path (lane a holds action a's logit)
      const unsigned lslot = (unsigned)leaf * uB + ub;
      // ---- 1. expand
      const float lg = lane < t.A ? t.net_logits[ub * uA + lane] : -INFINITY;
      const float nv = t.net_value[b], nu = t.net_ube[b];
      float m = lg;
#pragma unroll
      for (int s = 16; s > 0; s >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, s));  // context.py:135
      const float pl_leaf = __fsub_rn(lg, m);                                              // legal_action_mask is all True (:137)
      if (lane < t.A) t.edges[(size_t)(lslot * uA + lane)].pl = pl_leaf;
      const int term = (int)s_misc[2];
      const float value = term ? 0.0f : nv;  // :140
      const float var = term ? 0.0f : nu;    // :141
      float disc = sp.discount;
      if (sp.two_players) disc = __fmul_rn(disc, -1.0f);  // :142-143
      if (term) disc = 0.0f;                              // :144
      const float reward = __uint_as_float(s_misc[4]);
      const uint32_t my_pa = lane < L ? s_back[lane] : 0u;
      const int my_node = (int)(my_pa & 0xffffu), my_act = (int)(my_pa >> 16);
      const int last_node = __shfl_sync(0xffffffffu, my_node, L - 1), last_act = __shfl_sync(0xffffffffu, my_act, L - 1);
      if (lane == 0) {
        // update_tree_node: the leaf's record (visits + 1: a leaf can be re-expanded under a max_depth cut-off)
        uint4* ln = reinterpret_cast<uint4*>(t.nodes + lslot);
        ln[0] = make_uint4(1u, __float_as_uint(value), __float_as_uint(var), 0u);  // a fresh leaf (staging condition)
        ln[1] = make_uint4(__float_as_uint(value), __float_as_uint(var), (unsigned)(last_node + 1), (unsigned)(last_act + 1));
        EdgeRec* pe0 = t.edges + (size_t)(((unsigned)last_node * uB + ub) * uA + (unsigned)last_act);
        pe0->ci1 = leaf + 1;
        pe0->rew = reward;  // :139
        pe0->dis = disc;
      }
      if (trc) trc[1] = clock64();

      // ---- 2. backward (levels L-1 .. 0) in one round: lane = level
      const bool std_backup = (sp.flags & EAZ_FLAG_BACKUP_STD) != 0;
      float lv = value, lvar = std_backup ? __fsqrt_rn(var) : var;
      const bool have = lane < L;
      int nvis = 0, cvis = 0;
      float nval = 0.0f, nvar = 0.0f, rr = 0.0f, dd = 0.0f;
      if (have) {
        nvis = (int)s_back[32 + lane];
        nval = __uint_as_float(s_back[64 + lane]);
        nvar = __uint_as_float(s_back[96 + lane]);
        // the traversed edge (level, action) sits in the refresh staging: round level / kLPR, group level % kLPR, lane action
        const uint32_t* se = s_edge + (lane / kLevelsPerRound) * SG::kLaneWords * 32 + (lane % kLevelsPerRound) * G + my_act;
        cvis = (int)se[1 * 32];
        rr = __uint_as_float(se[3 * 32]);
        dd = __uint_as_float(se[6 * 32]);
        if (lane == L - 1) { rr = reward; dd = disc; }  // written by the expand step above
      }
      float my_lv = 0.0f, my_lvar = 0.0f;
      for (int i = L - 1; i >= 0; --i) {  // the recurrences, deepest level first, in the reference's op order
        const float r = __shfl_sync(0xffffffffu, rr, i), d = __shfl_sync(0xffffffffu, dd, i);
        lv = __fadd_rn(r, __fmul_rn(d, lv));
        lvar = std_backup ? __fadd_rn(0.0f, __fmul_rn(fabsf(d), lvar)) : __fadd_rn(0.0f, __fmul_rn(__fmul_rn(d, d), lvar));
        if (lane == i) { my_lv = lv; my_lvar = lvar; }
      }
      const float count = (float)nvis;
      const float pv = __fdiv_rn(__fadd_rn(__fmul_rn(nval, count), my_lv), __fadd_rn(count, 1.0f));
      float pvar;
      if (std_backup) {
        const float ps = __fdiv_rn(__fadd_rn(__fmul_rn(__fsqrt_rn(nvar), count), my_lvar), __fadd_rn(count, 1.0f));
        pvar = __fmul_rn(ps, ps);
      } else {
        pvar = __fdiv_rn(__fadd_rn(__fmul_rn(nvar, count), my_lvar), __fadd_rn(count, 1.0f));
      }
      // children_values[parent, a] = the child's CURRENT (already updated) mean: one level deeper
      float cval = __shfl_down_sync(0xffffffffu, pv, 1), cvarr = __shfl_down_sync(0xffffffffu, pvar, 1);
      if (lane == L - 1) { cval = value; cvarr = var; }
      if (have) {
        const unsigned pslot = (unsigned)my_node * uB + ub;
        EdgeRec* pe = t.edges + (size_t)(pslot * uA + (unsigned)my_act);
        reinterpret_cast<uint4*>(t.nodes + pslot)[0] = make_uint4((unsigned)(nvis + 1), __float_as_uint(pv), __float_as_uint(pvar), 0u);
        pe->vis = cvis + 1;
        *reinterpret_cast<float2*>(&pe->val) = make_float2(cval, cvarr);
      }
      if (trc) { trc[2] = clock64(); trc[6] = L; }
      if (!do_select) return;

      // ---- 3. refresh the cached selections of the path nodes and the leaf: staged records + this backward's updates
#pragma unroll
      for (int r = 0; r < SG::kRounds; ++r) {
        if (r * kLevelsPerRound > L) break;  // warp-uniform
        const int lev = r * kLevelsPerRound + glev;
        const bool act_on = lev <= L;
        const int src = lev & 31;  // the lane that owned level `lev` in the backward
        const int node_l = __shfl_sync(0xffffffffu, my_node, src), act_l = __shfl_sync(0xffffffffu, my_act, src);
        const float cval_l = __shfl_sync(0xffffffffu, cval, src), cvar_l = __shfl_sync(0xffffffffu, cvarr, src);
        const float pl_l = __shfl_sync(0xffffffffu, pl_leaf, gl);
        const int node = act_on ? (lev < L ? node_l : leaf) : 0;
        Edge<G, 1> e;
        e.ci[0] = -1; e.vis[0] = 0;
        e.pl[0] = 0.0f; e.rew[0] = 0.0f; e.dis[0] = 0.0f; e.val[0] = 0.0f; e.vvar[0] = 0.0f;
        float raw = 0.0f, raw_var = 0.0f, prior_p = 0.0f;
        if (act_on) {
          const uint32_t* sg0 = s_edge + r * SG::kLaneWords * 32 + (lane & ~(G - 1));  // the group's action-0 lane always holds raw / raw variance
          raw = __uint_as_float(sg0[7 * 32]);
          raw_var = __uint_as_float(sg0[8 * 32]);
          if (lev == L) { raw = value; raw_var = var; }  // the leaf: fresh raw values
          if (gl < t.A) {
            const uint32_t* se = s_edge + r * SG::kLaneWords * 32 + lane;
            e.ci[0] = (int)se[0] - 1;
            e.vis[0] = (int)se[1 * 32];
            e.pl[0] = __uint_as_float(se[2 * 32]);
            e.rew[0] = __uint_as_float(se[3 * 32]);
            e.val[0] = __uint_as_float(se[4 * 32]);
            e.vvar[0] = __uint_as_float(se[5 * 32]);
            e.dis[0] = __uint_as_float(se[6 * 32]);
            prior_p = __uint_as_float(se[9 * 32]);  // (unused for the fresh leaf: none of its children has visits)
            if (lev == L) {
              e.pl[0] = pl_l;  // fresh priors
            } else if (gl == act_l) {  // the edge this simulation went through
              e.vis[0] += 1;
              e.val[0] = cval_l;
              e.vvar[0] = cvar_l;
              if (lev == L - 1) { e.ci[0] = leaf; e.rew[0] = reward; e.dis[0] = disc; }
            }
          }
        }
        const bool is_root = act_on && node == 0;
        float g2 = 0.0f;
        bool inval = false;
        int considered_visit = 0;
        if (r == 0 && is_root && gl < t.A) {
          g2 = __uint_as_float(s_root[lane]);
          inval = s_root[32 + lane] != 0u;
          considered_visit = (int)s_misc[5];
        }
        int child, act;
        if (sp.flags & EAZ_FLAG_PUCT) {
          // muzero_action_selection (puct_select, search.cu) on the same staged + patched edge records; the node's own statistics after
          // this backward: visits + 1 / new mean / new variance of the path level's owner lane, or the fresh leaf's (1, value, var)
          const int nvis_l = __shfl_sync(0xffffffffu, nvis, src);
          const float pv_l = __shfl_sync(0xffffffffu, pv, src), pvar_l = __shfl_sync(0xffffffffu, pvar, src);
          const int n_vis = lev < L ? nvis_l + 1 : 1;
          const float n_val = lev < L ? pv_l : value, n_var = lev < L ? pvar_l : var;
          const bool inv1[1] = {r == 0 && is_root && gl < t.A && s_root[32 + lane] != 0u};
          act = puct_select<G, 1>(sp, e, valid, n_vis, n_val, n_var, beta, is_root || (sp.flags & EAZ_FLAG_BETA_INTERIOR) != 0, ub, (unsigned)node, inv1, gl);
          child = __shfl_sync(0xffffffffu, e.ci[0], (lane & ~(G - 1)) + (act & (G - 1)));
        } else {
          act = select_action_staged<G>(sp, e, valid[0], raw, raw_var, prior_p, beta, is_root, g2, inval, considered_visit, lane, gl, &child);
        }
        if (act_on && gl == 0) {
          const int packed = pack_next(act, child);
          t.nodes[(unsigned)node * uB + ub].pad0 = packed;
          s_next[node] = (uint32_t)packed;
        }
      }
      __syncwarp();
      if (trc) trc[3] = clock64();

      // ---- 4. simulate: follow the cached selections through the staged copy
      int node = 0, depth = 0, action = 0, child = -1;
      while (true) {
        const int nx = (int)s_next[node];
        action = nx & 0xff;
        child = (nx >> 8) - 1;
        if (lane == 0) t.path[(unsigned)depth * uB + ub] = make_int2(node, action);
        depth += 1;
        if (child < 0 || depth >= sp.max_depth) break;
        node = child;
      }
      if (trc) { trc[4] = clock64(); trc[5] = depth; }
      if (lane == 0) {
        const int new_leaf = child < 0 ? sim + 1 : child;  // search.py: node first expanded on simulation i gets index i+1
        t.path_len[b] = depth;
        t.parent[b] = node;
        t.action[b] = action;
        t.leaf[b] = new_leaf;
        if (env.kind == EAZ_ENV_DEEPSEA) {  // context.py:127 env.step fused here
          uint32_t* st = reinterpret_cast<uint32_t*>(t.states);
          float rw;
          const uint32_t ns = deepsea_step(s_state[node], action, env.size, env.action_map, &rw);
          st[(unsigned)new_leaf * uB + ub] = ns;
          t.reward[b] = rw;
          t.cell[b] = deepsea_obs_index(ns, env.size);
        }
      }
      if (env.kind == EAZ_ENV_SUBLEQ && sq_scratch) subleq_expand_fused(t, env, b, lane, node, action, child < 0 ? sim + 1 : child, sq_scratch);
      return;
    }
  }

  // ==================================================================== DIRECT path
  tree_step_direct<G, J>(t, sp, env, sim, do_backward, do_select, beta, invalid, b, lane, trc, sq_scratch);
}

// ======================================================================================================================
// Two trees per warp (16 lanes each) for small action counts (G lanes per node, G <= 4): the one-tree kernel keeps a handful
// of its 32 lanes busy -- the path is a few levels deep and a node has G actions -- and is bound by warp-instruction issue
// (1 421 warp instructions per tree at C2), so halving the warps nearly halves its cost.  Same STAGED scheme and the same
// arithmetic as tree_step_kernel; per tree the staging area holds 32 nodes (path + leaf) in rounds of 16 / G.  If either
// tree of a pair cannot be staged (first launch, path longer than 31, re-expanded leaf, PUCT) both take the DIRECT path,
// one after the other, with the whole warp.
//
// The staged step of one tree of a pair -- expand, backward, refresh (staged2_* below) -- is also the step of the persistent
// DeepSea search (psearch.cuh: ds_search_kernel).  The two staging areas share the layout these functions read and write:
//   edges  [round][word][lane of the tree]: in round r, node group glev = hl / G of the tree holds entry r * 16 / G + glev of
//          (path nodes..., leaf) and lane gl = hl % G its action gl, in the ten words of staged2_store_lane;
//   back   [node | action << 16, visits -> child value, value -> child variance, variance][level], levels 0..31;
//   misc   [8 + a]: the fresh leaf's prior logits.
// They differ in the number of rounds, in where the root's score terms are kept and in the width of the cached selections.
constexpr int kStaged2Lanes = 16;          // lanes per tree
constexpr int kStaged2LaneWords = 10;      // ci1, vis, pl, rew, val, vvar, dis, raw, rawvar, prior probability
constexpr int kStaged2BackWords = 4 * 32;  // [node | action << 16, visits -> child value, value -> child variance, variance][level]

template <int G>
struct Stage2 {
  static constexpr int kPerRound = kStaged2Lanes / G;  // nodes refreshed per round
  static constexpr int kRounds = 32 / kPerRound;       // 32 nodes (path + leaf) fit
  static constexpr int kEdgeWords = kRounds * kStaged2LaneWords * kStaged2Lanes;
  static constexpr int kRootWords = 2 * kStaged2Lanes;  // lanes 0..G-1: gumbel + (logit - max logit), invalid flag
  static constexpr int kMiscWords = 16;                 // [2] leaf terminal, [4] reward, [5] considered visit, [8..8+G) leaf priors
  static __host__ __device__ constexpr int words(int chase_cap) { return kEdgeWords + kStaged2BackWords + kRootWords + kMiscWords + 2 * chase_cap; }
};

// A lane of one tree of the pair: its coordinates, the tree's workspace column and its staging area
struct Staged2Lane {
  int lane, hl, hbase, gl, glev;  // lane of the warp, lane of the tree, the tree's first lane, action and node group of the lane
  bool valid, in_batch;           // action gl exists (gl < A); the tree is in the batch
  unsigned uB, uA, ub;            // batch, actions, the tree's column (0 outside the batch)
  uint32_t *s_edge, *s_back, *s_misc;
};
// The expansion of one simulation: path length, leaf, the reward into the leaf, and what staged2_expand derives from the leaf's
// network outputs: value, variance and the discount of the edge into the leaf
struct Staged2Leaf {
  int L, leaf;
  float reward, value, var, disc;
};

// the ten-word record of one staged (node, action) lane in round r: the edge record's ci1, vis, pl, rew (h0) and val, vvar, dis (h1),
// the node's raw value and variance (n1.x, n1.y) and p = max(tiny, softmax of the node's prior logits)
__device__ __forceinline__ void staged2_store_lane(uint32_t* s_edge, int r, int hl, uint4 h0, uint4 h1, uint4 n1, float p) {
  constexpr int kW = kStaged2Lanes;
  uint32_t* se = s_edge + r * kStaged2LaneWords * kW + hl;
  se[0 * kW] = h0.x; se[1 * kW] = h0.y; se[2 * kW] = h0.z; se[3 * kW] = h0.w;
  se[4 * kW] = h1.x; se[5 * kW] = h1.y; se[6 * kW] = h1.z;
  se[7 * kW] = n1.x; se[8 * kW] = n1.y;
  se[9 * kW] = __float_as_uint(eaz_max(EAZ_F32_TINY, p));
}

// ---- 1. expand the fresh leaf at the end of a path of L levels: lane a of the tree holds action a's logit lg (A <= G, -inf on the
// other lanes), nv / nu the leaf's value and UBE.  Writes the leaf's prior logits (edge records and s_misc[8 + a]), its node record and
// the edge into it.
template <int G>
__device__ __forceinline__ Staged2Leaf staged2_expand(const Tree& t, const SearchParams& sp, const Staged2Lane& w, int L, int leaf, float reward,
                                                      float lg, float nv, float nu, bool term) {
  const unsigned lslot = (unsigned)leaf * w.uB + w.ub;
  // context.py:135: the max over the logit lanes (all in the node group of the tree's first lane; fmaxf with -inf is exact)
  const float m = __shfl_sync(0xffffffffu, group_max<G>(lg), w.hbase);
  const float pl_leaf = __fsub_rn(lg, m);  // legal_action_mask is all True (:137)
  if (w.in_batch && w.hl < t.A) {
    t.edges[(size_t)(lslot * w.uA + w.hl)].pl = pl_leaf;
    w.s_misc[8 + w.hl] = __float_as_uint(pl_leaf);
  }
  Staged2Leaf f{L, leaf, reward};
  f.value = term ? 0.0f : nv;  // :140
  f.var = term ? 0.0f : nu;    // :141
  f.disc = sp.discount;
  if (sp.two_players) f.disc = __fmul_rn(f.disc, -1.0f);  // :142-143
  if (term) f.disc = 0.0f;                                // :144
  if (w.in_batch && w.hl == 0) {
    const uint32_t last = w.s_back[L - 1];
    const int last_node = (int)(last & 0xffffu), last_act = (int)(last >> 16);
    uint4* ln = reinterpret_cast<uint4*>(t.nodes + lslot);  // update_tree_node: a fresh leaf (staging condition)
    ln[0] = make_uint4(1u, __float_as_uint(f.value), __float_as_uint(f.var), 0u);
    ln[1] = make_uint4(__float_as_uint(f.value), __float_as_uint(f.var), (unsigned)(last_node + 1), (unsigned)(last_act + 1));
    EdgeRec* pe0 = t.edges + (size_t)(((unsigned)last_node * w.uB + w.ub) * w.uA + (unsigned)last_act);
    pe0->ci1 = leaf + 1;
    pe0->rew = reward;  // :139
    pe0->dis = f.disc;
  }
  return f;
}

// ---- 2. backward: rounds of 16 levels, deepest first; lane = level within the round.  std_backup: EAZ_FLAG_BACKUP_STD.  Leaves each
// traversed edge's new child value / variance in s_back[32 / 64 + level] for the refresh.
template <int G>
__device__ __forceinline__ void staged2_backward(const Tree& t, const Staged2Lane& w, const Staged2Leaf& f, bool std_backup) {
  constexpr int kW = kStaged2Lanes, kPR = kW / G;
  const int L = f.L, hl = w.hl, hbase = w.hbase;
  uint32_t* const s_back = w.s_back;
  float lv = f.value, lvar = std_backup ? __fsqrt_rn(f.var) : f.var;
  float below_val = f.value, below_var = f.var;
  const int Lw = max(L, __shfl_xor_sync(0xffffffffu, L, kW));
#pragma unroll 1
  for (int k = Lw > kW ? 1 : 0; k >= 0; --k) {
    const int lo = kW * k, cnt = min(max(L - lo, 0), kW);
    const int lev = lo + hl;
    const bool have = w.in_batch && hl < cnt;
    int my_node = 0, my_act = 0, nvis = 0, cvis = 0;
    float nval = 0.0f, nvar = 0.0f, rr = 0.0f, dd = 0.0f;
    if (have) {
      const uint32_t pa = s_back[lev];
      my_node = (int)(pa & 0xffffu);
      my_act = (int)(pa >> 16);
      nvis = (int)s_back[32 + lev];
      nval = __uint_as_float(s_back[64 + lev]);
      nvar = __uint_as_float(s_back[96 + lev]);
      const uint32_t* se = w.s_edge + (lev / kPR) * kStaged2LaneWords * kW + (lev % kPR) * G + my_act;  // the traversed edge in the refresh staging
      cvis = (int)se[1 * kW];
      rr = __uint_as_float(se[3 * kW]);
      dd = __uint_as_float(se[6 * kW]);
      if (lev == L - 1) { rr = f.reward; dd = f.disc; }  // written by the expand step
    }
    const int cmax = max(cnt, __shfl_xor_sync(0xffffffffu, cnt, kW));
    float my_lv = 0.0f, my_lvar = 0.0f;
    for (int i = cmax - 1; i >= 0; --i) {  // the recurrences, in the reference's op order
      const float r = __shfl_sync(0xffffffffu, rr, hbase + i), d = __shfl_sync(0xffffffffu, dd, hbase + i);
      if (i < cnt) {
        lv = __fadd_rn(r, __fmul_rn(d, lv));
        lvar = std_backup ? __fadd_rn(0.0f, __fmul_rn(fabsf(d), lvar)) : __fadd_rn(0.0f, __fmul_rn(__fmul_rn(d, d), lvar));
        if (hl == i) { my_lv = lv; my_lvar = lvar; }
      }
    }
    const float count = (float)nvis;
    const float pv = __fdiv_rn(__fadd_rn(__fmul_rn(nval, count), my_lv), __fadd_rn(count, 1.0f));
    float pvar;
    if (std_backup) {
      const float psd = __fdiv_rn(__fadd_rn(__fmul_rn(__fsqrt_rn(nvar), count), my_lvar), __fadd_rn(count, 1.0f));
      pvar = __fmul_rn(psd, psd);
    } else {
      pvar = __fdiv_rn(__fadd_rn(__fmul_rn(nvar, count), my_lvar), __fadd_rn(count, 1.0f));
    }
    // children_values[parent, a] = the child's CURRENT (already updated) mean: one level deeper
    float cval = __shfl_down_sync(0xffffffffu, pv, 1, kW), cvarr = __shfl_down_sync(0xffffffffu, pvar, 1, kW);
    if (hl == cnt - 1) { cval = below_val; cvarr = below_var; }
    if (have) {
      const unsigned pslot = (unsigned)my_node * w.uB + w.ub;
      EdgeRec* pe = t.edges + (size_t)(pslot * w.uA + (unsigned)my_act);
      reinterpret_cast<uint4*>(t.nodes + pslot)[0] = make_uint4((unsigned)(nvis + 1), __float_as_uint(pv), __float_as_uint(pvar), 0u);
      pe->vis = cvis + 1;
      *reinterpret_cast<float2*>(&pe->val) = make_float2(cval, cvarr);
      s_back[32 + lev] = __float_as_uint(cval);  // for the refresh: the traversed edge's new child value / variance
      s_back[64 + lev] = __float_as_uint(cvarr);
    }
    const float b0v = __shfl_sync(0xffffffffu, pv, hbase), b0r = __shfl_sync(0xffffffffu, pvar, hbase);
    if (cnt > 0) { below_val = b0v; below_var = b0r; }
  }
  __syncwarp();
}

// ---- 3. refresh the cached selections of the path nodes and the leaf: staged records + this backward's updates.  The root's score
// terms: root_g2[a] = gumbel + (logit - max logit), root_inval[a] its invalid flag, *considered the seq-halving visit target.  The
// selection is cached in the node record and in s_next[node]: 32 bits as NodeRec.pad0, or 16 bits (pack_next16).
template <int G, typename NextT>
__device__ __forceinline__ void staged2_refresh(const Tree& t, const SearchParams& sp, const Staged2Lane& w, const Staged2Leaf& f, float beta,
                                                const uint32_t* root_g2, const uint32_t* root_inval, const uint32_t* considered, NextT* s_next) {
  constexpr int kW = kStaged2Lanes, kPR = kW / G;
  const int L = f.L, hl = w.hl, gl = w.gl;
  const uint32_t* const s_back = w.s_back;
  const int rounds = w.in_batch ? (L + kPR) / kPR : 0;  // ceil((L + 1) / kPR)
  const int rmax = max(rounds, __shfl_xor_sync(0xffffffffu, rounds, kW));
#pragma unroll 1
  for (int r = 0; r < rmax; ++r) {
    const int lev = r * kPR + w.glev;
    const bool act_on = w.in_batch && lev <= L;
    int node = 0, act_l = 0;
    float cval_l = 0.0f, cvar_l = 0.0f;
    if (act_on && lev < L) {
      const uint32_t pa = s_back[lev];
      node = (int)(pa & 0xffffu);
      act_l = (int)(pa >> 16);
      cval_l = __uint_as_float(s_back[32 + lev]);
      cvar_l = __uint_as_float(s_back[64 + lev]);
    } else if (act_on) {
      node = f.leaf;
    }
    Edge<G, 1> e;
    e.ci[0] = -1; e.vis[0] = 0;
    e.pl[0] = 0.0f; e.rew[0] = 0.0f; e.dis[0] = 0.0f; e.val[0] = 0.0f; e.vvar[0] = 0.0f;
    float raw = 0.0f, raw_var = 0.0f, prior_p = 0.0f;
    if (act_on) {
      const uint32_t* sg0 = w.s_edge + r * kStaged2LaneWords * kW + (hl & ~(G - 1));  // the group's action-0 lane always holds raw / raw variance
      raw = __uint_as_float(sg0[7 * kW]);
      raw_var = __uint_as_float(sg0[8 * kW]);
      if (lev == L) { raw = f.value; raw_var = f.var; }  // the leaf: fresh raw values
      if (gl < t.A) {
        const uint32_t* se = w.s_edge + r * kStaged2LaneWords * kW + hl;
        e.ci[0] = (int)se[0] - 1;
        e.vis[0] = (int)se[1 * kW];
        e.pl[0] = __uint_as_float(se[2 * kW]);
        e.rew[0] = __uint_as_float(se[3 * kW]);
        e.val[0] = __uint_as_float(se[4 * kW]);
        e.vvar[0] = __uint_as_float(se[5 * kW]);
        e.dis[0] = __uint_as_float(se[6 * kW]);
        prior_p = __uint_as_float(se[9 * kW]);  // (unused for the fresh leaf: none of its children has visits)
        if (lev == L) {
          e.pl[0] = __uint_as_float(w.s_misc[8 + gl]);  // fresh priors
        } else if (gl == act_l) {  // the edge this simulation went through
          e.vis[0] += 1;
          e.val[0] = cval_l;
          e.vvar[0] = cvar_l;
          if (lev == L - 1) { e.ci[0] = f.leaf; e.rew[0] = f.reward; e.dis[0] = f.disc; }
        }
      }
    }
    const bool is_root = act_on && node == 0;  // (only at level 0: lane gl of the tree's first node group)
    float g2 = 0.0f;
    bool inval = false;
    int considered_visit = 0;
    if (r == 0 && is_root && gl < t.A) {
      g2 = __uint_as_float(root_g2[gl]);
      inval = root_inval[gl] != 0u;
      considered_visit = (int)*considered;
    }
    int child;
    const int act = select_action_staged<G>(sp, e, w.valid, raw, raw_var, prior_p, beta, is_root, g2, inval, considered_visit, w.lane, gl, &child);
    if (act_on && gl == 0) {
      const int packed = pack_next(act, child);
      t.nodes[(unsigned)node * w.uB + w.ub].pad0 = packed;
      if constexpr (sizeof(NextT) == 2) s_next[node] = (NextT)pack_next16(packed);
      else s_next[node] = (NextT)packed;
    }
  }
  __syncwarp();
}

template <int G>
__global__ void __launch_bounds__(128) tree_step2_kernel(Tree t, SearchParams sp, EnvDesc env, int sim, int do_backward, int do_select,
                                                          const float* __restrict__ beta_in, const uint8_t* __restrict__ invalid,
                                                          unsigned long long* tl, long long* trace, int chase_cap) {
  extern __shared__ __align__(16) uint32_t stage_smem[];
  unsigned long long t_entry = 0;
  if (tl && blockIdx.x == 0 && threadIdx.x == 0) t_entry = globaltimer_ns();
  using SG = Stage2<G>;
  constexpr int kW = kStaged2Lanes, kPR = SG::kPerRound;
  const int lane = threadIdx.x & 31, hl = lane & (kW - 1), hbase = lane & kW, sub = lane >> 4;
  const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int b = 2 * warp_global + sub;  // 16 lanes per tree
  const bool in_batch = b < t.B;
  const unsigned uB = (unsigned)t.B, uA = (unsigned)t.A, ub = (unsigned)(in_batch ? b : 0);
  const int gl = hl & (G - 1), glev = hl / G;
  const bool valid1[1] = {gl < t.A};
  uint32_t* const sw = stage_smem + ((threadIdx.x >> 5) * 2 + sub) * SG::words(chase_cap);
  uint32_t* const s_edge = sw;
  uint32_t* const s_back = sw + SG::kEdgeWords;
  uint32_t* const s_root = s_back + kStaged2BackWords;
  uint32_t* const s_misc = s_root + SG::kRootWords;
  uint32_t* const s_next = s_misc + SG::kMiscWords;
  uint32_t* const s_state = s_next + chase_cap;

  // ==================================================================== staging (before the grid-dependency wait)
  bool staged = false;
  int L = 0, leaf = 0;
  if (do_backward && chase_cap > sim + 1 && !(sp.flags & EAZ_FLAG_PUCT)) {  // warp-uniform
    bool ok = true;
    if (in_batch) {
      leaf = t.leaf[b];
      L = t.path_len[b];
      ok = L + 1 <= 32 && reinterpret_cast<const uint4*>(t.nodes + ((unsigned)leaf * uB + ub))[0].x == 0u;  // fits, and the leaf is fresh
    }
    if (__all_sync(0xffffffffu, ok)) {
      staged = true;
      const unsigned lslot = (unsigned)leaf * uB + ub;
      if (in_batch) {  // backward operands: this lane owns levels hl and hl + 16
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const int lev = hl + kW * k;
          if (lev < L) {
            const int2 pa = t.path[(unsigned)lev * uB + ub];
            const uint4 nrec = reinterpret_cast<const uint4*>(t.nodes + ((unsigned)pa.x * uB + ub))[0];
            s_back[0 * 32 + lev] = (uint32_t)pa.x | ((uint32_t)pa.y << 16);
            s_back[1 * 32 + lev] = nrec.x;
            s_back[2 * 32 + lev] = nrec.y;
            s_back[3 * 32 + lev] = nrec.z;
          }
        }
      }
      __syncwarp();
      const int Lw = max(L, __shfl_xor_sync(0xffffffffu, L, kW));
#pragma unroll
      for (int r = 0; r < SG::kRounds; ++r) {
        if (r * kPR <= Lw) {  // warp-uniform
          const int lev = r * kPR + glev;
          const bool on = in_batch && lev <= L && gl < t.A;
          uint4 h0 = make_uint4(0u, 0u, 0u, 0u), h1 = h0, n1 = h0;
          if (on) {
            const int node = lev < L ? (int)(s_back[lev] & 0xffffu) : leaf;
            const unsigned slot = (unsigned)node * uB + ub;
            const uint4* p = reinterpret_cast<const uint4*>(t.edges + (size_t)(slot * uA + (unsigned)gl));
            h0 = p[0];
            h1 = p[1];
            n1 = reinterpret_cast<const uint4*>(t.nodes + slot)[1];
          }
          const float xl[1] = {__uint_as_float(h0.z)};
          float pr[1];
          group_softmax<G, 1>(xl, valid1, pr);  // p = max(tiny, softmax(prior logits)) of _compute_mixed_value
          if (on) staged2_store_lane(s_edge, r, hl, h0, h1, n1, pr[0]);
          if (r == 0) {  // the root is level 0 of every path: its seq-halving score terms
            const bool rt = in_batch && glev == 0 && gl < t.A;
            const float gum = rt ? t.gumbel[ub * uA + gl] : 0.0f;
            const bool inval = rt && invalid && invalid[ub * uA + gl] != 0;
            const float m = group_max<G>(gl < t.A ? xl[0] : -INFINITY);
            const int num_valid = group_sum_i<G>((gl < t.A && !inval) ? 1 : 0);
            if (rt) {
              s_root[hl] = __float_as_uint(__fadd_rn(gum, __fsub_rn(xl[0], m)));
              s_root[kW + hl] = inval ? 1u : 0u;
            }
            if (in_batch && hl == 0) s_misc[5] = (uint32_t)t.table[min(sp.max_considered, num_valid) * sp.n + min(sim, sp.n - 1)];
          }
        }
      }
      if (in_batch && hl == 0) {
        s_misc[2] = env.kind == EAZ_ENV_DEEPSEA ? (uint32_t)EAZ_DS_TERM(reinterpret_cast<const uint32_t*>(t.states)[lslot])
                                                 : (uint32_t)(t.states[(size_t)lslot * t.S + 35] & EAZ_SQ_FLAG_TERM);
        s_misc[4] = __float_as_uint(t.reward[b]);
      }
      if (do_select && in_batch) {
        for (int nd = hl; nd <= sim; nd += kW) {
          s_next[nd] = (uint32_t)t.nodes[(unsigned)nd * uB + ub].pad0;
          if (env.kind == EAZ_ENV_DEEPSEA) s_state[nd] = reinterpret_cast<const uint32_t*>(t.states)[(unsigned)nd * uB + ub];
        }
      }
    }
  }
  __syncwarp();

  pdl_wait();     // the network kernel of this simulation has finished: its outputs are visible
  pdl_trigger();  // the next kernel may begin its prologue now
  unsigned long long t_wait = 0;
  if (tl && blockIdx.x == 0 && threadIdx.x == 0) t_wait = globaltimer_ns();
  struct TlExit {
    unsigned long long *tl, a, b;
    __device__ ~TlExit() {
      if (tl && blockIdx.x == 0 && threadIdx.x == 0) {
        const unsigned long long i = atomicAdd(tl, 1ull);
        if (i < 2000) { tl[8 + 4 * i] = a; tl[9 + 4 * i] = b; tl[10 + 4 * i] = globaltimer_ns(); tl[11 + 4 * i] = 0; }
      }
    }
  } tl_exit{tl, t_entry, t_wait};

  if (!staged) {  // both trees through the DIRECT path, one after the other, with the whole warp
#pragma unroll 1
    for (int s2 = 0; s2 < 2; ++s2) {
      const int bb = 2 * warp_global + s2;
      if (bb < t.B)
        tree_step_direct<G, 1>(t, sp, env, sim, do_backward, do_select, beta_in ? beta_in[bb] : 0.0f, invalid, bb, lane,
                               (trace && lane == 0) ? trace + ((size_t)sim * t.B + bb) * 8 : nullptr);
      __syncwarp();
    }
    return;
  }

  // ==================================================================== STAGED path, 16 lanes per tree
  long long* trc = (trace && hl == 0 && in_batch) ? trace + ((size_t)sim * t.B + b) * 8 : nullptr;
  if (trc) { trc[0] = clock64(); trc[7] = 2; }
  const float beta = (in_batch && beta_in) ? beta_in[b] : 0.0f;
  const Staged2Lane w{lane, hl, hbase, gl, glev, valid1[0], in_batch, uB, uA, ub, s_edge, s_back, s_misc};
  // ---- 1. expand (lane a of the tree holds action a's logit), 2. backward, 3. refresh
  const float lg = (in_batch && hl < t.A) ? t.net_logits[ub * uA + hl] : -INFINITY;
  const Staged2Leaf f = staged2_expand<G>(t, sp, w, L, leaf, in_batch ? __uint_as_float(s_misc[4]) : 0.0f, lg, in_batch ? t.net_value[b] : 0.0f,
                                          in_batch ? t.net_ube[b] : 0.0f, in_batch && s_misc[2] != 0u);
  if (trc) trc[1] = clock64();
  staged2_backward<G>(t, w, f, (sp.flags & EAZ_FLAG_BACKUP_STD) != 0);
  if (trc) { trc[2] = clock64(); trc[6] = L; }
  if (!do_select) return;
  staged2_refresh<G>(t, sp, w, f, beta, s_root, s_root + kStaged2Lanes, s_misc + 5, s_next);
  if (trc) trc[3] = clock64();

  // ---- 4. simulate: follow the cached selections through the staged copy (each tree until its own descent ends)
  int node = 0, depth = 0, action = 0, child = -1;
  bool active = in_batch;
  while (__any_sync(0xffffffffu, active)) {
    if (active) {
      const int nx = (int)s_next[node];
      action = nx & 0xff;
      child = (nx >> 8) - 1;
      if (hl == 0) t.path[(unsigned)depth * uB + ub] = make_int2(node, action);
      depth += 1;
      if (child < 0 || depth >= sp.max_depth) active = false;
      else node = child;
    }
  }
  if (trc) { trc[4] = clock64(); trc[5] = depth; }
  if (in_batch && hl == 0) {
    const int new_leaf = child < 0 ? sim + 1 : child;  // search.py: node first expanded on simulation i gets index i+1
    t.path_len[b] = depth;
    t.parent[b] = node;
    t.action[b] = action;
    t.leaf[b] = new_leaf;
    if (env.kind == EAZ_ENV_DEEPSEA) {  // context.py:127 env.step fused here
      uint32_t* st = reinterpret_cast<uint32_t*>(t.states);
      float rw;
      const uint32_t ns = deepsea_step(s_state[node], action, env.size, env.action_map, &rw);
      st[(unsigned)new_leaf * uB + ub] = ns;
      t.reward[b] = rw;
      t.cell[b] = deepsea_obs_index(ns, env.size);
    }
  }
}

}  // namespace eaz
