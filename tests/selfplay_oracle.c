/*
 * selfplay_oracle.c -- CPU ORACLE of the optional parts of the self-play step (TEST INFRASTRUCTURE, NOT PRODUCT CODE).
 *
 * A plain-C restatement of what csrc/search.cu adds for eaz_search_config.root_prior / action_sampling, checked bit for bit against
 * it by tests/test_gpu_selfplay_options.py.  One translation unit with the search oracle (oracle/eaz_oracle.c is included below) so
 * that the arithmetic is eaz_math.h's and the random stream is orc_xx_round, the very functions the search oracle uses.
 *
 *   Uniform root prior: the search of oracle/eaz_oracle.c on prior_logits = 0 (its _mask_invalid_actions then gives 0 / EAZ_F32_MIN)
 *     with the caller's or the network's root value / UBE; nothing here.
 *   The draw (orc_sample_actions): per row, x_a = eaz_log(max(w_a, tiny)) with w = visit_probs (EAZ_ACTION_VISITS) or action_weights
 *     (EAZ_ACTION_IMPROVED), m = max_a x_a, the action is the first argmax of (x_a - m) / max(tiny, temperature) + g_a with
 *     invalid actions at -inf (a row with every action invalid plays 0).
 *   The in-kernel noise (orc_stream_gumbel): h = seed + 0x9E3779B1, xx rounds by the draw counter, the tree (including the batch
 *     offset of an EAZ_FLAG_STREAMS sub-batch) and the action, one more by 0x53414D50 for the noise of the draw (not for the root
 *     noise), the xxhash avalanche, u = ((h >> 8) + 0.5) * 2^-24, g = -log(-log(u)).
 */
#include "../oracle/eaz_oracle.c"

float orc_stream_gumbel(uint32_t seed, uint32_t ctr, uint32_t tree, uint32_t a, int32_t sample) {
  uint32_t h = seed + 0x9E3779B1u;
  h = orc_xx_round(h, ctr);
  h = orc_xx_round(h, tree);
  h = orc_xx_round(h, a);
  if (sample) h = orc_xx_round(h, 0x53414D50u);
  h ^= h >> 15; h *= 0x85EBCA77u; h ^= h >> 13; h *= 0xC2B2AE3Du; h ^= h >> 16;
  const float u = eaz_mul(eaz_add((float)(h >> 8), 0.5f), 5.9604644775390625e-08f);
  return -eaz_log(-eaz_log(u));
}

/* g [B,A] of trees tree0 .. tree0 + B - 1 */
void orc_stream_gumbel_rows(uint32_t seed, uint32_t ctr, int32_t tree0, int32_t B, int32_t A, int32_t sample, float* g) {
  for (int b = 0; b < B; ++b)
    for (int a = 0; a < A; ++a) g[(size_t)b * A + a] = orc_stream_gumbel(seed, ctr, (uint32_t)(tree0 + b), (uint32_t)a, sample);
}

int orc_sample_actions(const float* w, const uint8_t* invalid, const float* g, int32_t B, int32_t A, float temperature, int32_t* action) {
  if (A < 1 || A > ORC_MAX_A) return EAZ_ERR_INVALID_ARG;
  float x[ORC_MAX_A];
  const float tdiv = eaz_max(EAZ_F32_TINY, temperature);
  for (int b = 0; b < B; ++b) {
    const size_t o = (size_t)b * A;
    for (int a = 0; a < A; ++a) x[a] = eaz_log(eaz_max(w[o + a], EAZ_F32_TINY));
    const float m = orc_maxv(x, A);
    for (int a = 0; a < A; ++a) x[a] = (invalid && invalid[o + a]) ? -INFINITY : eaz_add(eaz_div(eaz_sub(x[a], m), tdiv), g[o + a]);
    action[b] = orc_argmax(x, A);
  }
  return 0;
}
