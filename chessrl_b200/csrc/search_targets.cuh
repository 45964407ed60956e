// search_targets.cuh -- training targets from the alpha-beta root scores (crl_search_targets, DESIGN.md 3.8).
//
// For a position p with side to move c, legal moves m_0..m_{n-1} in generation order and root scores s_0..s_{n-1}
// (centipawns for c, +-(32000 - h) for mates), best = max_k s_k:
//   policy  pi_k = exp((s_k - best) / T) / sum_j exp((s_j - best) / T) in fp32, at the label index of m_k; every other
//           entry of the 1,968 is 0
//   value   v_s = tanh(best / 400) from white's point of view (negated when c is black)
// The sum runs in generation order, so a row's bits depend on its own inputs only.  Every function is CRL_HD: the
// TEST-ONLY g++ build (tests/hostsim/search_targets_hostsim.cpp) compiles this same code.
#pragma once
#include <math.h>
#include "../../include/chessrl_b200.h"
#include "chess_core.cuh"

namespace crl {

static constexpr float SEARCH_VALUE_SCALE = 400.0f;   // centipawns; a fixed constant of the definition

struct SearchRowStats {
  int best;
  float sum;   // sum_j exp((s_j - best) / T), in generation order
};

CRL_HD SearchRowStats search_row_stats(const int* s, int n, float temperature) {
  int best = s[0];
  for (int k = 1; k < n; ++k) best = s[k] > best ? s[k] : best;
  float sum = 0.0f;
  for (int k = 0; k < n; ++k) sum += expf((float)(s[k] - best) / temperature);
  return SearchRowStats{best, sum};
}

CRL_HD float search_prob(int s, const SearchRowStats& r, float temperature) {
  return expf((float)(s - r.best) / temperature) / r.sum;
}

CRL_HD float search_score_value(int best, int white_to_move) {
  const float v = tanhf((float)best / SEARCH_VALUE_SCALE);
  return white_to_move ? v : -v;
}

// label index of a move word (netencoder.get_uci_labels order), -1 if it has none
CRL_HD int search_label(const int16_t* label_of, u16 m) {
  return mv_promo(m) < 5 ? (int)label_of[(int)mv_promo(m) * 4096 + mv_from(m) * 64 + mv_to(m)] : -1;
}

// The whole row on one thread (the host build; the kernel splits the same steps over a block): regenerates b's legal
// moves into `moves` [MAX_MOVES], and when their count equals n_scores (> 0) writes the dense policy row [CRL_N_LABELS]
// and v_s.  Otherwise the row is all zeros and v_s is 0.  Returns the legal count.
CRL_HD int search_targets_row(const Board& b, const int* s, int n_scores, float temperature, const int16_t* label_of,
                              u16* moves, float* policy_row, float* score_value) {
  StoreSink sink{moves, 0};
  generate_legal(b, sink);
  for (int l = 0; l < CRL_N_LABELS; ++l) policy_row[l] = 0.0f;
  *score_value = 0.0f;
  if (sink.n != n_scores || sink.n == 0) return sink.n;
  const SearchRowStats r = search_row_stats(s, sink.n, temperature);
  for (int k = 0; k < sink.n; ++k) {
    const int l = search_label(label_of, moves[k]);
    if (l >= 0) policy_row[l] = search_prob(s[k], r, temperature);
  }
  *score_value = search_score_value(r.best, meta_turn(b.meta));
  return sink.n;
}

}  // namespace crl
