// TEST-ONLY host build of the alpha-beta search with repetitions on (chessrl_b200/csrc/ab_search.cuh ab_value<true>,
// crl_games_ab_search_host CRL_AB_REPETITIONS), compiled with g++ by tests/hostsim/ab_rep.py.  The same search, pick and
// window the kernels in kernels_ab.cu run, node counts included, so the CPU suite can check it against
// tests/ab_rep_oracle.py and the GPU suite can ask for the device's exact answer.  It is NOT part of libchessrl_b200.so
// and nothing under chessrl_b200/ loads it.
#include "../../chessrl_b200/csrc/ab_search.cuh"
#include <string.h>
using namespace crl;

static Board load(const uint64_t* rec) {
  Board b;
  memcpy(b.bb, rec, 64);
  b.meta = rec[8];
  return b;
}

extern "C" {

// crl_games_ab_search_host with CRL_AB_REPETITIONS for one lane: the picked root move (MOVE_NONE if the position is
// terminal), its score and the positions visited.  recs: n records in game order, the root last with the engine's ply and
// revlen in its meta; the window is the last min(revlen, ply) + 1 of them (k_ab_rep_stage's keys: each record's key as
// the game records it, en passant only if a capture is legal).  use_salt 0: the first best move.  -1 for limits out of
// range, -2 if fewer records than the window were given.
int hs_ab_rep(const uint64_t* recs, int n, int depth, int qdepth, int use_salt, int margin, int pick_plies,
              uint64_t salt, uint16_t* move, int32_t* score, uint64_t* nodes) {
  if (!ab_limits_ok(depth, qdepth) || !ab_pick_ok(margin, pick_plies)) return -1;
  if (n < 1) return -2;
  const Board root = load(recs + 9LL * (n - 1));
  int ngame = meta_revlen(root.meta);
  if (ngame > meta_ply(root.meta)) ngame = meta_ply(root.meta);
  if (ngame > AB_REP_KEYS - 1) ngame = AB_REP_KEYS - 1;
  if (ngame > n - 1) return -2;
  u64 game[AB_REP_KEYS];
  for (int i = 0; i <= ngame; ++i) {
    const Board b = load(recs + 9LL * (n - 1 - i));
    CountSink cs{0};
    game[i] = position_key(b, generate_legal(b, cs).ep_legal);
  }
  AbPath path;
  path.game = game;
  path.ngame = ngame;
  static thread_local AbStack st;
  u16 moves[MAX_MOVES];
  int scores[MAX_MOVES];
  StoreSink s{moves, 0};
  const GenInfo gi = generate_legal(root, s);
  *move = MOVE_NONE;
  *score = 0;
  *nodes = 1;
  if (ab_terminal(root, s.n, gi.in_check, 0, score)) return 0;
  unsigned long long total = 1;
  for (int k = 0; k < s.n; ++k) {
    unsigned long long nn = 0;
    scores[k] = ab_root_child<true>(st, root, moves[k], depth, qdepth, &nn, &path);
    total += nn;
  }
  const int k = ab_pick_index(scores, s.n, meta_ply(root.meta), use_salt ? margin : 0, pick_plies, salt);
  *move = moves[k];
  *score = scores[k];
  *nodes = total;
  return 0;
}

}  // extern "C"
