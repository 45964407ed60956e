// TEST-ONLY host build of the seeded near-best root pick (chessrl_b200/csrc/ab_search.cuh ab_pick_index, DESIGN.md 3.7),
// compiled with g++ by tests/hostsim/ab_pick.py.  The same search and pick code that kernels_ab.cu runs for
// crl_games_ab_pick_host, so the CPU suite can check it against oracle/ab_pick_oracle.py and the GPU suite can ask for
// the device's exact answer.  It is NOT part of libchessrl_b200.so and nothing under chessrl_b200/ loads it.
#include "../../chessrl_b200/csrc/ab_search.cuh"
#include <string.h>
using namespace crl;

extern "C" {

// crl_games_ab_pick_host for one position: the picked root move (MOVE_NONE if the position is terminal), its score and
// the positions visited (the root and every root child's subtree); the ply is the record's.  -1 for depth / qdepth /
// margin / pick_plies out of range.
int hs_ab_pick(const uint64_t* rec, int depth, int qdepth, int margin, int pick_plies, uint64_t salt, uint16_t* move,
               int32_t* score, uint64_t* nodes) {
  if (!ab_limits_ok(depth, qdepth) || !ab_pick_ok(margin, pick_plies)) return -1;
  static thread_local AbStack st;
  Board root;
  memcpy(root.bb, rec, 64);
  root.meta = rec[8];
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
    scores[k] = ab_root_child(st, root, moves[k], depth, qdepth, &nn);
    total += nn;
  }
  const int k = ab_pick_index(scores, s.n, meta_ply(root.meta), margin, pick_plies, salt);
  *move = moves[k];
  *score = scores[k];
  *nodes = total;
  return 0;
}

}  // extern "C"
