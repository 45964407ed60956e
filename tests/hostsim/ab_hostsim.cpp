// TEST-ONLY host build of chessrl_b200/csrc/ab_search.cuh (compiled with g++ by tests/hostsim/ab.py).
// The same search code the kernels in kernels_ab.cu run, root split and reduction included, so the CPU suite can check
// it against oracle/ab_oracle.py and the GPU suite can ask for the device's exact node counts.  It is NOT part of
// libchessrl_b200.so and nothing under chessrl_b200/ loads it.
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

int hs_ab_eval(const uint64_t* rec) { return ab_evaluate(load(rec)); }

// crl_games_ab_move_host for one position: the first best root move (MOVE_NONE if the position is terminal), its
// score and the positions visited (the root and every root child's subtree).  -1 for depth / qdepth out of range.
int hs_ab_root(const uint64_t* rec, int depth, int qdepth, uint16_t* move, int32_t* score, uint64_t* nodes) {
  if (!ab_limits_ok(depth, qdepth)) return -1;
  static thread_local AbStack st;
  const Board root = load(rec);
  u16 moves[MAX_MOVES];
  StoreSink s{moves, 0};
  const GenInfo gi = generate_legal(root, s);
  *move = MOVE_NONE;
  *score = 0;
  *nodes = 1;
  if (ab_terminal(root, s.n, gi.in_check, 0, score)) return 0;
  unsigned long long total = 1;
  int best = 0;
  for (int k = 0; k < s.n; ++k) {
    unsigned long long nn = 0;
    const int v = ab_root_child(st, root, moves[k], depth, qdepth, &nn);
    total += nn;
    if (k == 0 || v > best) {
      best = v;
      *move = moves[k];
    }
  }
  *score = best;
  *nodes = total;
  return 0;
}

}  // extern "C"
