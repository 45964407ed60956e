// TEST-ONLY host build of the search-target row (chessrl_b200/csrc/search_targets.cuh, DESIGN.md 3.8), compiled with g++
// by tests/hostsim/search_targets.py.  The same row code that kernels_encode.cu runs for crl_search_targets, so the CPU
// suite can check it against a numpy restatement and the GPU suite can compare the kernel with it.  It is NOT part of
// libchessrl_b200.so and nothing under chessrl_b200/ loads it.
#include "../../chessrl_b200/csrc/search_targets.cuh"
#include <string.h>
using namespace crl;

extern "C" {

// rows i = 0..n-1: record recs[9 i ..], scores scores[offsets[i] .. offsets[i+1]); label_of [5 * 4096]; writes
// policy [n][CRL_N_LABELS], value [n], legal [n]
void hs_search_targets(const uint64_t* recs, const int32_t* scores, const int32_t* offsets, int n, float temperature,
                       const int16_t* label_of, float* policy, float* value, int32_t* legal) {
  u16 moves[MAX_MOVES];
  for (int i = 0; i < n; ++i) {
    Board b;
    memcpy(b.bb, recs + 9LL * i, 64);
    b.meta = recs[9LL * i + 8];
    legal[i] = search_targets_row(b, scores + offsets[i], offsets[i + 1] - offsets[i], temperature, label_of, moves,
                                  policy + (long long)i * CRL_N_LABELS, value + i);
  }
}

}  // extern "C"
