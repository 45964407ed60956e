// kernels_ab.cu -- the fixed-depth alpha-beta opponent on the lanes of an engine (crl_games_ab_move_host, DESIGN.md 3.6).
//
// The root's legal moves are dealt one per thread: item (lane, k) searches root child k of its lane with a full window,
// so every child's value is exact and the per-lane reduction picks the first maximum in generation order.  The result is a
// function of the position alone, whatever the schedule; a batch of L lanes gives about 35 L independent searches.
//   k_ab_root    generates the root moves of every selected lane and appends its items to the item list
//   k_ab_items   each thread takes the next item from an atomic counter until none is left (subtrees differ by orders
//                of magnitude in size, so a fixed assignment would leave most threads idle behind the largest ones)
//   k_ab_reduce  per lane: the first maximum, its move, its score and the positions visited
//   k_ab_pick    in its place for crl_games_ab_pick_host: the seeded near-best pick (ab_search.cuh ab_pick_index)
// With repetitions on (crl_games_ab_search_host, CRL_AB_REPETITIONS) k_ab_rep_stage copies the keys of each searched
// root's reversible run out of the lane's key ring, and k_ab_items<true> scores a repeated position 0.  The plain
// search launches exactly what it launched before.
#include "engine.cuh"
#include "ab_search.cuh"

namespace crl {

static constexpr int AB_BLOCK = 128;

// item word: lane * MAX_MOVES + k, the same index as the lane's root moves, scores and node counts
__global__ void __launch_bounds__(AB_BLOCK) k_ab_root(Pools P, const u8* __restrict__ mask, u16* __restrict__ moves,
                                                      int* __restrict__ cnt, int* __restrict__ items,
                                                      unsigned long long* __restrict__ ctl) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= P.G) return;
  int n = -1;                                                          // -1: the lane is not searched
  if ((!mask || mask[g]) && P.g_active[g] && P.g_result[g] == RESULT_NONE) {
    StoreSink s{moves + (long long)g * MAX_MOVES, 0};
    generate_legal(load_soa(P.g_cur, P.G, g), s);
    n = s.n;
  }
  cnt[g] = n;
  if (n > 0) {
    const unsigned long long base = atomicAdd(&ctl[0], (unsigned long long)n);
    for (int k = 0; k < n; ++k) items[base + k] = g * MAX_MOVES + k;
  }
}

// per searched lane g (cnt[g] > 0): rep_keys[g][i] = the key of the position i plies before the root, i = 0..rep_n[g],
// rep_n[g] = min(revlen, ply) of the root record (the ring holds ply q in slot q % KEY_RING)
__global__ void __launch_bounds__(AB_BLOCK) k_ab_rep_stage(Pools P, const int* __restrict__ cnt,
                                                           u64* __restrict__ rep_keys, int* __restrict__ rep_n) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= P.G || cnt[g] <= 0) return;
  const u64 meta = P.g_cur[8LL * P.G + g];
  const int ply = meta_ply(meta);
  int n = meta_revlen(meta);
  if (n > ply) n = ply;
  if (n > AB_REP_KEYS - 1) n = AB_REP_KEYS - 1;
  for (int i = 0; i <= n; ++i)
    rep_keys[(long long)g * AB_REP_KEYS + i] = P.g_keys[(long long)((ply - i) % KEY_RING) * P.G + g];
  rep_n[g] = n;
}

// REP: repetitions on, with the staged keys of k_ab_rep_stage (unused by the plain search)
template <bool REP>
__global__ void __launch_bounds__(AB_BLOCK) k_ab_items(const u64* __restrict__ cur, int G, const u16* __restrict__ moves,
                                                       const int* __restrict__ items, int* __restrict__ score,
                                                       unsigned long long* __restrict__ nodes,
                                                       unsigned long long* __restrict__ ctl, int depth, int qdepth,
                                                       const u64* __restrict__ rep_keys, const int* __restrict__ rep_n) {
  AbStack st;
  const unsigned long long total = ctl[0];
  for (;;) {
    const unsigned long long it = atomicAdd(&ctl[1], 1ull);
    if (it >= total) return;
    const int w = items[it];
    unsigned long long nn = 0;
    if constexpr (REP) {
      const int g = w / MAX_MOVES;
      AbPath path;
      path.game = rep_keys + (long long)g * AB_REP_KEYS;
      path.ngame = rep_n[g];
      score[w] = ab_root_child<true>(st, load_soa(cur, G, g), moves[w], depth, qdepth, &nn, &path);
    } else {
      score[w] = ab_root_child(st, load_soa(cur, G, w / MAX_MOVES), moves[w], depth, qdepth, &nn);
    }
    nodes[w] = nn;
  }
}

__global__ void __launch_bounds__(AB_BLOCK) k_ab_reduce(int G, const int* __restrict__ cnt, const u16* __restrict__ moves,
                                                        const int* __restrict__ score,
                                                        const unsigned long long* __restrict__ nodes,
                                                        u16* __restrict__ out_move, int* __restrict__ out_score,
                                                        long long* __restrict__ out_nodes) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const int n = cnt[g];
  u16 mv = MOVE_NONE;
  int best = 0;
  unsigned long long total = 0;
  if (n > 0) {
    const long long o = (long long)g * MAX_MOVES;
    int bk = 0;
    best = score[o];
    total = 1 + nodes[o];                                              // the root and its children's subtrees
    for (int k = 1; k < n; ++k) {
      if (score[o + k] > best) {                                       // strict: the first maximum stays
        best = score[o + k];
        bk = k;
      }
      total += nodes[o + k];
    }
    mv = moves[o + bk];
  }
  out_move[g] = mv;
  out_score[g] = best;
  out_nodes[g] = (long long)total;
}

// k_ab_reduce with the seeded near-best pick of ab_pick_index (crl_games_ab_pick_host, DESIGN.md 3.7): salt[g] per lane,
// ply from the lane's record; the score is the picked child's, the node count the same sum
__global__ void __launch_bounds__(AB_BLOCK) k_ab_pick(const u64* __restrict__ cur, int G, const int* __restrict__ cnt,
                                                      const u16* __restrict__ moves, const int* __restrict__ score,
                                                      const unsigned long long* __restrict__ nodes,
                                                      const u64* __restrict__ salt, int margin, int pick_plies,
                                                      u16* __restrict__ out_move, int* __restrict__ out_score,
                                                      long long* __restrict__ out_nodes) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const int n = cnt[g];
  u16 mv = MOVE_NONE;
  int sc = 0;
  unsigned long long total = 0;
  if (n > 0) {
    const long long o = (long long)g * MAX_MOVES;
    const int k = ab_pick_index(score + o, n, meta_ply(cur[8LL * G + g]), margin, pick_plies, salt[g]);
    total = 1;
    for (int i = 0; i < n; ++i) total += nodes[o + i];
    mv = moves[o + k];
    sc = score[o + k];
  }
  out_move[g] = mv;
  out_score[g] = sc;
  out_nodes[g] = (long long)total;
}

// scratch of the search, allocated at the first call (an engine that never searches holds none of it)
static int ab_ensure(crl_engine_impl* e) {
  if (e->ab_moves) return CRL_OK;
  // enough threads to fill the GPU; each takes items until none is left
  int dev_sms = 0, per_sm = 0;
  CRL_CUDA(cudaDeviceGetAttribute(&dev_sms, cudaDevAttrMultiProcessorCount, e->device));
  CRL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_ab_items<false>, AB_BLOCK, 0));
  e->ab_grid = dev_sms * (per_sm > 0 ? per_sm : 1);
  const size_t items = (size_t)e->G * MAX_MOVES;
  const size_t bytes = items * (2 + 4 + 4 + 8) + (size_t)e->G * (4 + 2 + 4 + 8) + 16 * 8 + 64 * 10;
  char* p = nullptr;
  cudaError_t err = cudaMalloc(&p, bytes);
  if (err != cudaSuccess) {
    set_error("crl_games_ab_move_host: cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(err));
    return CRL_ENOMEM;
  }
  e->allocs.push_back(p);
  auto take = [&](size_t n) {
    char* q = p;
    p += (n + 63) / 64 * 64;
    return q;
  };
  e->ab_nodes = (unsigned long long*)take(items * 8);
  e->ab_out_nodes = (long long*)take((size_t)e->G * 8);
  e->ab_ctl = (unsigned long long*)take(16 * 8);
  e->ab_items = (int*)take(items * 4);
  e->ab_score = (int*)take(items * 4);
  e->ab_cnt = (int*)take((size_t)e->G * 4);
  e->ab_out_score = (int*)take((size_t)e->G * 4);
  e->ab_moves = (u16*)take(items * 2);
  e->ab_out_move = (u16*)take((size_t)e->G * 2);
  return CRL_OK;
}

// scratch of the repetition window, allocated at the first call with repetitions on
static int ab_rep_ensure(crl_engine_impl* e) {
  if (e->ab_rep_keys) return CRL_OK;
  int dev_sms = 0, per_sm = 0;
  CRL_CUDA(cudaDeviceGetAttribute(&dev_sms, cudaDevAttrMultiProcessorCount, e->device));
  CRL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_ab_items<true>, AB_BLOCK, 0));
  e->ab_rep_grid = dev_sms * (per_sm > 0 ? per_sm : 1);
  const size_t keys = (size_t)e->G * AB_REP_KEYS * 8, bytes = keys + (size_t)e->G * 4 + 64;
  char* p = nullptr;
  cudaError_t err = cudaMalloc(&p, bytes);
  if (err != cudaSuccess) {
    set_error("crl_games_ab_search_host: cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(err));
    return CRL_ENOMEM;
  }
  e->allocs.push_back(p);
  e->ab_rep_keys = (u64*)p;
  e->ab_rep_n = (int*)(p + (keys + 63) / 64 * 64);
  return CRL_OK;
}

int launch_ab_move(crl_engine_impl* e, const u8* mask_dev, int depth, int qdepth, const u64* salt_dev, int margin,
                   int pick_plies, bool reps, const char* fn) {
  if (!ab_limits_ok(depth, qdepth)) {
    set_error("%s: depth %d / qdepth %d out of range (1..%d / 0..%d)", fn, depth, qdepth, (int)AB_MAX_DEPTH,
              (int)AB_MAX_QDEPTH);
    return CRL_EINVAL;
  }
  if (salt_dev && !ab_pick_ok(margin, pick_plies)) {
    set_error("%s: margin %d / pick_plies %d must be >= 0", fn, margin, pick_plies);
    return CRL_EINVAL;
  }
  int rc = ab_ensure(e);
  if (rc) return rc;
  if (reps) {
    rc = ab_rep_ensure(e);
    if (rc) return rc;
  }
  CRL_CUDA(cudaMemsetAsync(e->ab_ctl, 0, 2 * sizeof(unsigned long long), e->stream));
  {
    LaunchScope ls(e, KC_MOVEGEN);
    k_ab_root<<<div_up(e->G, AB_BLOCK), AB_BLOCK, 0, e->stream>>>(e->P, mask_dev, e->ab_moves, e->ab_cnt, e->ab_items,
                                                                  e->ab_ctl);
    CRL_CUDA(cudaGetLastError());
  }
  if (reps) {
    LaunchScope ls(e, KC_MOVEGEN);
    k_ab_rep_stage<<<div_up(e->G, AB_BLOCK), AB_BLOCK, 0, e->stream>>>(e->P, e->ab_cnt, e->ab_rep_keys, e->ab_rep_n);
    CRL_CUDA(cudaGetLastError());
  }
  {
    // no more threads than items could exist (a few lanes need a few blocks)
    const int want = div_up((long long)e->G * MAX_MOVES, AB_BLOCK);
    LaunchScope ls(e, KC_MOVEGEN);
    if (reps)
      k_ab_items<true><<<want < e->ab_rep_grid ? want : e->ab_rep_grid, AB_BLOCK, 0, e->stream>>>(
          e->P.g_cur, e->G, e->ab_moves, e->ab_items, e->ab_score, e->ab_nodes, e->ab_ctl, depth, qdepth,
          e->ab_rep_keys, e->ab_rep_n);
    else
      k_ab_items<false><<<want < e->ab_grid ? want : e->ab_grid, AB_BLOCK, 0, e->stream>>>(
          e->P.g_cur, e->G, e->ab_moves, e->ab_items, e->ab_score, e->ab_nodes, e->ab_ctl, depth, qdepth, nullptr,
          nullptr);
    CRL_CUDA(cudaGetLastError());
  }
  {
    LaunchScope ls(e, KC_MOVEGEN);
    if (salt_dev)
      k_ab_pick<<<div_up(e->G, AB_BLOCK), AB_BLOCK, 0, e->stream>>>(
          e->P.g_cur, e->G, e->ab_cnt, e->ab_moves, e->ab_score, e->ab_nodes, salt_dev, margin, pick_plies,
          e->ab_out_move, e->ab_out_score, e->ab_out_nodes);
    else
      k_ab_reduce<<<div_up(e->G, AB_BLOCK), AB_BLOCK, 0, e->stream>>>(e->G, e->ab_cnt, e->ab_moves, e->ab_score,
                                                                      e->ab_nodes, e->ab_out_move, e->ab_out_score,
                                                                      e->ab_out_nodes);
    CRL_CUDA(cudaGetLastError());
  }
  return CRL_OK;
}

}  // namespace crl
