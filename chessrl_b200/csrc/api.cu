// api.cu -- the C ABI of libchessrl_b200.so (include/chessrl_b200.h).  No torch types, no exceptions across
// the boundary, no CPU compute path: every entry point that computes launches sm_100a kernels.
#include "engine.cuh"

#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

namespace crl {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int cuda_fail(cudaError_t err, const char* what) {
  set_error("CUDA error %d (%s) at %s", (int)err, cudaGetErrorString(err), what);
  return CRL_ECUDA;
}

template <class T>
static int pool_alloc(crl_engine_impl* e, T** p, size_t count) {
  void* q = nullptr;
  size_t bytes = count * sizeof(T);
  cudaError_t err = cudaMalloc(&q, bytes ? bytes : 8);
  if (err != cudaSuccess) {
    set_error("cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(err));
    return CRL_ENOMEM;
  }
  err = cudaMemsetAsync(q, 0, bytes ? bytes : 8, e->stream);
  if (err != cudaSuccess) return cuda_fail(err, "cudaMemsetAsync");
  e->allocs.push_back(q);
  *p = (T*)q;
  return CRL_OK;
}

// netencoder.get_uci_labels order (netencoder.py:94-134), rebuilt here as an index table:
// idx[promo][from][to], promo 0 = none, 1 N, 2 B, 3 R, 4 Q; squares a1 = 0 .. h8 = 63.
static void build_label_table(std::vector<int16_t>& t) {
  t.assign(5 * 4096, -1);
  int next = 0;
  static const int kn[8][2] = {{-2, -1}, {-1, -2}, {-2, 1}, {1, -2}, {2, -1}, {-1, 2}, {2, 1}, {1, 2}};
  for (int f = 0; f < 8; ++f)
    for (int r = 0; r < 8; ++r) {
      int dest[8 + 8 + 15 + 15 + 8][2];
      int nd = 0;
      for (int k = 0; k < 8; ++k) { dest[nd][0] = k; dest[nd][1] = r; ++nd; }
      for (int k = 0; k < 8; ++k) { dest[nd][0] = f; dest[nd][1] = k; ++nd; }
      for (int k = -7; k < 8; ++k) { dest[nd][0] = f + k; dest[nd][1] = r + k; ++nd; }
      for (int k = -7; k < 8; ++k) { dest[nd][0] = f + k; dest[nd][1] = r - k; ++nd; }
      for (int k = 0; k < 8; ++k) { dest[nd][0] = f + kn[k][0]; dest[nd][1] = r + kn[k][1]; ++nd; }
      for (int i = 0; i < nd; ++i) {
        int f2 = dest[i][0], r2 = dest[i][1];
        if ((f2 == f && r2 == r) || f2 < 0 || f2 > 7 || r2 < 0 || r2 > 7) continue;
        t[(r * 8 + f) * 64 + (r2 * 8 + f2)] = (int16_t)next++;
      }
    }
  static const int promo_code[4] = {4, 3, 2, 1};   // q r b n
  for (int f = 0; f < 8; ++f)
    for (int p = 0; p < 4; ++p) {
      static const int df[3] = {0, -1, 1};
      for (int d = 0; d < 3; ++d) {
        int f2 = f + df[d];
        if (f2 < 0 || f2 > 7) continue;
        t[promo_code[p] * 4096 + (1 * 8 + f) * 64 + (0 * 8 + f2)] = (int16_t)next++;   // x2 -> y1
        t[promo_code[p] * 4096 + (6 * 8 + f) * 64 + (7 * 8 + f2)] = (int16_t)next++;   // x7 -> y8
      }
    }
}

static int drain_profile(crl_engine_impl* e) {
  for (auto& it : e->prof_pending) {
    float ms = 0.f;
    cudaEventSynchronize(it.second.second);
    cudaEventElapsedTime(&ms, it.second.first, it.second.second);
    e->prof_ms[it.first] += ms;
    cudaEventDestroy(it.second.first);
    cudaEventDestroy(it.second.second);
  }
  e->prof_pending.clear();
  return CRL_OK;
}

// grows the device/pinned staging buffers
static int ensure_stage(crl_engine_impl* e, size_t bytes) {
  if (bytes <= e->d_stage_bytes) return CRL_OK;
  size_t want = bytes * 2 + 4096;
  if (e->d_stage) cudaFree(e->d_stage);
  if (e->h_stage) cudaFreeHost(e->h_stage);
  e->d_stage = nullptr;
  e->h_stage = nullptr;
  e->d_stage_bytes = e->h_stage_bytes = 0;
  CRL_CUDA(cudaMalloc(&e->d_stage, want));
  CRL_CUDA(cudaMallocHost(&e->h_stage, want));
  e->d_stage_bytes = e->h_stage_bytes = want;
  return CRL_OK;
}

// The slots a search routes rows to: slot 1 joins while some lane names it as a player (DESIGN.md 3.5)
static int route_slots(crl_engine_impl* e, const char* fn) {
  const int slots = e->lanes_on_slot1 > 0 ? 2 : 1;
  if (slots > 1) {
    if (!e->slot_configured[1]) {
      set_error("%s: %d lanes name network slot 1 as a player, but slot 1 has no evaluator (crl_net_select_slot, then "
                "crl_net_load_host or crl_set_evaluator)", fn, e->lanes_on_slot1);
      return CRL_ESTATE;
    }
    if (e->eval_kind[0] != e->eval_kind[1]) {
      set_error("%s: the network slots hold evaluators of different kinds (hash and network); one search reads both "
                "through one policy view", fn);
      return CRL_ESTATE;
    }
  }
  e->search_slots = slots;
  e->P.n_slots = slots;
  e->P.slot_stride = (int)e->slot_stride;
  return CRL_OK;
}

static int check_pool_errors(crl_engine_impl* e) {
  int err = 0;
  CRL_CUDA(cudaMemcpyAsync(&err, e->P.err, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  if (err) {
    // report once and clear: kernels only OR into the flag, and one overflowing game must not make every later call
    // on this engine fail (the offending lanes keep whatever partial state they have; callers reload them)
    CRL_CUDA(cudaMemsetAsync(e->P.err, 0, sizeof(int), e->stream));
    CRL_CUDA(cudaMemsetAsync(e->P.g_prev_root, 0xFF, sizeof(int) * (size_t)e->G, e->stream));   // no reuse of a broken tree
    set_error("pool overflow on the device (flags %d: 1 = nodes per game, 2 = edges per game, 4 = plies per game, 8 = more "
              "running games than crl_mcts_set_row_bound promised); create the engine with larger max_nodes / avg_moves", err);
    return CRL_ENOMEM;
  }
  return CRL_OK;
}

}  // namespace crl

namespace crl {
__global__ void k_root_stats(Pools P, int* visits, double* values, float* priors, u16* moves, u16* replies,
                             int8_t* results, int* n_children, int* root_visits, double* root_values) {
  const int g = blockIdx.x;
  const NodeRec& root = P.nodes[(long long)g * P.NN];
  const bool on = P.g_active[g] && P.g_nnodes[g] > 0;
  const int n = on ? root.n_exp : 0;
  if (threadIdx.x == 0) {
    if (n_children) n_children[g] = n;
    if (root_visits) root_visits[g] = on ? P.r_visits[g] : 0;
    if (root_values) root_values[g] = on ? P.r_value[g] : 0.0;
  }
  for (int k = threadIdx.x; k < MAX_MOVES; k += blockDim.x) {
    const long long o = (long long)g * MAX_MOVES + k;
    if (k < n) {
      const long long eidx = (long long)g * P.EA + root.edge0 + k;
      const NodeRec& c = P.nodes[(long long)g * P.NN + P.e_child[eidx]];
      if (visits) visits[o] = P.e_visits[eidx];
      if (values) values[o] = P.e_value[eidx];
      if (priors) priors[o] = P.e_prior[eidx];
      if (moves) moves[o] = c.move;
      if (replies) replies[o] = c.reply;
      if (results) results[o] = c.result;
    } else {
      if (visits) visits[o] = 0;
      if (values) values[o] = 0.0;
      if (priors) priors[o] = 0.f;
      if (moves) moves[o] = MOVE_NONE;
      if (replies) replies[o] = MOVE_NONE;
      if (results) results[o] = RESULT_NONE;
    }
  }
}

// lanes whose players changed: the previous tree was searched by another network, nothing of it is reused
__global__ void k_unlink_lanes(Pools P, int first, int n, const u8* changed) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && changed[i]) P.g_prev_root[first + i] = -1;
}

__global__ void k_node_dump(Pools P, int g, crl_node_host* out, int cap) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = P.g_nnodes[g];
  if (j >= n || j >= cap) return;
  const NodeRec& nd = P.nodes[(long long)g * P.NN + j];
  crl_node_host o;
  o.parent = nd.parent;
  o.slot = nd.slot;
  o.n_legal = nd.n_legal;
  o.n_children = nd.n_exp;
  o.result = nd.result;
  o.move = nd.move;
  o.reply = nd.reply;
  if (j == 0) {
    o.visits = P.r_visits[g];
    o.value = P.r_value[g];
    o.prior = 1.0f;
  } else {
    const NodeRec& pn = P.nodes[(long long)g * P.NN + nd.parent];
    const long long eidx = (long long)g * P.EA + pn.edge0 + nd.slot;
    o.visits = P.e_visits[eidx];
    o.value = P.e_value[eidx];
    // a child's prior exists once its parent was evaluated; Node.prior stays 1 until the parent is fully expanded
    o.prior = (pn.n_exp == pn.n_legal) ? P.e_prior[eidx] : 1.0f;
  }
  for (int k = 0; k < 9; ++k) o.board[k] = nd.p2[k];
  out[j] = o;
}
}  // namespace crl

using namespace crl;

#define CHECK_ENGINE(e)                          \
  do {                                           \
    if (!(e)) {                                  \
      set_error("null engine handle");           \
      return CRL_EINVAL;                         \
    }                                            \
    cudaError_t _d = cudaSetDevice((e)->device); \
    if (_d != cudaSuccess) return cuda_fail(_d, "cudaSetDevice"); \
  } while (0)

// kernels_encode.cu (declared here rather than in engine.cuh, whose lines the other kernels' line info refers to)
namespace crl {
int launch_search_targets(crl_engine_impl* e, const u64* boards, const int* scores, const int* offsets, int n,
                          float temperature, float* policy, float* score_value, int* legal_count);
}

extern "C" {

const char* crl_last_error(void) { return g_err; }
int crl_version(void) { return 100; }

int crl_create(crl_engine** out, int device, int max_games, int max_nodes, int avg_moves, void* stream) {
  return crl_create_ex(out, device, max_games, max_nodes, avg_moves, 1, stream);
}

int crl_create_ex(crl_engine** out, int device, int max_games, int max_nodes, int avg_moves, int max_inflight,
                  void* stream) {
  if (!out || max_games <= 0 || max_nodes <= 0 || max_inflight < 1 || max_inflight > CRL_MAX_INFLIGHT ||
      (long long)max_games * max_inflight > (1ll << 24) || avg_moves > MAX_MOVES ||
      ((long long)max_nodes + 1) * (avg_moves > 0 ? avg_moves : 64) > 0x7fffffffll) {   // per-game edge arena is int-indexed
    set_error("crl_create: bad arguments (max_games %d, max_nodes %d, avg_moves %d, max_inflight %d)", max_games, max_nodes,
              avg_moves, max_inflight);
    return CRL_EINVAL;
  }
  int n_dev = 0;
  cudaError_t err = cudaGetDeviceCount(&n_dev);
  if (err != cudaSuccess || n_dev == 0) {
    set_error("crl_create: no CUDA device (%s); this library has no CPU path", cudaGetErrorString(err));
    return CRL_ECUDA;
  }
  CRL_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  CRL_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_error("crl_create: device %d is sm_%d%d; libchessrl_b200 is built for sm_100a (B200) only", device, prop.major,
              prop.minor);
    return CRL_ECUDA;
  }
  crl_engine* e = new crl_engine();
  e->device = device;
  e->stream = (cudaStream_t)stream;
  if (e->stream == nullptr) {
    // the legacy default stream cannot be captured into a CUDA graph: use an own BLOCKING stream, which keeps the
    // implicit ordering with work the caller (torch) puts on the default stream
    cudaError_t se = cudaStreamCreate(&e->stream);
    if (se != cudaSuccess) {
      delete e;
      return cuda_fail(se, "cudaStreamCreate");
    }
    e->own_stream = true;
  }
  {
    const char* g = getenv("CRL_NO_GRAPH");
    e->use_graph = !(g && g[0] == '1');
    const char* pd = getenv("CRL_NO_PDL");
    e->perft_pdl = !(pd && pd[0] == '1');
    const char* pp = getenv("CRL_PERFT_PAIR");
    e->perft_pair = !pp ? 0 : pp[0] == '5' ? 5 : pp[0] == '6' ? 6 : 0;
  }
  e->G = max_games;
  e->Kmax = max_inflight;
  e->R = max_games * max_inflight;
  e->cur_rows = max_games;
  e->P.row_cap = max_games * max_inflight;
  e->NN = max_nodes + 1;
  if (avg_moves <= 0) avg_moves = 64;
  long long ea = (long long)e->NN * avg_moves;
  if (ea < 512) ea = 512;
  e->EA = (int)ea;
  Pools& P = e->P;
  P.G = e->G;
  P.NN = e->NN;
  P.EA = e->EA;
  P.K = 1;
  P.path_cap = 32;
  if (const char* pc = getenv("CRL_PATH_CAP")) {
    const int v = atoi(pc);
    if (v >= 0 && v <= 32) P.path_cap = v;
  }
  const size_t G = e->G, R = e->R;
  int rc = CRL_OK;
#define A(field, count) if (rc == CRL_OK) rc = pool_alloc(e, &P.field, (size_t)(count))
  A(g_cur, 9 * G);
  A(g_hist, (size_t)HIST_RING * 8 * G);
  A(g_keys, (size_t)KEY_RING * G);
  A(g_moves, G * MAX_GAME_PLIES);
  A(g_nmoves, G);
  A(g_result, G);
  A(g_active, G);
  A(nodes, G * e->NN);
  A(g_nnodes, G);
  A(g_nedges, G);
  A(e_move, G * e->EA);
  A(e_prior, G * e->EA);
  A(e_visits, G * e->EA);
  A(e_value, G * e->EA);
  A(e_child, G * e->EA);
  A(e_result, G * e->EA);
  A(e_vloss, G * e->EA);
  A(r_visits, G);
  A(r_value, G);
  A(g_prev_root, G);
  A(s_node, R);
  A(s_kind, R);
  A(s_moves, R * MAX_MOVES);
  A(s_nmoves, R);
  A(s_row, R);
  A(s_path, G * 32);
  A(s_depth, G);
  A(s_wave_n, G);
  A(g_sims_left, G);
  A(err, 1);
  A(counters, 4);
#undef A
  if (rc == CRL_OK) rc = pool_alloc(e, &e->d_list[0], R);
  if (rc == CRL_OK) rc = pool_alloc(e, &e->d_list[1], R);
  if (rc == CRL_OK) rc = pool_alloc(e, &e->d_n, 2 * SLOT_N_STRIDE);
  if (rc == CRL_OK) rc = pool_alloc(e, &e->d_tmp_moves, 2 * G);
  if (rc == CRL_OK) rc = pool_alloc(e, &e->d_tmp_pick, G);
  if (rc == CRL_OK) rc = pool_alloc(e, &e->d_planes, (R + 2) * 64 * 128);
  if (rc == CRL_OK) rc = pool_alloc(e, &e->d_policy, (R + 2) * CRL_N_LABELS);
  if (rc == CRL_OK) rc = pool_alloc(e, &e->d_value, R + 2);
  if (rc == CRL_OK) rc = pool_alloc(e, &e->d_stats, 2 * (R + 2));
  if (rc == CRL_OK) rc = pool_alloc(e, &e->d_label_of, 5 * 4096);
  if (rc == CRL_OK) {
    P.eval_list = e->d_list[0];
    P.eval_n = e->d_n;
    P.n_slots = 1;
    build_label_table(e->h_label_of);
    cudaError_t ce = cudaMemcpyAsync(e->d_label_of, e->h_label_of.data(), 5 * 4096 * sizeof(int16_t),
                                     cudaMemcpyHostToDevice, e->stream);
    if (ce != cudaSuccess) rc = cuda_fail(ce, "label table upload");
  }
  if (rc == CRL_OK) {
    cudaError_t ce = cudaMemsetAsync(P.g_prev_root, 0xFF, sizeof(int) * G, e->stream);
    if (ce != cudaSuccess) rc = cuda_fail(ce, "g_prev_root init");
  }
  if (rc == CRL_OK) rc = net_create(e, 0);
  if (rc == CRL_OK) {
    cudaError_t ce = cudaStreamSynchronize(e->stream);
    if (ce != cudaSuccess) rc = cuda_fail(ce, "crl_create sync");
  }
  if (rc != CRL_OK) {
    crl_destroy(e);
    return rc;
  }
  *out = e;
  return CRL_OK;
}

int crl_destroy(crl_engine* e) {
  if (e) {
    for (int i = 0; i < 2; ++i)
      if (e->perft_buf[i]) cudaFree(e->perft_buf[i]);
    e->perft_buf[0] = e->perft_buf[1] = nullptr;
  }
  if (!e) return CRL_OK;
  cudaSetDevice(e->device);
  cudaStreamSynchronize(e->stream);
  drain_profile(e);
  for (int i = 0; i < 2; ++i)
    if (e->sim_graph[i]) cudaGraphExecDestroy(e->sim_graph[i]);
  net_destroy(e);
  for (void* p : e->allocs) cudaFree(p);
  if (e->d_stage) cudaFree(e->d_stage);
  if (e->h_stage) cudaFreeHost(e->h_stage);
  if (e->own_stream) cudaStreamDestroy(e->stream);
  delete e;
  return CRL_OK;
}

// ---- rules -------------------------------------------------------------------------------------------
int crl_movegen(crl_engine* e, const uint64_t* boards_dev, int n, uint16_t* moves_dev, int32_t* counts_dev,
                uint8_t* flags_dev) {
  CHECK_ENGINE(e);
  if (n < 0 || (n > 0 && (!boards_dev || !moves_dev || !counts_dev))) {
    set_error("crl_movegen: bad arguments");
    return CRL_EINVAL;
  }
  return launch_movegen(e, boards_dev, n, moves_dev, counts_dev, flags_dev);
}
int crl_debug_movegen_warp(crl_engine* e, const uint64_t* boards_dev, int n, uint16_t* moves_dev, int32_t* counts_dev,
                           uint8_t* flags_dev) {
  CHECK_ENGINE(e);
  if (n < 0 || (n > 0 && (!boards_dev || !moves_dev || !counts_dev))) {
    set_error("crl_debug_movegen_warp: bad arguments");
    return CRL_EINVAL;
  }
  return launch_movegen_warp(e, boards_dev, n, moves_dev, counts_dev, flags_dev);
}
int crl_make_moves(crl_engine* e, uint64_t* boards_dev, int n, const uint16_t* moves_dev) {
  CHECK_ENGINE(e);
  if (n < 0 || (n > 0 && (!boards_dev || !moves_dev))) {
    set_error("crl_make_moves: bad arguments");
    return CRL_EINVAL;
  }
  return launch_make(e, boards_dev, n, moves_dev);
}
int crl_perft(crl_engine* e, const uint64_t* boards_dev, int n, int depth, int bulk, uint64_t* nodes_dev) {
  CHECK_ENGINE(e);
  if (n < 0 || depth < 0 || (n > 0 && (!boards_dev || !nodes_dev))) {
    set_error("crl_perft: bad arguments");
    return CRL_EINVAL;
  }
  return launch_perft(e, boards_dev, n, depth, bulk, (unsigned long long*)nodes_dev);
}
int crl_perft_root_host(crl_engine* e, const uint64_t* root_host, int depth, int bulk, int64_t min_frontier,
                        uint64_t* total_host, int64_t* lanes_host, int32_t* bfs_plies_host) {
  return crl_perft_root_shard_host(e, root_host, depth, bulk, min_frontier, 0, 1, 1, total_host, lanes_host, bfs_plies_host);
}

int crl_perft_root_shard_host(crl_engine* e, const uint64_t* root_host, int depth, int bulk, int64_t min_frontier, int shard,
                              int n_shards, int64_t shard_min_frontier, uint64_t* total_host, int64_t* lanes_host,
                              int32_t* bfs_plies_host) {
  CHECK_ENGINE(e);
  if (shard_min_frontier < 256) shard_min_frontier = 256;     // the first kernel's plies (<= 218 boards in) are never split
  if (!root_host || !total_host || depth < 0 || min_frontier < 1 || n_shards < 1 || shard < 0 || shard >= n_shards) {
    set_error("crl_perft_root_host: bad arguments");
    return CRL_EINVAL;
  }
  if (!e->perft_ctl) {
    CRL_CUDA(cudaMalloc((void**)&e->perft_ctl, 16 * sizeof(unsigned long long)));
    e->allocs.push_back(e->perft_ctl);
  }
  // capacity: the frontier stops growing once it holds min_frontier boards, so 16x leaves room for one more ply of a
  // quiet position; a bushier frontier overflows, which is detected on the device and retried with four times the room
  // (a sharded call replicates frontiers below shard_min boards, so the first filtered one is below 218 x shard_min / n)
  long long cap = min_frontier * 16;
  if (n_shards > 1 && shard_min_frontier * 64 > cap) cap = shard_min_frontier * 64;
  if (cap < (1 << 16)) cap = 1 << 16;
  const long long cap_max = 320LL << 20;       // 320 Mi boards = 23 GB per buffer: holds Kiwipete's depth-5 frontier
  if (cap > cap_max) cap = min_frontier * 2 > cap_max ? min_frontier * 2 : cap_max;
  for (int attempt = 0; attempt < 4; ++attempt, cap *= 4) {
    if (cap > e->perft_cap) {
      for (int i = 0; i < 2; ++i) {
        if (e->perft_buf[i]) cudaFree(e->perft_buf[i]);
        e->perft_buf[i] = nullptr;
      }
      e->perft_cap = 0;
      for (int i = 0; i < 2; ++i) {
        cudaError_t err = cudaMalloc((void**)&e->perft_buf[i], (size_t)cap * 72);
        if (err != cudaSuccess) {
          set_error("crl_perft_root_host: cudaMalloc(%lld boards) failed: %s", cap, cudaGetErrorString(err));
          return CRL_ENOMEM;
        }
      }
      e->perft_cap = cap;
    }
    const long long stride = e->perft_cap;
    // the root record travels as a kernel parameter (no copy), the control block is initialised on the device
    int rc = launch_perft_root(e, root_host, e->perft_buf[0], e->perft_buf[1], stride, e->perft_ctl, depth, bulk,
                               min_frontier, e->perft_pair, shard, n_shards, shard_min_frontier);
    if (rc) return rc;
    if ((rc = ensure_stage(e, 64))) return rc;
    unsigned long long* ctl = (unsigned long long*)e->h_stage;          // pinned: the read-back is one async copy
    CRL_CUDA(cudaMemcpyAsync(ctl, e->perft_ctl, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, e->stream));
    CRL_CUDA(cudaStreamSynchronize(e->stream));
    if (ctl[3] == 0) {
      *total_host = depth == 0 ? (shard == 0 ? 1 : 0) : ctl[4];
      // boards the walk ran on in lockstep: the stored frontier, or -- when the last two plies went through
      // k_perft_pair -- the boards of the last-but-one ply it dealt to its lanes (ctl[5]; never stored)
      if (lanes_host) *lanes_host = (int64_t)(ctl[5] ? ctl[5] : ctl[0]);
      if (bfs_plies_host) *bfs_plies_host = (int32_t)ctl[2];
      return CRL_OK;
    }
  }
  set_error("crl_perft_root_host: the breadth-first frontier does not fit (min_frontier %lld)", (long long)min_frontier);
  return CRL_ENOMEM;
}
int crl_expand_frontier(crl_engine* e, const uint64_t* boards_dev, int n, const int64_t* offsets_dev, uint64_t* out_dev,
                        int64_t out_n, int32_t* counts_dev) {
  CHECK_ENGINE(e);
  if (n < 0 || (n > 0 && !boards_dev) || (!out_dev && !counts_dev) || (out_dev && !offsets_dev)) {
    set_error("crl_expand_frontier: bad arguments");
    return CRL_EINVAL;
  }
  return launch_frontier(e, boards_dev, n, (const long long*)offsets_dev, out_dev, out_n, counts_dev);
}

static int game_replay_impl(crl_engine* e, const uint64_t* start_host, const uint16_t* moves_host, int n_moves,
                            uint16_t* legal_host, int32_t* n_legal_host, int8_t* result_host, uint8_t* accepted_host,
                            uint64_t* final_host, uint64_t* records_host, int32_t* n_records_host) {
  CHECK_ENGINE(e);
  if (!start_host || n_moves < 0 || (n_moves > 0 && !moves_host)) {
    set_error("crl_game_replay_host: bad arguments");
    return CRL_EINVAL;
  }
  const bool want_rec = records_host != nullptr;
  // staging layout: [start 72 B][n_moves int][moves u16 x n][accepted u8 x n][legal u16 x 256][n_legal int][n_records int]
  //                 [records 72 B x (n+1), only when asked for]
  size_t off_n = 72, off_mv = 80, off_acc = off_mv + ((size_t)n_moves * 2 + 7) / 8 * 8;
  size_t off_legal = off_acc + ((size_t)n_moves + 7) / 8 * 8, off_nl = off_legal + MAX_MOVES * 2;
  size_t off_rec = off_nl + 8;
  size_t total = off_rec + (want_rec ? ((size_t)n_moves + 1) * 72 : 0);
  int rc = ensure_stage(e, total);
  if (rc) return rc;
  char* h = (char*)e->h_stage;
  char* d = (char*)e->d_stage;
  memcpy(h, start_host, 72);
  memcpy(h + off_n, &n_moves, 4);
  if (n_moves) memcpy(h + off_mv, moves_host, (size_t)n_moves * 2);
  CRL_CUDA(cudaMemcpyAsync(d, h, off_acc, cudaMemcpyHostToDevice, e->stream));
  // the record stride of the kernel is (stride + 1) records per game: exactly n_moves + 1 here
  rc = launch_games_replay(e, 0, 1, (const u64*)d, (const u16*)(d + off_mv), (const int*)(d + off_n),
                           n_moves > 0 ? n_moves : 1, (u8*)(d + off_acc), want_rec ? (u64*)(d + off_rec) : nullptr,
                           (int*)(d + off_nl + 4));
  if (rc) return rc;
  rc = launch_game_info(e, 0, 1, (u16*)(d + off_legal), (int*)(d + off_nl));
  if (rc) return rc;
  CRL_CUDA(cudaMemcpyAsync(h + off_acc, d + off_acc, total - off_acc, cudaMemcpyDeviceToHost, e->stream));
  u64 rec[9];
  CRL_CUDA(cudaMemcpy2DAsync(rec, 8, e->P.g_cur, (size_t)e->G * 8, 8, 9, cudaMemcpyDeviceToHost, e->stream));
  int8_t res = 0;
  CRL_CUDA(cudaMemcpyAsync(&res, e->P.g_result, 1, cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  e->tree_ready = false;
  if (accepted_host && n_moves) memcpy(accepted_host, h + off_acc, n_moves);
  int nl = *(int*)(h + off_nl);
  if (n_legal_host) *n_legal_host = nl;
  if (legal_host) memcpy(legal_host, h + off_legal, (size_t)nl * 2);
  if (result_host) *result_host = res;
  if (final_host) memcpy(final_host, rec, 72);
  const int nrec = *(int*)(h + off_nl + 4);
  if (n_records_host) *n_records_host = nrec;
  if (want_rec) memcpy(records_host, h + off_rec, (size_t)nrec * 72);
  return check_pool_errors(e);
}

int crl_game_replay_host(crl_engine* e, const uint64_t* start_host, const uint16_t* moves_host, int n_moves,
                         uint16_t* legal_host, int32_t* n_legal_host, int8_t* result_host, uint8_t* accepted_host,
                         uint64_t* final_host) {
  return game_replay_impl(e, start_host, moves_host, n_moves, legal_host, n_legal_host, result_host, accepted_host,
                          final_host, nullptr, nullptr);
}
int crl_game_replay_records_host(crl_engine* e, const uint64_t* start_host, const uint16_t* moves_host, int n_moves,
                                 uint16_t* legal_host, int32_t* n_legal_host, int8_t* result_host,
                                 uint8_t* accepted_host, uint64_t* records_host, int32_t* n_records_host) {
  if (!records_host || !n_records_host) {
    set_error("crl_game_replay_records_host: null output");
    return CRL_EINVAL;
  }
  return game_replay_impl(e, start_host, moves_host, n_moves, legal_host, n_legal_host, result_host, accepted_host,
                          nullptr, records_host, n_records_host);
}

// ---- encoding ----------------------------------------------------------------------------------------
int crl_encode(crl_engine* e, const uint64_t* boards_dev, const uint64_t* hist_dev, const uint8_t* hist_len_dev, int n,
               void* planes_bf16_dev) {
  CHECK_ENGINE(e);
  if (n < 0 || (n > 0 && (!boards_dev || !planes_bf16_dev))) {
    set_error("crl_encode: bad arguments");
    return CRL_EINVAL;
  }
  return launch_encode_boards(e, boards_dev, hist_dev, hist_len_dev, n, (__nv_bfloat16*)planes_bf16_dev);
}
int crl_policy_index(crl_engine* e, const uint16_t* moves_dev, const int32_t* counts_dev, int n, int16_t* idx_dev) {
  CHECK_ENGINE(e);
  if (n < 0 || (n > 0 && (!moves_dev || !counts_dev || !idx_dev))) {
    set_error("crl_policy_index: bad arguments");
    return CRL_EINVAL;
  }
  return launch_policy_index(e, moves_dev, counts_dev, n, idx_dev);
}
int crl_search_targets(crl_engine* e, const uint64_t* boards_dev, const int32_t* scores_dev, const int32_t* offsets_dev,
                       int n, float temperature, float* policy_dev, float* score_value_dev, int32_t* legal_count_dev) {
  CHECK_ENGINE(e);
  if (n < 0 || (n > 0 && (!boards_dev || !scores_dev || !offsets_dev || !policy_dev || !score_value_dev ||
                          !legal_count_dev))) {
    set_error("crl_search_targets: bad arguments");
    return CRL_EINVAL;
  }
  if (!(temperature > 0.0f) || !isfinite(temperature)) {
    set_error("crl_search_targets: temperature %g must be positive and finite", (double)temperature);
    return CRL_EINVAL;
  }
  return launch_search_targets(e, boards_dev, scores_dev, offsets_dev, n, temperature, policy_dev, score_value_dev,
                               legal_count_dev);
}
int crl_label_table_host(crl_engine* e, int16_t* idx_host) {
  if (!idx_host) {
    set_error("crl_label_table_host: null output");
    return CRL_EINVAL;
  }
  if (!e) {   // no engine: hand out the table as built on the host (a format table, not a compute path)
    std::vector<int16_t> t;
    build_label_table(t);
    memcpy(idx_host, t.data(), t.size() * sizeof(int16_t));
    return CRL_OK;
  }
  CHECK_ENGINE(e);
  CRL_CUDA(cudaMemcpyAsync(idx_host, e->d_label_of, 5 * 4096 * sizeof(int16_t), cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  return CRL_OK;
}

// ---- network -----------------------------------------------------------------------------------------
int crl_net_select_slot(crl_engine* e, int slot) {
  CHECK_ENGINE(e);
  if (slot < 0 || slot >= CRL_NET_SLOTS) {
    set_error("crl_net_select_slot: slot %d (0..%d)", slot, CRL_NET_SLOTS - 1);
    return CRL_EINVAL;
  }
  e->sel_slot = slot;
  e->net = e->nets[slot];
  return CRL_OK;
}

// the selected slot gets what a configuration needs: slot 1 its rows in the result buffers, and its network when
// weights are loaded into it (slot 0 has both from crl_create)
static int configure_slot(crl_engine_impl* e, bool with_net) {
  if (e->sel_slot == 0) return CRL_OK;
  if (with_net) return net_slot_ensure(e, e->sel_slot);
  return net_two_slot_layout(e);
}

int crl_net_load_host(crl_engine* e, const float* const* weights_host, const int64_t* sizes, int n_tensors) {
  CHECK_ENGINE(e);
  if (!weights_host || !sizes) {
    set_error("crl_net_load_host: null arguments");
    return CRL_EINVAL;
  }
  int rc = configure_slot(e, true);
  if (rc == CRL_OK) rc = net_load(e, weights_host, sizes, n_tensors);
  if (rc == CRL_OK) e->slot_configured[e->sel_slot] = true;
  return rc;
}
int crl_net_forward(crl_engine* e, const void* planes_bf16_dev, int n, float* policy_dev, float* value_dev) {
  CHECK_ENGINE(e);
  if (n < 0 || (n > 0 && (!planes_bf16_dev || !policy_dev || !value_dev))) {
    set_error("crl_net_forward: bad arguments");
    return CRL_EINVAL;
  }
  return net_forward(e, (const __nv_bfloat16*)planes_bf16_dev, n, nullptr, policy_dev, value_dev);
}
int crl_debug_conv(crl_engine* e, int layer, const void* in_dev, int cin, int n, const void* residual_dev, void* out_dev,
                   int relu) {
  CHECK_ENGINE(e);
  return net_debug_conv(e, layer, (const __nv_bfloat16*)in_dev, cin, n, (const __nv_bfloat16*)residual_dev,
                        (__nv_bfloat16*)out_dev, relu);
}
int crl_debug_tower(crl_engine* e, const void* planes_bf16_dev, int n, int layer, void* act_out_dev, float* logits_out_dev,
                    void* pf_out_dev, float* vf_out_dev, float* policy_dev, float* value_dev) {
  CHECK_ENGINE(e);
  if (!planes_bf16_dev || !policy_dev || !value_dev) {
    set_error("crl_debug_tower: null planes / policy / value");
    return CRL_EINVAL;
  }
  return net_debug_tower(e, (const __nv_bfloat16*)planes_bf16_dev, n, layer, (__nv_bfloat16*)act_out_dev, logits_out_dev,
                         (__nv_bfloat16*)pf_out_dev, vf_out_dev, policy_dev, value_dev);
}
int crl_debug_forward_counted(crl_engine* e, const void* planes_bf16_dev, int n_bound, const int32_t* n_dev,
                              float* policy_dev, float* value_dev) {
  CHECK_ENGINE(e);
  if (n_bound < 0 || !n_dev || (n_bound > 0 && (!planes_bf16_dev || !policy_dev || !value_dev))) {
    set_error("crl_debug_forward_counted: bad arguments");
    return CRL_EINVAL;
  }
  // the launch sequence of a search batch: host bound, row count read on the device, production tower and heads
  return net_forward(e, (const __nv_bfloat16*)planes_bf16_dev, n_bound, (const int*)n_dev, policy_dev, value_dev, nullptr,
                     -1, nullptr);
}
int crl_net_calibrate_host(crl_engine* e, const void* planes_bf16_dev, int n, float* amax_host) {
  CHECK_ENGINE(e);
  if (!planes_bf16_dev || !amax_host) {
    set_error("crl_net_calibrate_host: null arguments");
    return CRL_EINVAL;
  }
  return net_calibrate(e, (const __nv_bfloat16*)planes_bf16_dev, n, amax_host);
}
int crl_net_load_fp8_host(crl_engine* e, const float* const* weights_host, const int64_t* sizes, int n_tensors,
                          const float* act_amax_host) {
  CHECK_ENGINE(e);
  if (!weights_host || !sizes || !act_amax_host) {
    set_error("crl_net_load_fp8_host: null arguments");
    return CRL_EINVAL;
  }
  int rc = configure_slot(e, true);
  if (rc == CRL_OK) rc = net_load_fp8(e, weights_host, sizes, n_tensors, act_amax_host);
  if (rc == CRL_OK) e->slot_configured[e->sel_slot] = true;
  return rc;
}
int crl_net_set_precision(crl_engine* e, int precision) {
  CHECK_ENGINE(e);
  return net_set_precision(e, precision);
}
int crl_hash_eval(crl_engine* e, const uint64_t* boards_dev, int n, uint64_t seed, int policy_bits, float* policy_dev,
                  float* value_dev) {
  CHECK_ENGINE(e);
  if (n < 0 || policy_bits < 1 || policy_bits > 24 || (n > 0 && (!boards_dev || !policy_dev || !value_dev))) {
    set_error("crl_hash_eval: bad arguments");
    return CRL_EINVAL;
  }
  return launch_hash_eval_boards(e, boards_dev, n, seed, policy_bits, policy_dev, value_dev);
}

// ---- games + search -----------------------------------------------------------------------------------
int crl_set_evaluator(crl_engine* e, int kind, uint64_t seed, int policy_bits) {
  CHECK_ENGINE(e);
  if ((kind != CRL_EVAL_NET && kind != CRL_EVAL_HASH) || (kind == CRL_EVAL_HASH && (policy_bits < 1 || policy_bits > 24))) {
    set_error("crl_set_evaluator: bad arguments");
    return CRL_EINVAL;
  }
  int rc = configure_slot(e, false);
  if (rc) return rc;
  const int k = e->sel_slot;
  e->eval_kind[k] = kind;
  e->eval_seed[k] = seed;
  e->eval_bits[k] = policy_bits;
  e->slot_configured[k] = true;
  return CRL_OK;
}

int crl_games_set_players_host(crl_engine* e, int first, int n, const uint8_t* white_slot_host,
                               const uint8_t* black_slot_host) {
  CHECK_ENGINE(e);
  if (first < 0 || n <= 0 || first + n > e->G || !white_slot_host || !black_slot_host) {
    set_error("crl_games_set_players_host: bad arguments (first %d, n %d, capacity %d)", first, n, e->G);
    return CRL_EINVAL;
  }
  for (int i = 0; i < n; ++i)
    if (white_slot_host[i] >= CRL_NET_SLOTS || black_slot_host[i] >= CRL_NET_SLOTS) {
      set_error("crl_games_set_players_host: lane %d names slot %d / %d (0..%d)", first + i, white_slot_host[i],
                black_slot_host[i], CRL_NET_SLOTS - 1);
      return CRL_EINVAL;
    }
  const size_t G = e->G;
  if (e->h_players.empty()) {        // the first call: the device copy and the per-lane searching slot
    u8* players = nullptr;
    int rc = pool_alloc(e, &players, 2 * G);
    if (rc == CRL_OK) rc = pool_alloc(e, &e->P.g_slot, G);
    if (rc) return rc;
    e->P.g_players = players;
    e->h_players.assign(2 * G, 0);
  }
  // staging: [white n][black n][changed n]; a lane whose players change is unlinked from its previous tree
  int rc = ensure_stage(e, 3 * (size_t)n);
  if (rc) return rc;
  u8* h = (u8*)e->h_stage;
  u8* d = (u8*)e->d_stage;
  int changed = 0;
  for (int i = 0; i < n; ++i) {
    const size_t g = (size_t)first + i;
    h[i] = white_slot_host[i];
    h[n + i] = black_slot_host[i];
    h[2 * n + i] = h[i] != e->h_players[g] || h[n + i] != e->h_players[G + g];
    changed += h[2 * n + i];
    e->lanes_on_slot1 += (h[i] == 1 || h[n + i] == 1) - (e->h_players[g] == 1 || e->h_players[G + g] == 1);
    e->h_players[g] = h[i];
    e->h_players[G + g] = h[n + i];
  }
  CRL_CUDA(cudaMemcpyAsync(d, h, 3 * (size_t)n, cudaMemcpyHostToDevice, e->stream));
  CRL_CUDA(cudaMemcpyAsync((u8*)e->P.g_players + first, d, n, cudaMemcpyDeviceToDevice, e->stream));
  CRL_CUDA(cudaMemcpyAsync((u8*)e->P.g_players + G + first, d + n, n, cudaMemcpyDeviceToDevice, e->stream));
  if (changed) {
    LaunchScope ls(e, KC_GAME);
    k_unlink_lanes<<<div_up(n, 128), 128, 0, e->stream>>>(e->P, first, n, d + 2 * n);
    CRL_CUDA(cudaGetLastError());
    e->tree_ready = false;
  }
  CRL_CUDA(cudaStreamSynchronize(e->stream));   // the staging buffer is reused by the next call
  return CRL_OK;
}

int crl_games_set_host(crl_engine* e, int first, int n, const uint64_t* start_host, const uint16_t* moves_host,
                       const int32_t* n_moves_host, int stride) {
  CHECK_ENGINE(e);
  if (first < 0 || n <= 0 || first + n > e->G || !start_host || stride < 0 || (stride > 0 && (!moves_host || !n_moves_host))) {
    set_error("crl_games_set_host: bad arguments (first %d, n %d, capacity %d)", first, n, e->G);
    return CRL_EINVAL;
  }
  size_t b_start = (size_t)n * 72, b_cnt = (size_t)n * 4, b_mv = ((size_t)n * stride * 2 + 7) / 8 * 8;
  int rc = ensure_stage(e, b_start + b_cnt + b_mv);
  if (rc) return rc;
  char* h = (char*)e->h_stage;
  char* d = (char*)e->d_stage;
  memcpy(h, start_host, b_start);
  if (stride > 0) {
    memcpy(h + b_start, n_moves_host, b_cnt);
    memcpy(h + b_start + b_cnt, moves_host, (size_t)n * stride * 2);
  } else {
    memset(h + b_start, 0, b_cnt);
  }
  CRL_CUDA(cudaMemcpyAsync(d, h, b_start + b_cnt + b_mv, cudaMemcpyHostToDevice, e->stream));
  rc = launch_games_replay(e, first, n, (const u64*)d, (const u16*)(d + b_start + b_cnt), (const int*)(d + b_start),
                           stride > 0 ? stride : 1, nullptr);
  if (rc) return rc;
  e->tree_ready = false;
  return check_pool_errors(e);
}

int crl_games_get_host(crl_engine* e, int first, int n, uint64_t* boards_host, int32_t* plies_host, int8_t* results_host) {
  CHECK_ENGINE(e);
  if (first < 0 || n <= 0 || first + n > e->G) {
    set_error("crl_games_get_host: bad range");
    return CRL_EINVAL;
  }
  if (boards_host) {
    int rc = ensure_stage(e, (size_t)n * 72);
    if (rc) return rc;
    CRL_CUDA(cudaMemcpy2DAsync(e->h_stage, (size_t)n * 8, e->P.g_cur + first, (size_t)e->G * 8, (size_t)n * 8, 9,
                               cudaMemcpyDeviceToHost, e->stream));
  }
  if (plies_host)
    CRL_CUDA(cudaMemcpyAsync(plies_host, e->P.g_nmoves + first, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
  if (results_host)
    CRL_CUDA(cudaMemcpyAsync(results_host, e->P.g_result + first, (size_t)n, cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  if (boards_host) {
    const u64* s = (const u64*)e->h_stage;
    for (int i = 0; i < n; ++i)
      for (int k = 0; k < 9; ++k) boards_host[(size_t)i * 9 + k] = s[(size_t)k * n + i];
  }
  return CRL_OK;
}

int crl_games_set_active_host(crl_engine* e, int first, int n, const uint8_t* active_host) {
  CHECK_ENGINE(e);
  if (first < 0 || n <= 0 || first + n > e->G || !active_host) {
    set_error("crl_games_set_active_host: bad arguments (first %d, n %d, capacity %d)", first, n, e->G);
    return CRL_EINVAL;
  }
  int rc = ensure_stage(e, (size_t)n);
  if (rc) return rc;
  u8* h = (u8*)e->h_stage;
  for (int i = 0; i < n; ++i) h[i] = active_host[i] ? 1 : 0;
  CRL_CUDA(cudaMemcpyAsync(e->P.g_active + first, h, (size_t)n, cudaMemcpyHostToDevice, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));   // the staging buffer is reused by the next call
  e->tree_ready = false;
  return CRL_OK;
}

int crl_game_moves_host(crl_engine* e, int game, uint16_t* moves_host, int cap, int32_t* n_host) {
  CHECK_ENGINE(e);
  if (game < 0 || game >= e->G || !n_host) {
    set_error("crl_game_moves_host: bad arguments");
    return CRL_EINVAL;
  }
  int n = 0;
  CRL_CUDA(cudaMemcpyAsync(&n, e->P.g_nmoves + game, 4, cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  *n_host = n;
  int m = n < cap ? n : cap;
  if (moves_host && m > 0) {
    CRL_CUDA(cudaMemcpyAsync(moves_host, e->P.g_moves + (size_t)game * MAX_GAME_PLIES, (size_t)m * 2,
                             cudaMemcpyDeviceToHost, e->stream));
    CRL_CUDA(cudaStreamSynchronize(e->stream));
  }
  return CRL_OK;
}

int crl_games_restart_host(crl_engine* e, const int32_t* lanes_host, int n, const uint64_t* start_host) {
  CHECK_ENGINE(e);
  if (n < 0 || (n > 0 && (!lanes_host || !start_host))) {
    set_error("crl_games_restart_host: bad arguments");
    return CRL_EINVAL;
  }
  if (n == 0) return CRL_OK;
  for (int i = 0; i < n; ++i)
    if (lanes_host[i] < 0 || lanes_host[i] >= e->G) {
      set_error("crl_games_restart_host: lane %d out of range (capacity %d)", lanes_host[i], e->G);
      return CRL_EINVAL;
    }
  const size_t b_lanes = ((size_t)n * 4 + 7) / 8 * 8;
  int rc = ensure_stage(e, 72 + b_lanes);
  if (rc) return rc;
  char* h = (char*)e->h_stage;
  char* d = (char*)e->d_stage;
  memcpy(h, start_host, 72);
  memcpy(h + 72, lanes_host, (size_t)n * 4);
  CRL_CUDA(cudaMemcpyAsync(d, h, 72 + b_lanes, cudaMemcpyHostToDevice, e->stream));
  rc = launch_games_replay(e, 0, n, (const u64*)d, nullptr, nullptr, 1, nullptr, nullptr, nullptr, (const int*)(d + 72));
  if (rc) return rc;
  e->tree_ready = false;
  return check_pool_errors(e);
}

int crl_games_moves_host(crl_engine* e, const int32_t* lanes_host, int n, uint16_t* moves_host, int cap, int32_t* n_moves_host) {
  CHECK_ENGINE(e);
  if (n < 0 || cap <= 0 || (n > 0 && (!lanes_host || !moves_host || !n_moves_host))) {
    set_error("crl_games_moves_host: bad arguments");
    return CRL_EINVAL;
  }
  if (n == 0) return CRL_OK;
  for (int i = 0; i < n; ++i)
    if (lanes_host[i] < 0 || lanes_host[i] >= e->G) {
      set_error("crl_games_moves_host: lane %d out of range (capacity %d)", lanes_host[i], e->G);
      return CRL_EINVAL;
    }
  const size_t b_lanes = ((size_t)n * 4 + 7) / 8 * 8, b_cnt = b_lanes, b_mv = (size_t)n * cap * 2;
  int rc = ensure_stage(e, b_lanes + b_cnt + b_mv);
  if (rc) return rc;
  char* h = (char*)e->h_stage;
  char* d = (char*)e->d_stage;
  memcpy(h, lanes_host, (size_t)n * 4);
  CRL_CUDA(cudaMemcpyAsync(d, h, b_lanes, cudaMemcpyHostToDevice, e->stream));
  rc = launch_gather_moves(e, (const int*)d, n, cap, (u16*)(d + b_lanes + b_cnt), (int*)(d + b_lanes));
  if (rc) return rc;
  CRL_CUDA(cudaMemcpyAsync(h + b_lanes, d + b_lanes, b_cnt + b_mv, cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  memcpy(n_moves_host, h + b_lanes, (size_t)n * 4);
  memcpy(moves_host, h + b_lanes + b_cnt, b_mv);
  return CRL_OK;
}

int crl_games_play_host(crl_engine* e, const uint16_t* moves_host, uint8_t* accepted_host) {
  CHECK_ENGINE(e);
  if (!moves_host) {
    set_error("crl_games_play_host: null moves");
    return CRL_EINVAL;
  }
  const size_t G = e->G, b_mv = (G * 2 + 7) / 8 * 8;
  int rc = ensure_stage(e, b_mv + G);
  if (rc) return rc;
  char* h = (char*)e->h_stage;
  char* d = (char*)e->d_stage;
  memcpy(h, moves_host, G * 2);
  CRL_CUDA(cudaMemcpyAsync(d, h, b_mv, cudaMemcpyHostToDevice, e->stream));
  rc = launch_game_moves(e, (const u16*)d, (u8*)(d + b_mv));
  if (rc) return rc;
  e->tree_ready = false;
  if (accepted_host) CRL_CUDA(cudaMemcpyAsync(accepted_host, d + b_mv, G, cudaMemcpyDeviceToHost, e->stream));
  return check_pool_errors(e);
}

int crl_games_legal_host(crl_engine* e, int first, int n, uint16_t* legal_host, int32_t* n_legal_host) {
  CHECK_ENGINE(e);
  if (first < 0 || n <= 0 || first + n > e->G || !legal_host || !n_legal_host) {
    set_error("crl_games_legal_host: bad arguments (first %d, n %d, capacity %d)", first, n, e->G);
    return CRL_EINVAL;
  }
  const size_t b_legal = (size_t)n * MAX_MOVES * 2, b_cnt = (size_t)n * 4;
  int rc = ensure_stage(e, b_legal + b_cnt);
  if (rc) return rc;
  char* d = (char*)e->d_stage;
  rc = launch_game_info(e, first, n, (u16*)d, (int*)(d + b_legal));
  if (rc) return rc;
  CRL_CUDA(cudaMemcpyAsync(legal_host, d, b_legal, cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaMemcpyAsync(n_legal_host, d + b_legal, b_cnt, cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  return CRL_OK;
}

int crl_games_policy_move_host(crl_engine* e, const uint8_t* mask_host, uint16_t* picks_host) {
  CHECK_ENGINE(e);
  const size_t G = e->G;
  int rc = route_slots(e, "crl_games_policy_move_host");
  if (rc) return rc;
  rc = ensure_stage(e, G);
  if (rc) return rc;
  const u8* mask_dev = nullptr;
  if (mask_host) {
    memcpy(e->h_stage, mask_host, G);
    CRL_CUDA(cudaMemcpyAsync(e->d_stage, e->h_stage, G, cudaMemcpyHostToDevice, e->stream));
    mask_dev = (const u8*)e->d_stage;
  }
  rc = tree_policy_move(e, mask_dev, e->d_tmp_moves);
  if (rc) return rc;
  e->tree_ready = false;
  if (picks_host) CRL_CUDA(cudaMemcpyAsync(picks_host, e->d_tmp_moves, G * 2, cudaMemcpyDeviceToHost, e->stream));
  return check_pool_errors(e);
}

// crl_games_ab_move_host (salt_host NULL), crl_games_ab_pick_host and crl_games_ab_search_host: stage the salts (offset
// 0) and the mask, search, copy the outputs back
static int ab_search_host(crl_engine* e, const char* fn, const uint8_t* mask_host, int depth, int qdepth, bool reps,
                          int margin, int pick_plies, const uint64_t* salt_host, uint16_t* move_host,
                          int32_t* score_host, int64_t* nodes_host) {
  const size_t G = e->G;
  const size_t off = salt_host ? G * 8 : 0;
  const u8* mask_dev = nullptr;
  if (salt_host || mask_host) {
    int rc = ensure_stage(e, off + G);
    if (rc) return rc;
    if (salt_host) memcpy(e->h_stage, salt_host, G * 8);
    if (mask_host) {
      memcpy((char*)e->h_stage + off, mask_host, G);
      mask_dev = (const u8*)e->d_stage + off;
    }
    CRL_CUDA(cudaMemcpyAsync(e->d_stage, e->h_stage, off + (mask_host ? G : 0), cudaMemcpyHostToDevice, e->stream));
  }
  int rc = launch_ab_move(e, mask_dev, depth, qdepth, salt_host ? (const u64*)e->d_stage : nullptr, margin, pick_plies,
                          reps, fn);
  if (rc) return rc;
  if (move_host) CRL_CUDA(cudaMemcpyAsync(move_host, e->ab_out_move, G * 2, cudaMemcpyDeviceToHost, e->stream));
  if (score_host) CRL_CUDA(cudaMemcpyAsync(score_host, e->ab_out_score, G * 4, cudaMemcpyDeviceToHost, e->stream));
  if (nodes_host) CRL_CUDA(cudaMemcpyAsync(nodes_host, e->ab_out_nodes, G * 8, cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  return CRL_OK;
}

int crl_games_ab_move_host(crl_engine* e, const uint8_t* mask_host, int depth, int qdepth, uint16_t* move_host,
                           int32_t* score_host, int64_t* nodes_host) {
  CHECK_ENGINE(e);
  return ab_search_host(e, "crl_games_ab_move_host", mask_host, depth, qdepth, false, 0, 0, nullptr, move_host,
                        score_host, nodes_host);
}

int crl_games_ab_pick_host(crl_engine* e, const uint8_t* mask_host, int depth, int qdepth, int margin, int pick_plies,
                           const uint64_t* salt_host, uint16_t* move_host, int32_t* score_host, int64_t* nodes_host) {
  CHECK_ENGINE(e);
  if (!salt_host) {
    set_error("crl_games_ab_pick_host: salt_host is NULL (one salt per lane)");
    return CRL_EINVAL;
  }
  return ab_search_host(e, "crl_games_ab_pick_host", mask_host, depth, qdepth, false, margin, pick_plies, salt_host,
                        move_host, score_host, nodes_host);
}

int crl_games_ab_search_host(crl_engine* e, const uint8_t* mask_host, int depth, int qdepth, int flags, int margin,
                             int pick_plies, const uint64_t* salt_host, uint16_t* move_host, int32_t* score_host,
                             int64_t* nodes_host) {
  CHECK_ENGINE(e);
  const char* fn = "crl_games_ab_search_host";
  if (flags & ~CRL_AB_REPETITIONS) {
    set_error("%s: unknown flag bits 0x%x", fn, (unsigned)(flags & ~CRL_AB_REPETITIONS));
    return CRL_EINVAL;
  }
  if (!salt_host && (margin || pick_plies)) {
    set_error("%s: margin %d / pick_plies %d without salt_host (they apply to the seeded pick only)", fn, margin,
              pick_plies);
    return CRL_EINVAL;
  }
  return ab_search_host(e, fn, mask_host, depth, qdepth, (flags & CRL_AB_REPETITIONS) != 0, margin, pick_plies,
                        salt_host, move_host, score_host, nodes_host);
}

int crl_games_ab_root_scores_host(crl_engine* e, int32_t* scores_host, int32_t* counts_host) {
  CHECK_ENGINE(e);
  if (!scores_host || !counts_host) {
    set_error("crl_games_ab_root_scores_host: null output");
    return CRL_EINVAL;
  }
  if (!e->ab_moves) {
    set_error("crl_games_ab_root_scores_host: no alpha-beta call has run on this engine");
    return CRL_ESTATE;
  }
  const size_t G = e->G;
  CRL_CUDA(cudaMemcpyAsync(scores_host, e->ab_score, G * MAX_MOVES * 4, cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaMemcpyAsync(counts_host, e->ab_cnt, G * 4, cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  for (size_t g = 0; g < G; ++g) {                   // entries past a lane's count hold older calls' scores
    const int c = counts_host[g] > 0 ? counts_host[g] : 0;
    memset(scores_host + g * MAX_MOVES + c, 0, (MAX_MOVES - c) * 4);
  }
  return CRL_OK;
}

int crl_set_reuse(crl_engine* e, int enable) {
  CHECK_ENGINE(e);
  if (enable && !e->P.nodes_prev) {
    // the second set of tree pools: node records, and the two edge arrays a twin lookup reads (child index, prior)
    const size_t G = e->G;
    int rc = pool_alloc(e, &e->P.nodes_prev, G * e->NN);
    if (rc == CRL_OK) rc = pool_alloc(e, &e->P.e_prior_prev, G * e->EA);
    if (rc == CRL_OK) rc = pool_alloc(e, &e->P.e_child_prev, G * e->EA);
    if (rc != CRL_OK) {
      e->P.nodes_prev = nullptr;   // (what was allocated stays in e->allocs and is freed with the engine)
      return rc;
    }
  }
  CRL_CUDA(cudaMemsetAsync(e->P.g_prev_root, 0xFF, sizeof(int) * (size_t)e->G, e->stream));
  e->reuse = enable != 0;
  e->tree_ready = false;
  return CRL_OK;
}

int crl_mcts_set_row_bound(crl_engine* e, int max_running_games) {
  CHECK_ENGINE(e);
  e->row_bound = max_running_games > 0 && max_running_games < e->G ? max_running_games : 0;
  return CRL_OK;
}

int crl_reuse_count_host(crl_engine* e, int64_t* reused_host) {
  CHECK_ENGINE(e);
  if (!reused_host) {
    set_error("crl_reuse_count_host: null output");
    return CRL_EINVAL;
  }
  long long c = 0;
  CRL_CUDA(cudaMemcpyAsync(&c, e->P.counters + 2, sizeof(c), cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  *reused_host = c;
  return CRL_OK;
}

int crl_mcts_begin_move(crl_engine* e) {
  CHECK_ENGINE(e);
  int rc = route_slots(e, "crl_mcts_begin_move");
  if (rc) return rc;
  rc = tree_begin_move(e, nullptr, e->reuse);
  if (rc) return rc;
  e->tree_ready = true;
  return CRL_OK;
}

int crl_mcts_simulate(crl_engine* e, int n_sims, int inflight) {
  CHECK_ENGINE(e);
  if (!e->tree_ready) {
    set_error("crl_mcts_simulate: call crl_mcts_begin_move first");
    return CRL_ESTATE;
  }
  if (inflight < 1 || inflight > e->Kmax) {
    set_error("crl_mcts_simulate: inflight = %d, but the engine was created for at most %d in-flight simulations "
              "per game (crl_create_ex max_inflight)", inflight, e->Kmax);
    return CRL_EINVAL;
  }
  if (n_sims < 0 || n_sims > e->NN - 1) {
    set_error("crl_mcts_simulate: %d simulations exceed the node pool (%d per game)", n_sims, e->NN - 1);
    return CRL_EINVAL;
  }
  int rc = route_slots(e, "crl_mcts_simulate");
  if (rc) return rc;
  return tree_simulate(e, n_sims, inflight);
}

int crl_mcts_root_stats_host(crl_engine* e, int32_t* child_visits, double* child_values, float* child_priors,
                             uint16_t* child_moves, uint16_t* child_replies, int8_t* child_results, int32_t* n_children,
                             int32_t* root_visits, double* root_values) {
  CHECK_ENGINE(e);
  const size_t G = e->G, GM = G * MAX_MOVES;
  // staging layout
  size_t o_vis = 0, o_val = o_vis + GM * 4, o_pri = o_val + GM * 8, o_mv = o_pri + GM * 4, o_rp = o_mv + GM * 2,
         o_rs = o_rp + GM * 2, o_nc = (o_rs + GM + 7) / 8 * 8, o_rv = o_nc + G * 4, o_rw = (o_rv + G * 4 + 7) / 8 * 8,
         total = o_rw + G * 8;
  int rc = ensure_stage(e, total);
  if (rc) return rc;
  char* d = (char*)e->d_stage;
  {
    LaunchScope ls(e, KC_TREE);
    k_root_stats<<<e->G, 64, 0, e->stream>>>(e->P, (int*)(d + o_vis), (double*)(d + o_val), (float*)(d + o_pri),
                                             (u16*)(d + o_mv), (u16*)(d + o_rp), (int8_t*)(d + o_rs), (int*)(d + o_nc),
                                             (int*)(d + o_rv), (double*)(d + o_rw));
    CRL_CUDA(cudaGetLastError());
  }
#define OUT(ptr, off, bytes) \
  if (ptr) CRL_CUDA(cudaMemcpyAsync(ptr, d + (off), (bytes), cudaMemcpyDeviceToHost, e->stream))
  OUT(child_visits, o_vis, GM * 4);
  OUT(child_values, o_val, GM * 8);
  OUT(child_priors, o_pri, GM * 4);
  OUT(child_moves, o_mv, GM * 2);
  OUT(child_replies, o_rp, GM * 2);
  OUT(child_results, o_rs, GM);
  OUT(n_children, o_nc, G * 4);
  OUT(root_visits, o_rv, G * 4);
  OUT(root_values, o_rw, G * 8);
#undef OUT
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  drain_profile(e);
  return check_pool_errors(e);
}

int crl_mcts_commit_host(crl_engine* e, const int32_t* pick_host, uint16_t* out_moves_host, int apply) {
  CHECK_ENGINE(e);
  if (!pick_host) {
    set_error("crl_mcts_commit_host: null picks");
    return CRL_EINVAL;
  }
  const size_t G = e->G;
  CRL_CUDA(cudaMemcpyAsync(e->d_tmp_pick, pick_host, G * 4, cudaMemcpyHostToDevice, e->stream));
  int rc = tree_commit(e, e->d_tmp_pick, e->d_tmp_moves, apply);
  if (rc) return rc;
  if (out_moves_host)
    CRL_CUDA(cudaMemcpyAsync(out_moves_host, e->d_tmp_moves, G * 4, cudaMemcpyDeviceToHost, e->stream));
  if (apply) e->tree_ready = false;
  return check_pool_errors(e);
}

int crl_mcts_node_dump_host(crl_engine* e, int game, crl_node_host* out, int cap, int32_t* n_host) {
  CHECK_ENGINE(e);
  if (game < 0 || game >= e->G || !out || cap <= 0 || !n_host) {
    set_error("crl_mcts_node_dump_host: bad arguments");
    return CRL_EINVAL;
  }
  int n = 0;
  CRL_CUDA(cudaMemcpyAsync(&n, e->P.g_nnodes + game, 4, cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  *n_host = n;
  int m = n < cap ? n : cap;
  if (m <= 0) return CRL_OK;
  int rc = ensure_stage(e, (size_t)m * sizeof(crl_node_host));
  if (rc) return rc;
  {
    LaunchScope ls(e, KC_TREE);
    k_node_dump<<<div_up(m, 128), 128, 0, e->stream>>>(e->P, game, (crl_node_host*)e->d_stage, m);
    CRL_CUDA(cudaGetLastError());
  }
  CRL_CUDA(cudaMemcpyAsync(out, e->d_stage, (size_t)m * sizeof(crl_node_host), cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  return CRL_OK;
}

int crl_counters_host(crl_engine* e, int64_t* out3) {
  CHECK_ENGINE(e);
  if (!out3) return CRL_EINVAL;
  long long c[4];
  CRL_CUDA(cudaMemcpyAsync(c, e->P.counters, sizeof(c), cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  out3[0] = c[0];
  out3[1] = c[1];
  out3[2] = e->launches;
  return CRL_OK;
}

int crl_profile(crl_engine* e, int enable) {
  CHECK_ENGINE(e);
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  drain_profile(e);
  e->profiling = enable != 0;
  for (int i = 0; i < KC_COUNT; ++i) {
    e->prof_ms[i] = 0;
    e->prof_launches[i] = 0;
  }
  return CRL_OK;
}
int crl_profile_read_host(crl_engine* e, double* ms_by_class, int64_t* launches_by_class, int n_classes) {
  CHECK_ENGINE(e);
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  drain_profile(e);
  for (int i = 0; i < n_classes && i < KC_COUNT; ++i) {
    if (ms_by_class) ms_by_class[i] = e->prof_ms[i];
    if (launches_by_class) launches_by_class[i] = e->prof_launches[i];
  }
  return CRL_OK;
}

}  // extern "C"
