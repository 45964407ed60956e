// engine.cuh -- host-side engine object behind the C ABI (include/chessrl_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <utility>
#include <vector>

#include "../../include/chessrl_b200.h"
#include "tree_core.cuh"

namespace crl {

enum KernelClass {
  KC_MOVEGEN = 0,   // movegen / make / perft / frontier
  KC_ENCODE = 1,    // board -> planes
  KC_CONV = 2,      // tcgen05 implicit-GEMM 3x3 convolutions (the dominant kernel)
  KC_HEADS = 3,     // policy / value heads
  KC_TREE = 4,      // select / expand / reply / backup
  KC_GAME = 5,      // game record kernels
  KC_HASHEVAL = 6,
  KC_COUNT = 7
};

struct NetWeights;   // net.cu

struct crl_engine_impl {
  int device = 0;
  cudaStream_t stream = nullptr;
  int G = 0, NN = 0, EA = 0;
  int Kmax = 1;                    // in-flight simulations per game the workspaces are sized for
  int R = 0;                       // evaluation row capacity = G * Kmax
  int cur_rows = 0;                // host bound on the rows of the batch being launched (G, or G*K in wave mode)
  int row_bound = 0;               // crl_mcts_set_row_bound: at most this many games are running (0 = no promise)
  Pools P{};                       // device pointers
  std::vector<void*> allocs;       // everything cudaMalloc'ed
  int16_t* d_label_of = nullptr;   // [5][64][64]
  std::vector<int16_t> h_label_of;
  // evaluator of every network slot (crl_net_select_slot picks the slot the configuration calls act on)
  int eval_kind[CRL_NET_SLOTS] = {CRL_EVAL_NET, CRL_EVAL_NET};
  uint64_t eval_seed[CRL_NET_SLOTS] = {0, 0};
  int eval_bits[CRL_NET_SLOTS] = {24, 24};
  bool slot_configured[CRL_NET_SLOTS] = {true, false};   // slot 1 has no evaluator until a load or crl_set_evaluator
  int sel_slot = 0;
  // two-network routing (DESIGN.md 3.5): slot k's rows of a batch are rows k * slot_stride + r of the list, policy, value
  // and statistics buffers below (and of the logits); 0 until slot 1 is first configured, the buffers then hold 2 slots
  long long slot_stride = 0;
  std::vector<uint8_t> h_players;      // [2][G] host copy of the players (white slot, black slot); empty = all slot 0
  int lanes_on_slot1 = 0;              // lanes that name slot 1 as a player
  int search_slots = 1;                // slots the current search routes rows to (2 iff lanes_on_slot1 > 0)
  // evaluation workspaces (sized for G rows)
  __nv_bfloat16* d_planes = nullptr;   // [G][64][128]
  float* d_policy = nullptr;           // [G][1968]
  float* d_value = nullptr;            // [G]
  float* d_stats = nullptr;            // [G][2] softmax statistics (max logit, 1 / sum exp) of the rows evaluated by the network
  PolicyView pview{};                  // how the search kernels read the last evaluation batch (set by launch_eval_batch)
  NetWeights* nets[CRL_NET_SLOTS] = {nullptr, nullptr};
  NetWeights* net = nullptr;           // nets[sel_slot]
  bool tree_ready = false;
  int* d_list[2] = {nullptr, nullptr};   // compacted evaluation batches A (after our move) / B (leaf)
  int* d_n = nullptr;                    // row counts: [0] / [1] batches A / B (slot 0), [2] scratch, [4] / [5] slot 1's
  u16* d_tmp_moves = nullptr;            // [2*G] scratch for picks
  int* d_tmp_pick = nullptr;             // [G]
  // device-driven perft (crl_perft_root_host): two frontier buffers of perft_cap boards + control block
  u64* perft_buf[2] = {nullptr, nullptr};
  long long perft_cap = 0;
  unsigned long long* perft_ctl = nullptr;
  int perft_pair = 0;                    // 0: expand the last-but-one ply into HBM, then walk it (default: measured
                                         // faster); CRL_PERFT_PAIR=5 / 6: the last two plies in one pass (k_perft_pair,
                                         // 96- / 80-register build)
  bool perft_pdl = true;                 // plies launched as programmatic dependent launches (CRL_NO_PDL=1: plain launches)
  // fixed-depth alpha-beta (crl_games_ab_move_host): scratch allocated at the first call; items are lane * MAX_MOVES + k
  u16* ab_moves = nullptr;               // [G][MAX_MOVES] root moves
  int* ab_cnt = nullptr;                 // [G] root move count, -1 for a lane that is not searched
  int* ab_items = nullptr;               // [G * MAX_MOVES] items of this call (k_ab_root appends them)
  int* ab_score = nullptr;               // [G][MAX_MOVES] exact value of every root child
  unsigned long long* ab_nodes = nullptr;   // [G][MAX_MOVES] positions visited below every root child
  unsigned long long* ab_ctl = nullptr;  // [0] items, [1] items taken
  u16* ab_out_move = nullptr;            // [G]
  int* ab_out_score = nullptr;           // [G]
  long long* ab_out_nodes = nullptr;     // [G]
  int ab_grid = 0;                       // blocks of k_ab_items that fill the GPU
  // repetitions on (crl_games_ab_search_host CRL_AB_REPETITIONS): allocated at the first such call
  u64* ab_rep_keys = nullptr;            // [G][AB_REP_KEYS] keys of each searched root's reversible run, root first
  int* ab_rep_n = nullptr;               // [G] earlier positions staged per lane
  int ab_rep_grid = 0;                   // blocks of k_ab_items<true> that fill the GPU
  // pinned staging
  void* h_stage = nullptr;
  size_t h_stage_bytes = 0;
  void* d_stage = nullptr;
  size_t d_stage_bytes = 0;
  // CUDA graph of one lockstep simulation (replayed n_sims times); rebuilt when the evaluator changes
  bool own_stream = false;
  bool use_graph = true;
  cudaGraphExec_t sim_graph[2] = {nullptr, nullptr};   // one per tree parity (the pools swap roles under evaluation reuse)
  unsigned long long sim_graph_key[2] = {0, 0};
  int tree_parity = 0;
  bool reuse = false;              // crl_set_reuse: expansions take evaluations from the previous move's tree
  long long sim_graph_launches = 0;
  bool capturing = false;
  // accounting
  long long launches = 0;
  bool profiling = false;
  double prof_ms[KC_COUNT] = {0};
  long long prof_launches[KC_COUNT] = {0};
  std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> prof_pending;
};

void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t err, const char* what);

#define CRL_CUDA(expr)                                        \
  do {                                                        \
    cudaError_t _e = (expr);                                  \
    if (_e != cudaSuccess) return cuda_fail(_e, #expr);       \
  } while (0)

// RAII bracket that counts a launch and, in profiling mode, times it with CUDA events on the engine stream
struct LaunchScope {
  crl_engine_impl* e;
  int cls;
  cudaEvent_t a = nullptr, b = nullptr;
  LaunchScope(crl_engine_impl* e_, int cls_, int n_launches = 1) : e(e_), cls(cls_) {
    e->launches += n_launches;
    e->prof_launches[cls] += n_launches;
    if (e->profiling && !e->capturing) {
      cudaEventCreate(&a);
      cudaEventCreate(&b);
      cudaEventRecord(a, e->stream);
    }
  }
  ~LaunchScope() {
    if (e->profiling && !e->capturing) {
      cudaEventRecord(b, e->stream);
      e->prof_pending.push_back({cls, {a, b}});
    }
  }
};

inline int div_up(long long a, long long b) { return (int)((a + b - 1) / b); }

// ---- kernel launchers (defined in the .cu files) ---------------------------------------------------
int launch_movegen(crl_engine_impl* e, const u64* boards, int n, u16* moves, int* counts, u8* flags);
int launch_movegen_warp(crl_engine_impl* e, const u64* boards, int n, u16* moves, int* counts, u8* flags);
int launch_make(crl_engine_impl* e, u64* boards, int n, const u16* moves);
int launch_perft(crl_engine_impl* e, const u64* boards, int n, int depth, int bulk, unsigned long long* nodes);
int launch_frontier(crl_engine_impl* e, const u64* boards, int n, const long long* offsets, u64* out,
                    long long out_n, int* counts);
int launch_perft_root(crl_engine_impl* e, const u64* root, u64* buf0, u64* buf1, long long cap, unsigned long long* ctl,
                      int depth, int bulk, long long min_frontier, int pair, int shard, int n_shards, long long shard_min);
int launch_encode_boards(crl_engine_impl* e, const u64* boards, const u64* hist, const u8* hist_len, int n,
                         __nv_bfloat16* planes);
int launch_policy_index(crl_engine_impl* e, const u16* moves, const int* counts, int n, int16_t* idx);
// fixed-depth alpha-beta of every active, unfinished lane with mask_dev[g] != 0 (null: all) into e->ab_out_*; salt_dev null:
// the first maximum, else the seeded near-best pick of DESIGN.md 3.7 (a salt per lane); reps: repetitions scored 0
// (DESIGN.md 3.6).  CRL_EINVAL for out-of-range limits, reported as function `fn`
int launch_ab_move(crl_engine_impl* e, const u8* mask_dev, int depth, int qdepth, const u64* salt_dev, int margin,
                   int pick_plies, bool reps, const char* fn);
int launch_hash_eval_boards(crl_engine_impl* e, const u64* boards, int n, u64 seed, int bits, float* policy,
                            float* value);

// tree / game
int launch_games_replay(crl_engine_impl* e, int first, int n, const u64* start_aos, const u16* moves,
                        const int* n_moves, int stride, u8* accepted, u64* records = nullptr,
                        int* n_records = nullptr, const int* lanes = nullptr);
int launch_gather_moves(crl_engine_impl* e, const int* lanes, int n, int cap, u16* out, int* n_out);
int launch_game_info(crl_engine_impl* e, int first, int n, u16* legal, int* n_legal);
int launch_game_moves(crl_engine_impl* e, const u16* moves_per_game /*[G]*/, u8* accepted /*[G] or null*/);
int launch_eval_batch(crl_engine_impl* e, int which_mode);   // encodes eval_list rows and runs the evaluator
int tree_begin_move(crl_engine_impl* e, const u8* mask_dev, bool use_prev);
int tree_simulate(crl_engine_impl* e, int n_sims, int K);
int tree_run_steps(crl_engine_impl* e, int n_steps, int K);
int tree_policy_move(crl_engine_impl* e, const u8* mask_dev, u16* picks_dev);
int tree_commit(crl_engine_impl* e, const int* pick_dev, u16* out_moves_dev, int apply);

// net
int net_create(crl_engine_impl* e, int slot);
void net_destroy(crl_engine_impl* e);
// the network of slot k, created with its planes buffer on first use (the result buffers must hold two slots already)
int net_slot_ensure(crl_engine_impl* e, int slot);
// lays the row lists and result buffers out for two slots (once, at the first configuration of slot 1)
int net_two_slot_layout(crl_engine_impl* e);
int net_load(crl_engine_impl* e, const float* const* w, const int64_t* sizes, int n);
// n_dev may be null (then n_host rows); otherwise the row count is read on the device and n_host is the bound
// view_out != null: the caller reads the policy through a PolicyView (the search kernels); where the network path allows it
// the softmax kernel then writes only its statistics to e->d_stats and *view_out points at the logits, otherwise at `policy`
int net_forward(crl_engine_impl* e, const __nv_bfloat16* planes, int n_host, const int* n_dev, float* policy,
                float* value, __nv_bfloat16* dbg_out = nullptr, int dbg_layer = -1, PolicyView* view_out = nullptr);
// net_forward with the network of slot `slot` (a search batch of that slot's rows; `planes` = net_planes_buf)
int net_forward_slot(crl_engine_impl* e, int slot, const void* planes, int n_host, const int* n_dev, float* policy,
                     float* value, PolicyView* view_out);
// the buffer the search encodes slot `slot`'s rows into (R + 2 bf16 rows; e4m3 rows while the slot runs fp8)
void* net_planes_buf(const crl_engine_impl* e, int slot);
int net_debug_tower(crl_engine_impl* e, const __nv_bfloat16* planes, int n, int layer, __nv_bfloat16* act_out,
                    float* logits_out, __nv_bfloat16* pf_out, float* vf_out, float* policy, float* value);
int net_debug_conv(crl_engine_impl* e, int layer, const __nv_bfloat16* in, int cin, int n, const __nv_bfloat16* residual,
                   __nv_bfloat16* out, int relu);
// fp8 evaluation (crl_net_calibrate_host, crl_net_load_fp8_host, crl_net_set_precision)
int net_calibrate(crl_engine_impl* e, const __nv_bfloat16* planes, int n, float* amax_host);
int net_load_fp8(crl_engine_impl* e, const float* const* w, const int64_t* sizes, int n, const float* act_amax);
int net_set_precision(crl_engine_impl* e, int precision);
// true while slot `slot`'s fp8 tower is selected: the search then encodes e4m3 planes for that slot
bool net_fp8(const crl_engine_impl* e, int slot);

}  // namespace crl

struct crl_engine : public crl::crl_engine_impl {};
