/* chessrl_b200.h -- C ABI of libchessrl_b200.so, the B200-native lockstep self-play engine that stands in
 * for the self-play hot path of AIRLegend/ChessRL.
 *
 * The reference has no FFI: its hot path sits behind Python classes whose arithmetic lives in python-chess
 * and TensorFlow.  Each entry point below names the reference interface it replaces (file:line under
 * /root/reference/src/chessrl); INTEGRATION.md shows the ctypes binding a maintainer adds on the reference
 * side.  All compute runs in sm_100a CUDA kernels; there is no CPU path behind any of these calls.
 *
 * Conventions
 *   - every function returns CRL_OK (0) or a negative crl_status; crl_last_error() gives the text.
 *   - "dev" pointers are CUDA device pointers owned by the caller (e.g. torch tensors); "host" pointers are
 *     ordinary host memory.  The library owns only what crl_create allocates.
 *   - launches go to the cudaStream_t given at crl_create (pass torch's current stream); functions taking
 *     only device pointers do not synchronise; functions with host pointers synchronise that stream.
 *   - one engine per (process, GPU); calls on one handle are not re-entrant.
 *
 * Data formats
 *   board record : 9 x uint64.  [0..5] pawns knights bishops rooks queens kings, [6] white, [7] black,
 *                  [8] meta = turn(bit0,1=white) | castling KQkq(bits1-4) | ep+1(bits5-11) |
 *                  halfmove(bits12-23) | fullmove(bits24-37) | ply=len(move_stack)(bits38-51) |
 *                  reversible-run length(bits52-59).
 *                  Device batches are structure-of-arrays: word k of board i at boards[k*n + i].
 *                  Host batches (the *_host calls) are array-of-structures: board i at boards[9*i].
 *   move word    : from | to<<6 | promo<<12 (promo 0 none, 1 N, 2 B, 3 R, 4 Q); 0xFFFF = no move.
 *   planes       : bf16 [n][8][8][128], NHWC, row 0 = rank 8, channel order of netencoder.get_game_state,
 *                  channel 127 = zero padding.
 *   policy index : position in netencoder.get_uci_labels() (0..1967).
 */
#ifndef CHESSRL_B200_H
#define CHESSRL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CRL_RECORD_WORDS 9
#define CRL_MAX_MOVES 256
#define CRL_N_LABELS 1968
#define CRL_PLANE_C 128
#define CRL_RESULT_NONE 2
#define CRL_MOVE_NONE 0xFFFF
#define CRL_N_WEIGHT_TENSORS 140
#define CRL_MAX_INFLIGHT 64

typedef enum {
  CRL_OK = 0,
  CRL_EINVAL = -1,   /* bad argument */
  CRL_ECUDA = -2,    /* CUDA runtime / driver error */
  CRL_ENOMEM = -3,   /* allocation failed or a node / edge pool overflowed */
  CRL_ESTATE = -4    /* call order violated (e.g. simulate before begin_move, no weights loaded) */
} crl_status;

typedef struct crl_engine crl_engine;

/* evaluator used by the tree search */
#define CRL_EVAL_NET 0   /* the policy/value ResNet (model.py:31-63) on tcgen05 tensor cores            */
#define CRL_EVAL_HASH 1  /* deterministic position-hash evaluator, bit-identical to                     */
                         /* oracle/chessrl_oracle.py hash_evaluator -- for visit-count parity tests     */

/* ---- lifecycle ---------------------------------------------------------------------------------- */
/* max_games: lockstep lanes; max_nodes: tree nodes per game (>= sims per move + 1); avg_moves: edge-pool
 * sizing hint (edges per game = max_nodes * avg_moves, 0 -> 64); stream: cudaStream_t or NULL. */
int crl_create(crl_engine** out, int device, int max_games, int max_nodes, int avg_moves, void* stream);
/* max_inflight (1..CRL_MAX_INFLIGHT): in-flight simulations per game the evaluation workspaces are sized for =
 * the reference's `threads` (SelfPlayTree(root, threads), mctree.py:155-157; selfplay.py --threads, default 6).
 * crl_create == crl_create_ex(..., 1, stream). */
int crl_create_ex(crl_engine** out, int device, int max_games, int max_nodes, int avg_moves, int max_inflight,
                  void* stream);
int crl_destroy(crl_engine* e);
const char* crl_last_error(void);
int crl_version(void);

/* ---- rules: python-chess behind game.Game ------------------------------------------------------- */
/* Game.get_legal_moves (game.py:43-57): legal moves in python-chess generation order.
 * moves_dev [n][CRL_MAX_MOVES], counts_dev [n], flags_dev [n] (bit0 in check, bit1 legal ep exists; may be NULL) */
int crl_movegen(crl_engine* e, const uint64_t* boards_dev, int n, uint16_t* moves_dev, int32_t* counts_dev,
                uint8_t* flags_dev);
/* test hook: the same lists from the WARP-COOPERATIVE generator (32 lanes on one board; csrc/warp_gen.cuh) that the tree
 * kernels and the small breadth-first perft plies use where boards are few and latency is everything */
int crl_debug_movegen_warp(crl_engine* e, const uint64_t* boards_dev, int n, uint16_t* moves_dev, int32_t* counts_dev,
                           uint8_t* flags_dev);
/* Board.push behind Game.move (game.py:28-41), no legality check; in place. moves_dev [n]; 0xFFFF = skip */
int crl_make_moves(crl_engine* e, uint64_t* boards_dev, int n, const uint16_t* moves_dev);
/* perft: each lane walks its own subtree depth-first; bulk != 0 counts the last ply without making moves */
int crl_perft(crl_engine* e, const uint64_t* boards_dev, int n, int depth, int bulk, uint64_t* nodes_dev);
/* perft of ONE position in one call, no host round trip between plies: breadth-first plies on the device (children
 * placed with warp-aggregated atomics, arbitrary order) until the frontier holds >= min_frontier boards, then one
 * depth-first walk per lane (bulk as in crl_perft).  root_host [9] (AoS record).  Outputs: *total_host = perft(depth);
 * Experimental, off by default (measured slower): CRL_PERFT_PAIR=5 or 6 in the environment at crl_create time runs the
 * last two plies as ONE pass when the stored frontier sits two plies above the leaves (each board's children are dealt
 * to the lanes of a warp, made in registers and counted; the last-but-one ply is never stored).
 * optional *lanes_host = boards the walk ran on in lockstep (the stored frontier, or the boards of the last-but-one ply
 * when the two-ply pass ran), *bfs_plies_host = plies expanded breadth-first into HBM.
 * The frontier buffers are owned by the engine and grow on demand (CRL_ENOMEM if they cannot). */
int crl_perft_root_host(crl_engine* e, const uint64_t* root_host, int depth, int bulk, int64_t min_frontier,
                        uint64_t* total_host, int64_t* lanes_host, int32_t* bfs_plies_host);
/* the same perft SHARDED over n_shards callers (one per GPU): every caller expands the same first plies on its own device;
 * the first ply whose input frontier holds >= shard_min_frontier boards keeps only the children whose record hashes to
 * `shard` (the atomic placement orders a frontier differently in every call, so an index range would not partition it),
 * and the caller goes on alone (further plies until its own frontier holds >= min_frontier boards, then the walk).
 * *total_host = THIS shard's count; the sum over the shards is perft(depth) (one all_reduce(sum), SURVEY.md 8e).  No board
 * crosses a link. */
int crl_perft_root_shard_host(crl_engine* e, const uint64_t* root_host, int depth, int bulk, int64_t min_frontier, int shard,
                              int n_shards, int64_t shard_min_frontier, uint64_t* total_host, int64_t* lanes_host,
                              int32_t* bfs_plies_host);
/* one breadth-first ply: children of board i are written at offsets_dev[i] (exclusive scan of counts).
 * Call with out_dev == NULL to get counts only. */
int crl_expand_frontier(crl_engine* e, const uint64_t* boards_dev, int n, const int64_t* offsets_dev,
                        uint64_t* out_dev, int64_t out_n, int32_t* counts_dev);
/* host-buffer convenience (AoS records): replay `n_moves` moves through Game.move semantics (illegal moves are
 * rejected and skipped, game.py:37-41) and report what Game exposes.  Outputs may be NULL.
 *   legal_host [CRL_MAX_MOVES], n_legal_host, result_host (Game.get_result, CRL_RESULT_NONE = None),
 *   accepted_host [n_moves] (1 = move was legal and played), final_host [9] */
int crl_game_replay_host(crl_engine* e, const uint64_t* start_host, const uint16_t* moves_host, int n_moves,
                         uint16_t* legal_host, int32_t* n_legal_host, int8_t* result_host,
                         uint8_t* accepted_host, uint64_t* final_host);

/* the same replay, additionally returning the record after EVERY accepted move (records_host [(n_moves+1)][9],
 * record 0 = start position; *n_records_host = accepted moves + 1): the positions Board.copy() + pop() walks back
 * through for the history planes (netencoder.py:58-67) and DatasetGame.augment_game replays ply by ply
 * (dataset.py:21-43) -- one device round trip per game instead of one per ply. */
int crl_game_replay_records_host(crl_engine* e, const uint64_t* start_host, const uint16_t* moves_host, int n_moves,
                                 uint16_t* legal_host, int32_t* n_legal_host, int8_t* result_host,
                                 uint8_t* accepted_host, uint64_t* records_host, int32_t* n_records_host);

/* ---- encoding: netencoder ------------------------------------------------------------------------- */
/* netencoder.get_game_state (netencoder.py:72-91).  hist_dev: bitboards of the previous positions,
 * word k of the i-th previous position of board b at hist_dev[((i*8)+k)*n + b], i = 0..7 (may be NULL);
 * hist_len_dev [n]: how many of them exist (stack depth, clipped to 8; NULL = 0). */
int crl_encode(crl_engine* e, const uint64_t* boards_dev, const uint64_t* hist_dev, const uint8_t* hist_len_dev,
               int n, void* planes_bf16_dev);
/* uci_dict lookup (agentdistributed.py:31-32,80-82): label index of every move; -1 for CRL_MOVE_NONE */
int crl_policy_index(crl_engine* e, const uint16_t* moves_dev, const int32_t* counts_dev, int n,
                     int16_t* idx_dev);
/* copies the 64x64 (+ promotion) label table the kernels use: idx_host[promo*4096 + from*64 + to], promo 0..4
 * (e may be NULL: the table is then produced without touching a device) */
int crl_label_table_host(crl_engine* e, int16_t* idx_host);

/* ---- network: model.ChessModel forward (model.py:31-63, 74-75, 111-122) ---------------------------- */
/* weights_host: CRL_N_WEIGHT_TENSORS fp32 tensors in the order documented in DESIGN.md ("weight pack"),
 * Keras layouts (conv HWIO, dense [in][out]); BatchNorm is folded on upload. */
int crl_net_load_host(crl_engine* e, const float* const* weights_host, const int64_t* sizes, int n_tensors);
/* planes_bf16_dev [n][8][8][128] -> policy_dev [n][1968] (softmax), value_dev [n] (tanh) */
int crl_net_forward(crl_engine* e, const void* planes_bf16_dev, int n, float* policy_dev, float* value_dev);
/* test hook: run convolution `layer` (0 = stem, 1..20 = residual tower) alone: in_dev [n][8][8][cin] bf16,
 * optional residual_dev / out_dev [n][8][8][256] bf16 */
int crl_debug_conv(crl_engine* e, int layer, const void* in_dev, int cin, int n, const void* residual_dev,
                   void* out_dev, int relu);
/* test hook: the PRODUCTION forward pass (the whole-tower kernel k_trunk4, the policy GEMM, the softmax / value kernel)
 * on planes_bf16_dev [n][8][8][128], with taps for parity tests against model.py:31-63, 111-122 layer by layer:
 *   act_out_dev    [n][8][8][256] bf16  output of convolution `layer` (0 = stem, 1..20 = tower; after BatchNorm, skip
 *                                       connection and ReLU where the graph has them), written by k_trunk4's own epilogue
 *   logits_out_dev [n][1968] f32        policy logits before the softmax
 *   pf_out_dev     [n][128] bf16, vf_out_dev [n][64] f32   inputs of the two dense heads (1x1 conv + BN + ReLU, flattened)
 *   policy_dev [n][1968], value_dev [n] as crl_net_forward.  Any tap may be NULL. */
int crl_debug_tower(crl_engine* e, const void* planes_bf16_dev, int n, int layer, void* act_out_dev, float* logits_out_dev,
                    void* pf_out_dev, float* vf_out_dev, float* policy_dev, float* value_dev);
/* test hook: crl_net_forward with the row count of a search batch -- the kernels are launched for n_bound rows of
 * planes_bf16_dev and read the count *n_dev (device int32) themselves; only rows below min(n_bound, *n_dev) are
 * evaluated and only those rows of policy_dev [n_bound][1968] / value_dev [n_bound] are written */
int crl_debug_forward_counted(crl_engine* e, const void* planes_bf16_dev, int n_bound, const int32_t* n_dev,
                              float* policy_dev, float* value_dev);
/* Opt-in fp8 evaluation.  The 21 tower convolutions run on e4m3 operands (tcgen05 kind::f8f6f4, fp32 accumulation):
 * planes exactly, weights per output channel scaled to max |W| = 448, each layer's output (but the last, which feeds
 * the bf16 heads) as e4m3 x a power-of-two scale max(2^ceil(log2(amax / 448)), 2^-126) from calibration (1 for
 * amax 0; the floor keeps 1 / scale finite).  Heads, softmax and search are unchanged.  Not bit-exact with bf16; DESIGN.md section 3.1 states the definition and the measured deviation.
 *   crl_net_calibrate_host : runs the bf16 tower on planes_bf16_dev [n][8][8][128] and writes max |output| of each
 *                            convolution to amax_host [21]
 *   crl_net_load_fp8_host  : crl_net_load_host, then the fp8 tower from the same pack and act_amax_host [21] (finite,
 *                            >= 0, else CRL_EINVAL); selects fp8.  On any error the engine is left in bf16.
 *   crl_net_set_precision  : CRL_NET_BF16 or CRL_NET_FP8 (CRL_ESTATE without an fp8 load).  crl_net_load_host returns
 *                            the engine to bf16 and drops the fp8 tower.
 * In fp8 mode crl_net_forward, crl_debug_tower and crl_debug_forward_counted take bf16 planes as before and convert
 * them. */
#define CRL_NET_BF16 0
#define CRL_NET_FP8 1
int crl_net_calibrate_host(crl_engine* e, const void* planes_bf16_dev, int n, float* amax_host);
int crl_net_load_fp8_host(crl_engine* e, const float* const* weights_host, const int64_t* sizes, int n_tensors,
                          const float* act_amax_host);
int crl_net_set_precision(crl_engine* e, int precision);
/* the deterministic test evaluator on raw boards (SoA), same outputs as the oracle's hash_evaluator */
int crl_hash_eval(crl_engine* e, const uint64_t* boards_dev, int n, uint64_t seed, int policy_bits,
                  float* policy_dev, float* value_dev);

/* ---- lockstep games + tree search: selfplay.play_game / mctree.SelfPlayTree ------------------------ */
int crl_set_evaluator(crl_engine* e, int kind, uint64_t seed, int policy_bits);
/* load n games (slots first..first+n-1): start records (AoS host) and the moves already played
 * (moves_host [n][stride], n_moves_host [n]); moves are replayed on the device so history planes and
 * repetition keys exist.  Replaces Game(...) + Game.move replay (dataset.py:50-58). */
int crl_games_set_host(crl_engine* e, int first, int n, const uint64_t* start_host, const uint16_t* moves_host,
                       const int32_t* n_moves_host, int stride);
/* per game: current record (AoS), plies played, Game.get_result (CRL_RESULT_NONE = running). NULLs allowed */
int crl_games_get_host(crl_engine* e, int first, int n, uint64_t* boards_host, int32_t* plies_host,
                       int8_t* results_host);
/* lanes first..first+n-1: active_host[i] == 0 parks the lane (no search, no moves; its record stays readable),
 * != 0 resumes it.  crl_games_set_host activates the lanes it loads.  Used by the lockstep driver when no game is
 * left to start in a lane (per-GPU slot refill, the many-games form of selfplay.py:142-162's game loop). */
int crl_games_set_active_host(crl_engine* e, int first, int n, const uint8_t* active_host);
/* the moves of one game so far (DatasetGame / Game.get_history 'moves') */
int crl_game_moves_host(crl_engine* e, int game, uint16_t* moves_host, int cap, int32_t* n_host);
/* the batched forms of the calls above, one device round trip for many lanes (the lockstep driver's harvest / refill):
 *   crl_games_restart_host : Game() in every listed lane (scattered lanes, all from the record start_host [9]) -- the
 *                            `for game in range(games)` loop of selfplay.py:142-162 refilling a lane as its game ends
 *   crl_games_moves_host   : Game.get_history()['moves'] (game.py:59-66) of the listed lanes: moves_host [n][cap],
 *                            n_moves_host [n] (the true length, even where it exceeds cap)
 *   crl_games_play_host    : Game.move (game.py:28-41) of one optional move per lane (moves_host [n_games], 0xFFFF =
 *                            none); accepted_host [n_games] (may be NULL) = whether it was legal and played
 *   crl_games_legal_host   : Game.get_legal_moves (game.py:43-57) of lanes first..first+n-1: legal_host [n][256],
 *                            n_legal_host [n] */
int crl_games_restart_host(crl_engine* e, const int32_t* lanes_host, int n, const uint64_t* start_host);
int crl_games_moves_host(crl_engine* e, const int32_t* lanes_host, int n, uint16_t* moves_host, int cap,
                         int32_t* n_moves_host);
int crl_games_play_host(crl_engine* e, const uint16_t* moves_host, uint8_t* accepted_host);
int crl_games_legal_host(crl_engine* e, int first, int n, uint16_t* legal_host, int32_t* n_legal_host);
/* AgentDistributed.best_move(real_game=True) (agentdistributed.py:56-58): policy argmax over legal moves for
 * every game with mask_host[g] != 0 (NULL = all running games); writes picks_host [n_games] and plays them. */
int crl_games_policy_move_host(crl_engine* e, const uint8_t* mask_host, uint16_t* picks_host);
/* Fixed-depth alpha-beta (DESIGN.md 3.6) on the current position of every lane with mask_host[i] != 0 that is
   active and unfinished: its move (MOVE_NONE for every other lane), its score in centipawns for the side to move
   and the positions the search visited.  Plays nothing and leaves every other engine state unchanged.
   CRL_EINVAL for depth / qdepth out of range (1..5 / 0..8).  mask_host NULL = all lanes; move_host [n_games],
   score_host [n_games] and nodes_host [n_games] may each be NULL. */
int crl_games_ab_move_host(crl_engine* e, const uint8_t* mask_host, int depth, int qdepth,
                           uint16_t* move_host, int32_t* score_host, int64_t* nodes_host);
/* crl_games_ab_move_host with a seeded near-best root pick (DESIGN.md 3.7), for generating varied training games: a
   lane at ply < pick_plies whose best score is not a mate plays one of the root moves scored within `margin`
   centipawns of the best, chosen by splitmix64(salt_host[lane] + ply); otherwise the first best move, as
   crl_games_ab_move_host.  score_host is the picked move's score; nodes_host is unchanged.  margin 0 gives
   crl_games_ab_move_host's answer.  salt_host [n_games] is required.  CRL_EINVAL for the depth / qdepth limits above
   and for margin < 0 or pick_plies < 0.  Plays nothing and leaves every other engine state unchanged. */
int crl_games_ab_pick_host(crl_engine* e, const uint8_t* mask_host, int depth, int qdepth, int margin, int pick_plies,
                           const uint64_t* salt_host, uint16_t* move_host, int32_t* score_host, int64_t* nodes_host);
/* The alpha-beta search of crl_games_ab_move_host / crl_games_ab_pick_host with options in `flags`:
 *   CRL_AB_REPETITIONS  a position at least one ply below the root that repeats an earlier position of its reversible
 *                       run -- on the search path, the root included, or in the lane's game before the root, back to the
 *                       last irreversible move -- scores 0 (python-chess's board.is_repetition(2) on the game's moves
 *                       followed by the path; DESIGN.md 3.6).  It counts as one visited position and generates no
 *                       moves.  The root itself is never scored by the rule.
 * salt_host NULL: the first best move, and margin and pick_plies must be 0.  Otherwise the seeded near-best pick of
 * crl_games_ab_pick_host.  With flags 0 the outputs equal those two calls'.  CRL_EINVAL for unknown flag bits, the
 * depth / qdepth limits, margin < 0 or pick_plies < 0, and a margin or pick_plies without a salt.  Plays nothing and
 * leaves every other engine state unchanged. */
#define CRL_AB_REPETITIONS 1
int crl_games_ab_search_host(crl_engine* e, const uint8_t* mask_host, int depth, int qdepth, int flags,
                             int margin, int pick_plies, const uint64_t* salt_host,
                             uint16_t* move_host, int32_t* score_host, int64_t* nodes_host);
/* Two networks in one engine: a match between them in one lockstep batch (chessrl_b200/arena.py, DESIGN.md 3.5).
 *   crl_net_select_slot       : the network slot (0 or 1, else CRL_EINVAL) that crl_net_load_host,
 *                               crl_net_load_fp8_host, crl_net_calibrate_host, crl_net_set_precision, crl_set_evaluator,
 *                               crl_net_forward, crl_debug_tower, crl_debug_forward_counted and crl_debug_conv act on.
 *                               Each slot has its own weights, precision and evaluator (kind, seed, policy bits).  The
 *                               slot is 0 after crl_create; slot 1 allocates nothing until a load or crl_set_evaluator
 *                               configures it, and configuring one slot leaves the other's outputs bit-identical.
 *   crl_games_set_players_host: for lanes first..first+n-1, the slot that plays white (white_slot_host [n]) and the one
 *                               that plays black (black_slot_host [n]); 0 and 0 after crl_create.  They persist through
 *                               crl_games_set_host / crl_games_restart_host.  A lane whose players change loses its
 *                               evaluation-reuse twin, and a search must begin again (crl_mcts_begin_move).
 * A search (crl_mcts_begin_move, crl_mcts_simulate, K = 1 and wave mode) and crl_games_policy_move_host evaluate every
 * row of a lane with the slot of the side to move at the lane's root: the root, the opponent replies it predicts and
 * its leaves.  While no lane names slot 1 the search runs exactly as with one network.  CRL_ESTATE when a lane names
 * slot 1 but slot 1 has no evaluator, or when the two slots hold evaluators of different kinds (hash and network). */
#define CRL_NET_SLOTS 2
int crl_net_select_slot(crl_engine* e, int slot);
int crl_games_set_players_host(crl_engine* e, int first, int n, const uint8_t* white_slot_host,
                               const uint8_t* black_slot_host);
/* Tree(root) (mctree.py:104-111): a fresh tree per running game rooted at its current position,
 * root.visits = 1, root evaluated once for its children's priors. */
int crl_mcts_begin_move(crl_engine* e);
/* Evaluation reuse across consecutive move searches of a game (off by default).  The reference builds a new tree for
 * every move (agentdistributed.py:61-63) and therefore asks the network again about positions its previous search
 * already evaluated: once the game has played (our move, reply) of root child c (selfplay.py:77-78), the new root IS c
 * and everything below c in the old tree is the same position reached by the same plies -- same history planes
 * (netencoder.py:47-69), same network input, same output.  With reuse on, the engine keeps the previous tree (a second
 * set of node / prior / child pools that swaps roles at every crl_mcts_begin_move) and an expansion whose node has a
 * TWIN there takes the opponent's reply, the value and the children's priors from it instead of running the two
 * evaluations.  The new tree itself is built from scratch exactly as before -- statistics start at zero, the schedule
 * is the reference's -- so visit counts, value sums and the games played are bit-identical with reuse on and off.
 * Twins are linked when crl_mcts_commit_host(apply = 1) plays a root child's two plies; any other change of a game
 * (set / restart / play / policy move) unlinks it.  Exact schedule (inflight = 1) only; waves evaluate everything.
 * crl_reuse_count_host: evaluations taken from the previous tree so far (crl_counters_host counts only those run). */
int crl_set_reuse(crl_engine* e, int enable);
/* A promise by the host that at most max_running_games games are running (active and unfinished) until it says otherwise
 * (0 = no promise).  The evaluation batches are compacted on the device, so the engine otherwise sizes every launch for all
 * max_games lanes; with a bound the launches shrink, and a batch bound of at most 296 positions runs the tower's single-tile
 * instantiation (one 4-board tile per CTA pair: ~1.2 x faster evaluations) -- the drain of a finite selfplay.py run
 * (selfplay.py:142-163), when few of the lanes still hold a game.  A broken promise is detected on the device and
 * reported as CRL_ENOMEM by the next call that checks the pools; nothing is evaluated silently wrong. */
int crl_mcts_set_row_bound(crl_engine* e, int max_running_games);
int crl_reuse_count_host(crl_engine* e, int64_t* reused_host);
/* n_sims x SelfPlayTree.explore_tree (mctree.py:200-214) for every running game in lockstep.
 * inflight = 1: the deterministic threads=1 schedule.
 * inflight = K > 1 (<= max_inflight): WAVES of up to K simulations per game = one legal schedule of the reference's
 * ThreadPoolExecutor(max_workers=K) (mctree.py:173-176): the wave's selects run one after the other (each adds its
 * virtual loss to its leaf, mctree.py:226-227), then its evaluations as one batch, then its backprops in the same
 * order (mctree.py:278-296, virtual loss removed).  A select that would enter a node created earlier in the same
 * wave (whose opponent reply is still being evaluated) is deferred to the next wave.  Deterministic; every game
 * runs exactly n_sims simulations. */
int crl_mcts_simulate(crl_engine* e, int n_sims, int inflight);
/* root children in creation order (mctree.py:305-322 needs visits): arrays [n_games][CRL_MAX_MOVES] except
 * n_children/root_visits/root_ply [n_games]; any may be NULL */
int crl_mcts_root_stats_host(crl_engine* e, int32_t* child_visits, double* child_values, float* child_priors,
                             uint16_t* child_moves, uint16_t* child_replies, int8_t* child_results,
                             int32_t* n_children, int32_t* root_visits, double* root_values);
/* search_move's return value (mctree.py:178-198) for pick_host[g] = index of the chosen root child
 * (-1 = skip the game): out_moves_host [n_games][2] = (move_stack[-2], move_stack[-1]) of that child, then
 * plays both through Game.move like selfplay.py:77-78 when `apply` != 0. */
int crl_mcts_commit_host(crl_engine* e, const int32_t* pick_host, uint16_t* out_moves_host, int apply);
/* flat dump of one game's tree for Node views / parity tests; arrays sized by `cap` nodes */
typedef struct {
  int32_t parent;      /* -1 for the root */
  int32_t slot;        /* index among the parent's children (creation order) */
  int32_t visits;
  int32_t n_legal;     /* legal moves of the node's state */
  int32_t n_children;  /* expanded so far */
  int32_t result;      /* Game.get_result of the node's state, CRL_RESULT_NONE if not over */
  uint16_t move;       /* our move leading here, 0xFFFF for the root */
  uint16_t reply;      /* opponent reply, 0xFFFF if the game ended on our move */
  float prior;
  double value;        /* sum of backed-up values */
  uint64_t board[9];   /* the node's state */
} crl_node_host;
int crl_mcts_node_dump_host(crl_engine* e, int game, crl_node_host* out, int cap, int32_t* n_host);
/* counters since crl_create: [0] simulations, [1] net/hash evaluations requested, [2] kernels launched */
int crl_counters_host(crl_engine* e, int64_t* out3);
/* optional per-kernel-class timing (CUDA events on the engine stream); see DESIGN.md */
int crl_profile(crl_engine* e, int enable);
int crl_profile_read_host(crl_engine* e, double* ms_by_class, int64_t* launches_by_class, int n_classes);

/* ---- training targets from the alpha-beta search (DESIGN.md 3.8) ------------------------------------ */
/* root-child scores of the last crl_games_ab_* call: [n_games][CRL_MAX_MOVES], counts -1 = lane not searched */
int crl_games_ab_root_scores_host(crl_engine* e, int32_t* scores_host, int32_t* counts_host);
/* soft policy [n][CRL_N_LABELS] and score value [n] from the root scores of rows offsets[i]..offsets[i+1] */
int crl_search_targets(crl_engine* e, const uint64_t* boards_dev, const int32_t* scores_dev, const int32_t* offsets_dev,
                       int n, float temperature, float* policy_dev, float* score_value_dev, int32_t* legal_count_dev);

#ifdef __cplusplus
}
#endif
#endif
