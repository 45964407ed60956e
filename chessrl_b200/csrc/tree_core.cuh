// tree_core.cuh -- per-game logic of the lockstep PUCT search and of the game records, over flat
// structure-of-arrays pools in HBM.
//
// Replaces (reference file:line):  mctree.Node fields + get_value/get_best_child (mctree.py:15-95),
// SelfPlayTree.select/expand/simulate/backprop/_update_prior (mctree.py:216-303), the policy-argmax reply
// of AgentDistributed.best_move(real_game=True) (agentdistributed.py:56-58) and the history walk of
// netencoder._get_game_history (netencoder.py:47-69).
//
// Layout decisions (see DESIGN.md "data layout"):
//   * a NODE is the state after (our move, opponent reply) -- exactly one mctree.Node.  It stores both
//     positions (P1 after our move, P2 after the reply) because history planes and repetition keys of
//     descendants need every ply on the path.
//   * node STATISTICS live on the parent's edge slots (visits / value / prior / child / result, one SoA
//     slot per legal move, children in creation order), so the PUCT scan of a node reads contiguous
//     arrays instead of chasing child pointers.  sum(child.visits for child in node.children), which
//     get_value needs, equals visits-1 for an expanded non-terminal child and 0 otherwise (SURVEY.md a8).
//   * priors are attached at child creation from the parent's cached legal-move policy; the reference
//     writes them when the parent becomes fully expanded and never reads them earlier (mctree.py:254-255),
//     so the results are identical and the third network evaluation per simulation disappears.
// Every function is CRL_HD: the device kernels in tree_kernels.cu call them one game per thread (or per
// warp for the child scan); the TEST-ONLY host harness calls the same code serially.
#pragma once
#include "chess_core.cuh"

namespace crl {

enum { HIST_RING = 8, KEY_RING = 128, MAX_GAME_PLIES = 2048 };
enum { KIND_IDLE = 0, KIND_TERMINAL = 1, KIND_NEED_REPLY = 2, KIND_NEW_TERMINAL = 3, KIND_EVAL_LEAF = 4,
       KIND_EVAL_REUSED = 5 };   // new leaf whose value / priors came from its twin in the previous move's tree
enum { ERR_NODE_OVERFLOW = 1, ERR_EDGE_OVERFLOW = 2, ERR_PLY_OVERFLOW = 4, ERR_ROW_OVERFLOW = 8 };

struct NodeRec {
  u64 p2[9];      // state of the node (after the reply; = p1 when the game ended on our move)
  u64 p1[9];      // state after our move
  u64 key1, key2; // Board._transposition_key hashes of p1 / p2
  int parent;     // node index inside the game, -1 for the root
  int edge0;      // first edge slot of this node inside the game's edge arena
  u16 n_legal;    // legal moves of p2
  u16 n_exp;      // children created so far
  u16 move;       // our move (MOVE_NONE for the root)
  u16 reply;      // opponent reply (MOVE_NONE if none)
  int8_t result;  // Game.get_result of p2, RESULT_NONE while running
  u8 slot;        // index among the parent's children (creation order)
  u8 has_p1;      // 0 for the root
  u8 pending;     // wave mode: created in the current wave, its reply (network evaluation of p1) is not known yet
  // --- evaluation reuse across consecutive searches of one game (see "evaluation reuse" below) ---
  int prev;       // node of the PREVIOUS move's tree that is this same node (same game, same path), -1 if none
  float v;        // network value of p2 (valid when evald)
  u8 evald;       // 1 once the node has been evaluated: reply, n_legal, v and its children's priors are final
};

static constexpr int SLOT_N_STRIDE = 4;   // distance between the row counters of slot 0 and slot 1

struct Pools {
  int G, NN, EA;
  // --- games ---
  u64* g_cur;       // [9][G]
  u64* g_hist;      // [HIST_RING][8][G]   bitboards of the position at ply q live in slot q % 8
  u64* g_keys;      // [KEY_RING][G]       transposition key of the position at ply q in slot q % 128
  u16* g_moves;     // [G][MAX_GAME_PLIES]
  int* g_nmoves;    // [G]
  int8_t* g_result; // [G]
  u8* g_active;     // [G]
  // --- trees ---
  NodeRec* nodes;   // [G][NN]
  int* g_nnodes;    // [G]
  int* g_nedges;    // [G]
  u16* e_move;      // [G][EA]
  float* e_prior;
  int* e_visits;
  double* e_value;
  int* e_child;
  int8_t* e_result;
  u8* e_vloss;      // [G][EA] Node.vloss of the child on this edge (mctree.py:36, 226-227, 292-293); 0 outside a wave
  int* r_visits;    // [G]
  double* r_value;  // [G]
  // --- evaluation reuse: the tree of the previous move search (the pools swap roles at every crl_mcts_begin_move) ---
  int reuse;            // 1: expansions look their twin up in the previous tree (exact schedule, K = 1, only)
  NodeRec* nodes_prev;  // [G][NN]
  float* e_prior_prev;  // [G][EA]
  int* e_child_prev;    // [G][EA]
  int* g_prev_root;     // [G] node of the previous tree whose state is the game's current position, -1 = none
  // --- per-simulation scratch: one SLOT per in-flight simulation, slot = g*K + j (K = 1: slot = game) ---
  int K;            // in-flight simulations per game of the kernels being launched (1 = the exact threads=1 schedule)
  int* s_node;      // [G*K] selected node / new child
  int* s_kind;      // [G*K]
  u16* s_moves;     // [G*K][MAX_MOVES] legal moves of the position awaiting its reply
  int* s_nmoves;    // [G*K]
  int* s_row;       // [G*K] row of this slot in the current evaluation batch
  int* s_path;      // [G][32] exact schedule: edge (index inside the game's arena) taken at every level of the select
  int* s_depth;     // [G] levels recorded in s_path, -1 = deeper than path_cap (the backup then chases parent pointers)
  int path_cap;     // 32; CRL_PATH_CAP=n (0..32) lowers it so that tests exercise both backup forms in one search
  int* s_wave_n;    // [G] slots used by the current wave
  int* g_sims_left; // [G] simulations of the current crl_mcts_simulate call still to run (wave mode)
  int* eval_list;   // [G*K] slot of every batch row
  int* eval_n;      // [1]
  int row_cap;      // rows the evaluation kernels of this launch sequence cover (G*K, or the host's bound: crl_mcts_set_row_bound)
  // --- two networks (crl_games_set_players_host, DESIGN.md 3.5): a lane's rows go to the batch of the slot that moves at
  // its root; slot k's rows are rows k * slot_stride + r of the list, policy, value and statistics buffers, and its row
  // count is eval_n[SLOT_N_STRIDE * k] (likewise for batch B's counter)
  int n_slots;          // 1: every row belongs to slot 0 (g_players / g_slot are not read)
  int slot_stride;
  const u8* g_players;  // [2][G] slot playing white / black
  u8* g_slot;           // [G] slot searching at the lane's root (set by k_root_init)
  int* err;         // [1] ERR_* flags
  long long* counters;  // [0] simulations [1] evaluations run [2] evaluations taken from the previous tree instead
};

// The evaluator's policy output as the search kernels read it.  stats == null: base[row][label] IS the probability
// (hash evaluator, crl_net_forward).  stats != null (network inside the search): base holds the policy LOGITS and
// stats[row] = (max logit, 1 / sum exp) -- the softmax kernel then writes 8 bytes per row instead of the 7.9 KB
// probability row of which the search reads ~35 entries; expf(x - max) * inv is the very expression k_softmax_value
// evaluates for a full row, so both views give the same bits.
struct PolicyView {
  const float* base;
  int ld;
  const float* stats;
};
CRL_HD float policy_at(const PolicyView& pv, int row, int label) {
  const float x = pv.base[(long long)row * pv.ld + label];
  if (!pv.stats) return x;
#if defined(__CUDA_ARCH__)
  return expf(x - pv.stats[2 * row]) * pv.stats[2 * row + 1];
#else
  return __builtin_expf(x - pv.stats[2 * row]) * pv.stats[2 * row + 1];
#endif
}

CRL_HD Board load_soa(const u64* base, long long stride, long long i) {
  Board b;
#pragma unroll
  for (int k = 0; k < 8; ++k) b.bb[k] = base[k * stride + i];
  b.meta = base[8 * stride + i];
  return b;
}
CRL_HD void store_soa(u64* base, long long stride, long long i, const Board& b) {
#pragma unroll
  for (int k = 0; k < 8; ++k) base[k * stride + i] = b.bb[k];
  base[8 * stride + i] = b.meta;
}
CRL_HD Board load_rec(const u64* r) {
  Board b;
#pragma unroll
  for (int k = 0; k < 8; ++k) b.bb[k] = r[k];
  b.meta = r[8];
  return b;
}
CRL_HD void store_rec(u64* r, const Board& b) {
#pragma unroll
  for (int k = 0; k < 8; ++k) r[k] = b.bb[k];
  r[8] = b.meta;
}

// ---------------------------------------------------------------------------------------------------
// history walks.  Positions before (node, which) in reverse play order: P1(node) [if which==2],
// P2(parent), P1(parent), ..., P2(root) = current game position, then the game's own ring.
// ---------------------------------------------------------------------------------------------------
struct Cursor {
  int node;    // >= 0: tree position; -1: inside the game ring
  int which;   // 1 or 2 for tree positions
  int ply;     // ply of the position the cursor points at
};

// step to the previous position; returns false when the move stack is exhausted
CRL_HD bool cursor_prev(const Pools& P, int g, Cursor& c) {
  if (c.ply <= 0) return false;
  if (c.node > 0) {
    const NodeRec& n = P.nodes[(long long)g * P.NN + c.node];
    if (c.which == 2 && n.reply != MOVE_NONE) {
      c.which = 1;
    } else {
      c.node = n.parent;   // parent's P2 (for the root: the current game position)
      c.which = 2;
    }
  } else {
    c.node = -1;           // from the root (node 0) or deeper in the ring
  }
  c.ply -= 1;
  return true;
}
CRL_HD void cursor_bitboards(const Pools& P, int g, const Cursor& c, u64* out8) {
  if (c.node >= 0) {
    const NodeRec& n = P.nodes[(long long)g * P.NN + c.node];
    const u64* r = (c.which == 2) ? n.p2 : n.p1;
#pragma unroll
    for (int k = 0; k < 8; ++k) out8[k] = r[k];
  } else {
    const u64* h = P.g_hist + (long long)(c.ply % HIST_RING) * 8 * P.G + g;
#pragma unroll
    for (int k = 0; k < 8; ++k) out8[k] = h[(long long)k * P.G];
  }
}
CRL_HD u64 cursor_key(const Pools& P, int g, const Cursor& c) {
  if (c.node >= 0) {
    const NodeRec& n = P.nodes[(long long)g * P.NN + c.node];
    return c.which == 2 ? n.key2 : n.key1;
  }
  return P.g_keys[(long long)(c.ply % KEY_RING) * P.G + g];
}

// earlier occurrences of `key` inside the reversible run that ends at the cursor position
// (Board.is_fivefold_repetition walks the stack back until an irreversible move)
CRL_HD int count_repetitions(const Pools& P, int g, Cursor c, u64 key, int revlen) {
  int reps = 0;
  if (revlen > KEY_RING - 1) revlen = KEY_RING - 1;
  for (int i = 0; i < revlen; ++i) {
    if (!cursor_prev(P, g, c)) break;
    if (cursor_key(P, g, c) == key) ++reps;
  }
  return reps;
}

// ---------------------------------------------------------------------------------------------------
// PUCT score of one edge: Node.get_value (mctree.py:71-87), float64 with the one float32 product
// ---------------------------------------------------------------------------------------------------
CRL_HD double edge_score(int visits, double value, float prior, int child_result, int vloss = 0) {
  double n1 = (double)(1 + visits);
  int sub = (child_result != RESULT_NONE || visits < 2) ? 0 : visits - 1;
  float cp = 10.0f * prior;                      // int * np.float32 -> float32
#if defined(__CUDA_ARCH__)
  double q = __ddiv_rn(value, n1);
  double u = __dmul_rn((double)cp, __ddiv_rn(__dsqrt_rn((double)sub), n1));
  return __dsub_rn(__dadd_rn(q, u), (double)vloss);   // "return value - self.vloss" (mctree.py:87)
#else
  volatile double q = value / n1;
  volatile double s = __builtin_sqrt((double)sub);
  volatile double r = s / n1;
  volatile double u = (double)cp * r;
  volatile double qu = q + u;
  return qu - (double)vloss;
#endif
}

// serial child scan (first maximum).  The device kernel uses a warp-cooperative version of this loop.
CRL_HD int best_edge_serial(const Pools& P, int g, const NodeRec& n, bool with_vloss = false) {
  long long base = (long long)g * P.EA + n.edge0;
  int best = 0;
  double best_s = 0;
  for (int k = 0; k < n.n_exp; ++k) {
    double s = edge_score(P.e_visits[base + k], P.e_value[base + k], P.e_prior[base + k], P.e_result[base + k],
                          with_vloss ? (int)P.e_vloss[base + k] : 0);
    if (k == 0 || s > best_s) {
      best_s = s;
      best = k;
    }
  }
  return best;
}

// SelfPlayTree.select without the expansion (mctree.py:216-229): returns the node to expand, or a terminal
// leaf.  `scan` abstracts the child scan so the warp kernel can plug in its cooperative version.
template <class Scan>
CRL_HD void select_descend(const Pools& P, int g, Scan scan, int* out_node, int* out_terminal) {
  int node = 0;
  for (;;) {
    const NodeRec& n = P.nodes[(long long)g * P.NN + node];
    if (n.result != RESULT_NONE) {
      *out_node = node;
      *out_terminal = 1;
      return;
    }
    if (n.n_exp < n.n_legal) {
      *out_node = node;
      *out_terminal = 0;
      return;
    }
    int k = scan(n);
    node = P.e_child[(long long)g * P.EA + n.edge0 + k];
  }
}

// Wave mode (K > 1 in-flight simulations per game = one legal schedule of the reference's threads=K pool: the K
// selects run one after the other, then the K simulates, then the K backprops in the same order).  A select of the
// wave may not enter a node created earlier in the SAME wave whose opponent reply is still unknown (it needs the
// network evaluation of this wave): the wave is cut there and the simulation runs in the next wave -- which is the
// schedule "fewer than K workers were active", equally legal for the reference.
// returns 0 = expand *out_node, 1 = *out_node is a terminal leaf, 2 = cut (pending node reached)
template <class Scan>
CRL_HD int select_descend_wave(const Pools& P, int g, Scan scan, int* out_node) {
  int node = 0;
  for (;;) {
    const NodeRec& n = P.nodes[(long long)g * P.NN + node];
    if (n.pending) return 2;
    *out_node = node;
    if (n.result != RESULT_NONE) return 1;
    if (n.n_exp < n.n_legal) return 0;
    int k = scan(n);
    node = P.e_child[(long long)g * P.EA + n.edge0 + k];
  }
}

// leaf.vloss += d (mctree.py:226-227 / 292-293); the root's vloss is never read (its score is never compared)
CRL_HD void vloss_add(const Pools& P, int g, int node, int d) {
  if (node <= 0) return;
  const NodeRec& n = P.nodes[(long long)g * P.NN + node];
  const NodeRec& pn = P.nodes[(long long)g * P.NN + n.parent];
  long long e = (long long)g * P.EA + pn.edge0 + n.slot;
  P.e_vloss[e] = (u8)((int)P.e_vloss[e] + d);
}

// ---------------------------------------------------------------------------------------------------
// evaluation reuse.  The reference builds a fresh tree for every move (agentdistributed.py:61-63), so the network
// is asked again about positions the previous search already evaluated: after the game has played (our move,
// reply) of root child c, the new root IS c, and every node below c in the old tree is the same position reached
// by the same plies -- same history planes, same network input, same output.  The new search still builds its
// tree from scratch (all statistics start at zero, the selection order is the reference's); only the two network
// evaluations of an expansion are looked up instead of run when the old tree holds the node's TWIN.  Twins are
// found without hashing: children are created in a fixed order (last legal move first), so the child the new
// node creates at slot k is the twin of the child at slot k of the parent's twin.  Results are bit-identical by
// construction (tests: reuse on / off plays the same games with the same root statistics).
// ---------------------------------------------------------------------------------------------------
CRL_HD int twin_of_child(const Pools& P, int g, const NodeRec& parent, int k) {
  if (!P.reuse || parent.prev < 0) return -1;
  const NodeRec& on = P.nodes_prev[(long long)g * P.NN + parent.prev];
  if (k >= on.n_exp) return -1;
  const int oc = P.e_child_prev[(long long)g * P.EA + on.edge0 + k];
  return P.nodes_prev[(long long)g * P.NN + oc].evald ? oc : -1;
}

// index of `mv` in a move list, -1 if absent
CRL_HD int find_move(const u16* moves, int n, u16 mv) {
  for (int i = 0; i < n; ++i)
    if (moves[i] == mv) return i;
  return -1;
}

// hand the twin's value and its children's priors to `node` (just built by reply_child); false if they do not fit
CRL_HD bool adopt_evaluation(const Pools& P, int g, int node, int twin) {
  NodeRec& n = P.nodes[(long long)g * P.NN + node];
  const NodeRec& t = P.nodes_prev[(long long)g * P.NN + twin];
  if (t.result != RESULT_NONE || t.n_legal != n.n_legal) return false;
  const long long dst = (long long)g * P.EA + n.edge0, src = (long long)g * P.EA + t.edge0;
  for (int i = 0; i < n.n_legal; ++i) P.e_prior[dst + i] = P.e_prior_prev[src + i];
  n.v = t.v;
  n.evald = 1;
  return true;
}

// generate the legal moves of `b`, its transposition key and Game.get_result, given where it sits
CRL_HD int analyse_position(const Pools& P, int g, const Board& b, Cursor at, u16* moves, int* n_moves, u64* key) {
  StoreSink sink{moves, 0};
  GenInfo gi = generate_legal(b, sink);
  *n_moves = sink.n;
  *key = position_key(b, gi.ep_legal);
  int reps = 0;
  int rev = meta_revlen(b.meta);
  if (rev >= 8 && sink.n > 0 && meta_halfmove(b.meta) < 100 && !insufficient_material(b))
    reps = count_repetitions(P, g, at, *key, rev);
  return game_result(b, sink.n, gi.in_check, reps);
}

// SelfPlayTree.expand, first half (mctree.py:241-244): pop the last unexpanded action of `parent`, play it,
// create the child.  Returns the kind of follow-up the child needs.
CRL_HD int expand_child(const Pools& P, int g, int slot, int parent, int* out_child) {
  NodeRec& pn = P.nodes[(long long)g * P.NN + parent];
  int child = P.g_nnodes[g];
  if (child >= P.NN) {
    *P.err |= ERR_NODE_OVERFLOW;
    *out_child = parent;
    return KIND_IDLE;
  }
  P.g_nnodes[g] = child + 1;
  int k = pn.n_exp;
  long long ebase = (long long)g * P.EA + pn.edge0;
  u16 mv = P.e_move[ebase + (pn.n_legal - 1 - k)];       // unexpanded_actions.pop(): last legal move first
  NodeRec& cn = P.nodes[(long long)g * P.NN + child];
  Board b = load_rec(pn.p2);
  make_move(b, mv);
  store_rec(cn.p1, b);
  cn.parent = parent;
  cn.slot = (u8)k;
  cn.has_p1 = 1;
  cn.move = mv;
  cn.reply = MOVE_NONE;
  cn.n_exp = 0;
  cn.n_legal = 0;
  cn.edge0 = 0;
  cn.pending = 0;
  cn.prev = twin_of_child(P, g, pn, k);
  cn.v = 0.f;
  cn.evald = 0;
  P.e_child[ebase + k] = child;
  P.e_visits[ebase + k] = 0;
  P.e_value[ebase + k] = 0.0;
  P.e_vloss[ebase + k] = 0;
  // e_prior[k] already holds this child's prior: store_priors() wrote the parent's legal-order policy
  // mirrored (legal move j -> slot n_legal-1-j), which is zip(priors, reversed(children)) (mctree.py:298-303).
  pn.n_exp = (u16)(k + 1);

  Cursor at{child, 1, meta_ply(b.meta)};
  u16* moves = P.s_moves + (long long)slot * MAX_MOVES;
  int n_moves;
  u64 key;
  int res = analyse_position(P, g, b, at, moves, &n_moves, &key);
  cn.key1 = key;
  P.s_nmoves[slot] = n_moves;
  *out_child = child;
  if (res != RESULT_NONE) {        // the game ended on our move: the child's state is P1 (mctree.py:244)
    store_rec(cn.p2, b);
    cn.key2 = key;
    cn.result = (int8_t)res;
    cn.n_legal = (u16)n_moves;
    P.e_result[ebase + k] = (int8_t)res;
    return KIND_NEW_TERMINAL;
  }
  cn.result = RESULT_NONE;
  cn.pending = 1;                  // until reply_child; only wave-mode selects can meet it
  P.e_result[ebase + k] = RESULT_NONE;
  return KIND_NEED_REPLY;
}

// first maximum of the legal-masked policy (agentdistributed.py:56-58, 80-82)
// `row(label)` = probability of a label in the evaluated row
template <class Row>
CRL_HD int argmax_legal_of(Row row, const int16_t* label_of, const u16* moves, int n) {
  int best = 0;
  float best_p = 0.f;
  for (int i = 0; i < n; ++i) {
    u16 m = moves[i];
    float p = row((int)label_of[(int)mv_promo(m) * 4096 + mv_from(m) * 64 + mv_to(m)]);
    if (i == 0 || p > best_p) {
      best_p = p;
      best = i;
    }
  }
  return best;
}
struct PlainRow {
  const float* p;
  CRL_HD float operator()(int label) const { return p[label]; }
};
CRL_HD int argmax_legal(const float* policy_row, const int16_t* label_of, const u16* moves, int n) {
  return argmax_legal_of(PlainRow{policy_row}, label_of, moves, n);
}

// SelfPlayTree.expand, second half (mctree.py:245-249): the opponent answers with its policy argmax, the
// child's state becomes P2, Node(new_state) lists its legal moves.
CRL_HD int reply_child(const Pools& P, int g, int slot, int child, const float* policy_row, const int16_t* label_of,
                       int pick = -1) {
  NodeRec& cn = P.nodes[(long long)g * P.NN + child];
  const u16* moves1 = P.s_moves + (long long)slot * MAX_MOVES;
  if (pick < 0) pick = argmax_legal(policy_row, label_of, moves1, P.s_nmoves[slot]);
  u16 reply = moves1[pick];
  Board b = load_rec(cn.p1);
  make_move(b, reply);
  store_rec(cn.p2, b);
  cn.reply = reply;

  Cursor at{child, 2, meta_ply(b.meta)};
  u16 moves2[MAX_MOVES];
  int n2;
  u64 key;
  int res = analyse_position(P, g, b, at, moves2, &n2, &key);
  cn.key2 = key;
  cn.result = (int8_t)res;
  cn.n_legal = (u16)n2;
  cn.pending = 0;
  const NodeRec& pn = P.nodes[(long long)g * P.NN + cn.parent];
  P.e_result[(long long)g * P.EA + pn.edge0 + cn.slot] = (int8_t)res;
  if (res != RESULT_NONE) return KIND_NEW_TERMINAL;
  // reserve the node's edge slots and remember its legal moves (Node.unexpanded_actions, mctree.py:31).
  // In wave mode several rows of one game run concurrently, hence the atomic; where a node's edges sit inside
  // the game's arena has no influence on any result.
#if defined(__CUDA_ARCH__)
  int e0 = atomicAdd(&P.g_nedges[g], n2);
#else
  int e0 = P.g_nedges[g];
  P.g_nedges[g] = e0 + n2;
#endif
  if (e0 + n2 > P.EA) {
    *P.err |= ERR_EDGE_OVERFLOW;
    cn.n_legal = 0;
    cn.result = 0;   // poison as a drawn leaf so the search stays well-defined; the host raises on err
    P.e_result[(long long)g * P.EA + pn.edge0 + cn.slot] = 0;
    return KIND_NEW_TERMINAL;
  }
  cn.edge0 = e0;
  long long ebase = (long long)g * P.EA + e0;
  for (int i = 0; i < n2; ++i) P.e_move[ebase + i] = moves2[i];
  return KIND_EVAL_LEAF;
}

// wave mode, the serial part of one select (mctree.py:216-229): `what`/`node` come from select_descend_wave.
// Fills scratch slot `slot`, adds the leaf's virtual loss, returns the slot's kind.
CRL_HD int wave_take_slot(const Pools& P, int g, int slot, int what, int node) {
  if (what == 1) {
    P.s_node[slot] = node;
    P.s_kind[slot] = KIND_TERMINAL;
    vloss_add(P, g, node, 1);
    return KIND_TERMINAL;
  }
  int child;
  const int kind = expand_child(P, g, slot, node, &child);
  P.s_node[slot] = child;
  P.s_kind[slot] = kind;
  if (kind != KIND_IDLE) vloss_add(P, g, child, 1);
  return kind;
}

// cache the legal-order policy of an evaluated node on its edge slots (what _update_prior will hand out)
template <class Row>
CRL_HD void store_priors_of(const Pools& P, int g, int node, Row row, const int16_t* label_of) {
  const NodeRec& n = P.nodes[(long long)g * P.NN + node];
  long long ebase = (long long)g * P.EA + n.edge0;
  for (int i = 0; i < n.n_legal; ++i) {
    u16 m = P.e_move[ebase + i];
    // mirror index: legal move i is expanded as child (n_legal-1-i), whose prior slot is (n_legal-1-i)
    P.e_prior[ebase + (n.n_legal - 1 - i)] = row((int)label_of[(int)mv_promo(m) * 4096 + mv_from(m) * 64 + mv_to(m)]);
  }
}
CRL_HD void store_priors(const Pools& P, int g, int node, const float* policy_row, const int16_t* label_of) {
  store_priors_of(P, g, node, PlainRow{policy_row}, label_of);
}

// SelfPlayTree.backprop (mctree.py:278-296): visits += 1, value += v from the leaf to the root
CRL_HD void backup(const Pools& P, int g, int leaf, double v) {
  int node = leaf;
  while (node > 0) {
    const NodeRec& n = P.nodes[(long long)g * P.NN + node];
    const NodeRec& pn = P.nodes[(long long)g * P.NN + n.parent];
    long long e = (long long)g * P.EA + pn.edge0 + n.slot;
    P.e_visits[e] += 1;
    P.e_value[e] += v;
    node = n.parent;
  }
  P.r_visits[g] += 1;
  P.r_value[g] += v;
}

// ---------------------------------------------------------------------------------------------------
// game records
// ---------------------------------------------------------------------------------------------------
// refresh result / key of the current position of game g (after a reset or a move)
CRL_HD void game_refresh(const Pools& P, int g, u16* legal_out, int* n_legal_out) {
  Board b = load_soa(P.g_cur, P.G, g);
  u16 local[MAX_MOVES];
  u16* moves = legal_out ? legal_out : local;
  StoreSink sink{moves, 0};
  GenInfo gi = generate_legal(b, sink);
  u64 key = position_key(b, gi.ep_legal);
  int ply = meta_ply(b.meta);
  P.g_keys[(long long)(ply % KEY_RING) * P.G + g] = key;
  int reps = 0, rev = meta_revlen(b.meta);
  if (rev > KEY_RING - 1) rev = KEY_RING - 1;
  for (int i = 1; i <= rev && ply - i >= 0; ++i)
    if (P.g_keys[(long long)((ply - i) % KEY_RING) * P.G + g] == key) ++reps;
  P.g_result[g] = (int8_t)game_result(b, sink.n, gi.in_check, reps);
  if (n_legal_out) *n_legal_out = sink.n;
}

// Game.move (game.py:28-41): play `mv` if it is legal in the current position; returns 1 if played
CRL_HD int game_move(const Pools& P, int g, u16 mv) {
  Board b = load_soa(P.g_cur, P.G, g);
  u16 legal[MAX_MOVES];
  StoreSink sink{legal, 0};
  generate_legal(b, sink);
  bool ok = false;
  for (int i = 0; i < sink.n; ++i) ok = ok || legal[i] == mv;
  if (!ok || mv == MOVE_NONE) return 0;
  int ply = meta_ply(b.meta);
  if (P.g_nmoves[g] >= MAX_GAME_PLIES) {
    *P.err |= ERR_PLY_OVERFLOW;
    return 0;
  }
  // the position being left becomes history (netencoder._get_game_history pops back through it)
  u64* h = P.g_hist + (long long)(ply % HIST_RING) * 8 * P.G + g;
#pragma unroll
  for (int k = 0; k < 8; ++k) h[(long long)k * P.G] = b.bb[k];
  make_move(b, mv);
  store_soa(P.g_cur, P.G, g, b);
  P.g_moves[(long long)g * MAX_GAME_PLIES + P.g_nmoves[g]] = mv;
  P.g_nmoves[g] += 1;
  game_refresh(P, g, nullptr, nullptr);
  return 1;
}

// Tree(root) (mctree.py:104-111): node 0 = copy of the current game position, visits = 1.
// Returns 1 if the root's policy has to be evaluated, 0 if its priors were taken over from its twin in the previous
// tree (use_prev: the pools have just swapped roles and g_prev_root names the node the game moved to).
CRL_HD int root_init(const Pools& P, int g, bool use_prev = false) {
  Board b = load_soa(P.g_cur, P.G, g);
  NodeRec& r = P.nodes[(long long)g * P.NN];
  store_rec(r.p2, b);
  store_rec(r.p1, b);
  r.parent = -1;
  r.slot = 0;
  r.has_p1 = 0;
  r.move = MOVE_NONE;
  r.reply = MOVE_NONE;
  r.n_exp = 0;
  r.edge0 = 0;
  r.pending = 0;
  r.prev = -1;
  r.v = 0.f;
  r.evald = 0;
  int ply = meta_ply(b.meta);
  r.key2 = r.key1 = P.g_keys[(long long)(ply % KEY_RING) * P.G + g];
  r.result = P.g_result[g];
  u16 moves[MAX_MOVES];
  StoreSink sink{moves, 0};
  generate_legal(b, sink);
  r.n_legal = (u16)sink.n;
  P.g_nnodes[g] = 1;
  P.g_nedges[g] = sink.n;
  P.r_visits[g] = 1;
  P.r_value[g] = 0.0;
  const int twin = (use_prev && P.reuse) ? P.g_prev_root[g] : -1;
  P.g_prev_root[g] = -1;              // consumed: it named a node of the pool that is the previous tree only now
  if (sink.n > P.EA) {
    *P.err |= ERR_EDGE_OVERFLOW;
    r.n_legal = 0;
    return 0;
  }
  long long ebase = (long long)g * P.EA;
  for (int i = 0; i < sink.n; ++i) P.e_move[ebase + i] = moves[i];
  if (twin >= 0) {
    const NodeRec& t = P.nodes_prev[(long long)g * P.NN + twin];
    bool same = t.evald && t.result == RESULT_NONE && t.n_legal == sink.n;
    for (int k = 0; k < 9; ++k) same = same && t.p2[k] == r.p2[k];
    if (same) {                       // the game really is where that node stands: its priors are the root's priors
      const long long src = (long long)g * P.EA + t.edge0;
      for (int i = 0; i < sink.n; ++i) P.e_prior[ebase + i] = P.e_prior_prev[src + i];
      r.prev = twin;
      return 0;
    }
  }
  return 1;
}

}  // namespace crl
