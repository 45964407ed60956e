// kernels_tree.cu -- the lockstep PUCT search kernels and the game-record kernels.
//
// One simulation of every running game (SelfPlayTree.explore_tree, mctree.py:200-214) is the fixed kernel
// sequence  [backup of the previous simulation +] select+expand -> [evaluate P1] -> reply -> [evaluate P2] ; games
// that need no network evaluation in a phase (terminal leaves) simply do not enter that phase's compacted batch.
// simulate + backprop of a simulation run at the head of the NEXT launch of k_select_expand (k_finalize after the last).
//   * k_select_expand : one WARP per game.  The warp walks down from the root; at every fully expanded node
//     the 32 lanes scan the node's contiguous edge statistics (visits i32, value f64, prior f32, result i8)
//     with coalesced loads, score them in float64 exactly as Node.get_value does, and reduce to the FIRST
//     maximum with shuffles (np.argmax semantics).  Lane 0 then pops the last unexpanded action and creates
//     the child.
//   * expansion (SelfPlayTree.expand, mctree.py:231-257) stays with the game's warp: the legal moves of the new
//     position come from the WARP-COOPERATIVE generator (warp_gen.cuh: every lane owns two squares, a packed prefix sum
//     orders the list as python-chess does), make-move / transposition key / Game.get_result are computed redundantly
//     by all lanes (uniform, no divergence), lane 0 writes the node.  Measured alternatives, both slower at 4,096
//     games: lane 0 running the scalar generator (31 lanes idle through ~3,000 dependent instructions, 26 + 34 us for
//     select / reply) and packing 8 games' scalar generators into one warp (divergence between the 8 boards: 35 + 44 us).
// With one in-flight simulation per game (the reference's deterministic threads=1 schedule) no atomics are
// needed on the statistics; the only atomics are the batch-compaction counters.
#include "engine.cuh"
#include "warp_gen.cuh"

#include <math_constants.h>

namespace crl {

static constexpr int TREE_BLOCK = 128;
static constexpr int TREE_WARPS = TREE_BLOCK / 32;

// next row of a compacted evaluation batch.  The launches that follow cover P.row_cap rows (all lanes, or fewer when the
// host promised an upper bound on the running games): a row beyond that would silently go unevaluated, so it is an error.
__device__ __forceinline__ int take_row(const Pools& P, int* counter) {
  const int r = atomicAdd(counter, 1);
  if (r >= P.row_cap) atomicOr(P.err, ERR_ROW_OVERFLOW);
  return r;
}

// slot that searches lane g (two-network routing, DESIGN.md 3.5): the slot of the side to move at the lane's root
__device__ __forceinline__ int lane_slot(const Pools& P, int g) { return P.n_slots > 1 ? (int)P.g_slot[g] : 0; }

// a row of slot k's share of a batch: the buffer row k * slot_stride + r, which lists `item`
__device__ __forceinline__ int take_slot_row(const Pools& P, int* list, int* counter, int k, int item) {
  const int row = k * P.slot_stride + take_row(P, counter + SLOT_N_STRIDE * k);
  list[row] = item;
  return row;
}

__device__ __forceinline__ bool game_running(const Pools& P, int g) {
  return P.g_active[g] && P.g_result[g] == RESULT_NONE;
}

// VL: subtract the children's virtual loss (wave mode; with one in-flight simulation it is always zero).
// Every lane also loads the child index of the edges it scores, so the winner's child comes out of the reduction and the
// descent does not pay another dependent load per level (`child`, when asked for).
template <bool VL>
struct WarpScan {
  const Pools& P;
  int g, lane;
  __device__ __forceinline__ int operator()(const NodeRec& n, int* child = nullptr) const {
    const long long base = (long long)g * P.EA + n.edge0;
    const int cnt = n.n_exp;
    double best_s = -CUDART_INF;
    int best_k = 0x7fffffff, best_c = 0;
    for (int k = lane; k < cnt; k += 32) {
      const int c = child ? P.e_child[base + k] : 0;
      double s = edge_score(P.e_visits[base + k], P.e_value[base + k], P.e_prior[base + k], P.e_result[base + k],
                            VL ? (int)P.e_vloss[base + k] : 0);
      if (s > best_s) {
        best_s = s;
        best_k = k;
        best_c = c;
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      double os = __shfl_xor_sync(0xffffffffu, best_s, off);
      int ok = __shfl_xor_sync(0xffffffffu, best_k, off);
      int oc = __shfl_xor_sync(0xffffffffu, best_c, off);
      if (os > best_s || (os == best_s && ok < best_k)) {
        best_s = os;
        best_k = ok;
        best_c = oc;
      }
    }
    if (child) *child = best_c;
    return best_k;
  }
};

// count_repetitions (tree_core.cuh) by the whole warp: the walk through the tree's own positions is a pointer chase and
// stays serial (a handful of steps, the same in every lane); once it reaches the game's key ring the remaining positions
// have known addresses, so the lanes compare them in parallel -- up to 127 dependent loads become four.
__device__ __forceinline__ int count_repetitions_warp(const Pools& P, int g, Cursor c, u64 key, int revlen, int lane) {
  if (revlen > KEY_RING - 1) revlen = KEY_RING - 1;
  int reps = 0, i = 0;
  while (i < revlen && c.node >= 0) {
    if (!cursor_prev(P, g, c)) return reps;
    ++i;
    if (c.node >= 0 && cursor_key(P, g, c) == key) ++reps;
  }
  if (c.node >= 0) return reps;                    // the reversible run ended inside the tree
  // c now points at the ring position of ply c.ply, reached by step i but not compared yet; the serial walk would
  // compare it and then step (revlen - i) more times, never below ply 0
  int m = revlen - i + 1;
  if (m > c.ply + 1) m = c.ply + 1;
  int mine = 0;
  for (int j = lane; j < m; j += 32)
    mine += P.g_keys[(long long)((c.ply - j) % KEY_RING) * P.G + g] == key;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, off);
  return reps + mine;
}

// analyse_position (tree_core.cuh) with the warp-cooperative generator: every lane calls it with the same arguments
// and gets the same results; the legal moves land in `moves` (shared or global memory).
__device__ __forceinline__ int analyse_position_warp(const Pools& P, int g, const Board& b, Cursor at, u16* moves, int lane,
                                                     int* n_moves, u64* key) {
  int in_check, ep_legal;
  const int n = warp_generate_legal(b, moves, lane, &in_check, &ep_legal);
  *n_moves = n;
  *key = position_key(b, ep_legal);
  int reps = 0;
  const int rev = meta_revlen(b.meta);
  if (rev >= 8 && n > 0 && meta_halfmove(b.meta) < 100 && !insufficient_material(b))
    reps = count_repetitions_warp(P, g, at, *key, rev, lane);
  return game_result(b, n, in_check, reps);
}

// expand_child (tree_core.cuh; mctree.py:241-244) run by the whole warp: uniform reads and arithmetic in every lane,
// the node's fields written by lane 0, the legal moves of P1 generated cooperatively into the slot's move row.
__device__ __forceinline__ int expand_child_warp(const Pools& P, int g, int slot, int parent, int lane, int* out_child,
                                                 int* out_twin = nullptr, int* out_n_moves = nullptr) {
  NodeRec& pn = P.nodes[(long long)g * P.NN + parent];
  const int child = P.g_nnodes[g];
  const int k = pn.n_exp;
  const int twin = twin_of_child(P, g, pn, k);                 // same node in the previous move's tree, or -1
  if (out_twin) *out_twin = twin;
  const long long ebase = (long long)g * P.EA + pn.edge0;
  const u16 mv = P.e_move[ebase + (pn.n_legal - 1 - k)];       // unexpanded_actions.pop(): last legal move first
  Board b = load_rec(pn.p2);
  __syncwarp();                                                // every lane has read what lane 0 is about to change
  if (child >= P.NN) {
    if (lane == 0) *P.err |= ERR_NODE_OVERFLOW;
    *out_child = parent;
    return KIND_IDLE;
  }
  make_move(b, mv);
  NodeRec& cn = P.nodes[(long long)g * P.NN + child];
  if (lane == 0) {
    P.g_nnodes[g] = child + 1;
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
    cn.prev = twin;
    cn.v = 0.f;
    cn.evald = 0;
    P.e_child[ebase + k] = child;
    P.e_visits[ebase + k] = 0;
    P.e_value[ebase + k] = 0.0;
    P.e_vloss[ebase + k] = 0;
    pn.n_exp = (u16)(k + 1);
  }
  __syncwarp();                                                // the repetition walk reads cn.parent in every lane
  const Cursor at{child, 1, meta_ply(b.meta)};
  int n_moves;
  u64 key;
  const int res = analyse_position_warp(P, g, b, at, P.s_moves + (long long)slot * MAX_MOVES, lane, &n_moves, &key);
  *out_child = child;
  if (out_n_moves) *out_n_moves = n_moves;
  if (lane == 0) {
    cn.key1 = key;
    P.s_nmoves[slot] = n_moves;
    if (res != RESULT_NONE) {          // the game ended on our move: the child's state is P1 (mctree.py:244)
      store_rec(cn.p2, b);
      cn.key2 = key;
      cn.result = (int8_t)res;
      cn.n_legal = (u16)n_moves;
    } else {
      cn.result = RESULT_NONE;
      cn.pending = 1;                  // until the reply is known; only wave-mode selects can meet it
    }
    P.e_result[ebase + k] = (int8_t)res;
  }
  return res != RESULT_NONE ? KIND_NEW_TERMINAL : KIND_NEED_REPLY;
}

// reply_child (tree_core.cuh; mctree.py:245-249) run by the whole warp; `gen` = this warp's shared-memory move row
__device__ __forceinline__ int reply_child_warp(const Pools& P, int g, int slot, int child, int pick, int lane, u16* gen) {
  NodeRec& cn = P.nodes[(long long)g * P.NN + child];
  const u16 reply = P.s_moves[(long long)slot * MAX_MOVES + pick];
  Board b = load_rec(cn.p1);
  const int parent = cn.parent, cslot = cn.slot;
  make_move(b, reply);
  const Cursor at{child, 2, meta_ply(b.meta)};
  int n2;
  u64 key;
  if (lane == 0) cn.reply = reply;     // the walk from P2 steps to P1 of this node only if it has a reply
  __syncwarp();
  const int res = analyse_position_warp(P, g, b, at, gen, lane, &n2, &key);
  const NodeRec& pn = P.nodes[(long long)g * P.NN + parent];
  const long long pedge = (long long)g * P.EA + pn.edge0 + cslot;
  int e0 = 0;
  if (lane == 0) {
    store_rec(cn.p2, b);
    cn.key2 = key;
    cn.result = (int8_t)res;
    cn.n_legal = (u16)n2;
    cn.pending = 0;
    P.e_result[pedge] = (int8_t)res;
    // reserve the node's edge slots (Node.unexpanded_actions, mctree.py:31); atomic because in wave mode several
    // rows of one game run concurrently -- where a node's edges sit inside the arena influences no result
    if (res == RESULT_NONE) e0 = atomicAdd(&P.g_nedges[g], n2);
  }
  if (res != RESULT_NONE) return KIND_NEW_TERMINAL;
  e0 = __shfl_sync(0xffffffffu, e0, 0);
  if (e0 + n2 > P.EA) {
    if (lane == 0) {
      *P.err |= ERR_EDGE_OVERFLOW;
      cn.n_legal = 0;
      cn.result = 0;                   // poison as a drawn leaf so the search stays well-defined; the host raises on err
      P.e_result[pedge] = 0;
    }
    return KIND_NEW_TERMINAL;
  }
  if (lane == 0) cn.edge0 = e0;
  __syncwarp();                        // the generated list in shared memory is complete
  const long long ebase = (long long)g * P.EA + e0;
  for (int i = lane; i < n2; i += 32) P.e_move[ebase + i] = gen[i];
  return KIND_EVAL_LEAF;
}

// adopt_evaluation (tree_core.cuh) by the whole warp: the twin's value and its children's priors become the node's
__device__ __forceinline__ bool adopt_evaluation_warp(const Pools& P, int g, int node, int twin, int lane) {
  NodeRec& n = P.nodes[(long long)g * P.NN + node];
  const NodeRec& t = P.nodes_prev[(long long)g * P.NN + twin];
  const int L = n.n_legal;
  if (t.result != RESULT_NONE || t.n_legal != L) return false;
  const long long dst = (long long)g * P.EA + n.edge0, src = (long long)g * P.EA + t.edge0;
  for (int i = lane; i < L; i += 32) P.e_prior[dst + i] = P.e_prior_prev[src + i];
  if (lane == 0) {
    n.v = t.v;
    n.evald = 1;
  }
  return true;
}

// SelfPlayTree.simulate + backprop (mctree.py:259-296) of the simulation a game has in flight (exact schedule), by the
// game's warp: the lanes cache the evaluated node's legal-order policy on its edge slots, then apply the backup to the
// RECORDED path -- k_select_expand left the edge index of depth d in s_path[g][d] -- one lane per level: the
// (visits += 1, value += v) updates of different edges are independent, so up to 32 levels cost one round of memory
// latency instead of a parent-pointer chase of three dependent loads per level.  Deeper paths fall back to the chase.
__device__ __forceinline__ void finalize_pending(const Pools& P, int g, int lane, const PolicyView& pv,
                                                 const float* __restrict__ value, const int16_t* __restrict__ label_of) {
  const int kind = P.s_kind[g];
  if (kind == KIND_IDLE || kind == KIND_NEED_REPLY) return;   // nothing in flight (NEED_REPLY: a row the evaluator never saw)
  const int node = P.s_node[g];
  NodeRec& n = P.nodes[(long long)g * P.NN + node];
  double v;
  if (kind == KIND_EVAL_LEAF) {
    const int row = P.s_row[g];
    const long long ebase = (long long)g * P.EA + n.edge0;
    const int L = n.n_legal;
    for (int i = lane; i < L; i += 32) {     // store_priors, mirrored: legal move i -> child slot L-1-i
      const u16 m = P.e_move[ebase + i];
      P.e_prior[ebase + (L - 1 - i)] = policy_at(pv, row, label_of[(int)mv_promo(m) * 4096 + mv_from(m) * 64 + mv_to(m)]);
    }
    const float vf = value[row];
    v = (double)vf;                                           // float(v) of a float32 (predict_worker.py:111)
    if (lane == 0) {
      n.v = vf;                                               // kept for the next move's search (evaluation reuse)
      n.evald = 1;
      atomicAdd((unsigned long long*)&P.counters[1], 1ull);   // the evaluation of this leaf
    }
  } else if (kind == KIND_EVAL_REUSED) {
    v = (double)n.v;                                          // the same float32 the previous search got from the network
  } else {
    v = (double)n.result;                                     // terminal: Game.get_result (mctree.py:268)
  }
  const int depth = P.s_depth[g];
  if (depth >= 0) {
    if (lane < depth) {
      const long long e = (long long)g * P.EA + P.s_path[(long long)g * 32 + lane];
      P.e_visits[e] += 1;
      P.e_value[e] += v;
    }
    if (lane == 0) {
      P.r_visits[g] += 1;
      P.r_value[g] += v;
    }
  } else if (lane == 0) {
    backup(P, g, node, v);
  }
  if (lane == 0) {
    atomicAdd((unsigned long long*)&P.counters[0], 1ull);
    P.s_kind[g] = KIND_IDLE;
  }
  __syncwarp();                                               // the select that follows reads these statistics
}

// The head of one lockstep simulation: finish the simulation the game still has in flight (its evaluation batch B ran
// after the previous launch of this kernel), then select + expand the next one.  Fusing the two removes a launch and its
// tail from every simulation and lets the backup run level-parallel on the recorded path.
// (7 blocks = 28 warps per SM: 148 x 28 = 4,144 resident warps, so 4,096 games run as ONE wave instead of 1.5)
// list_b / n_b: batch B of this simulation (node states to evaluate), which k_reply fills; with evaluation reuse a warp
// whose new child has a twin in the previous tree plays the twin's reply at once -- no batch-A row -- and normally takes
// the twin's value and priors as well, so that simulation runs without the network.
__global__ void __launch_bounds__(TREE_BLOCK, 7) k_select_expand(Pools P, PolicyView pv, const float* __restrict__ value,
                                                              const int16_t* __restrict__ label_of, int* list_b, int* n_b) {
  __shared__ u16 s_gen[TREE_WARPS][MAX_MOVES];
  const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (g >= P.G) return;
  finalize_pending(P, g, lane, pv, value, label_of);
  if (!game_running(P, g)) return;             // s_kind[g] is KIND_IDLE
  // SelfPlayTree.select (mctree.py:216-229), recording the edge taken at every level
  int node = 0, depth = 0, my_edge = 0, term = 0;
  const WarpScan<false> scan{P, g, lane};
  for (;;) {
    const NodeRec& n = P.nodes[(long long)g * P.NN + node];
    if (n.result != RESULT_NONE) {
      term = 1;
      break;
    }
    if (n.n_exp < n.n_legal) break;
    int next;
    const int e = n.edge0 + scan(n, &next);
    if (lane == (depth & 31)) my_edge = e;
    ++depth;
    node = next;
  }
  if (term) {
    if (depth <= P.path_cap) P.s_path[(long long)g * 32 + lane] = my_edge;
    if (lane == 0) {
      P.s_depth[g] = depth <= P.path_cap ? depth : -1;
      P.s_node[g] = node;
      P.s_kind[g] = KIND_TERMINAL;
    }
    return;
  }
  {
    const NodeRec& pn = P.nodes[(long long)g * P.NN + node];
    const int e = pn.edge0 + pn.n_exp;         // the edge the new child is about to take
    if (lane == (depth & 31)) my_edge = e;
    ++depth;
    if (depth <= P.path_cap) P.s_path[(long long)g * 32 + lane] = my_edge;
    if (lane == 0) P.s_depth[g] = depth <= P.path_cap ? depth : -1;
  }
  int child, twin, n1;
  int kind = expand_child_warp(P, g, g, node, lane, &child, &twin, &n1);
  if (kind == KIND_NEED_REPLY && twin >= 0) {
    const u16 reply = P.nodes_prev[(long long)g * P.NN + twin].reply;
    const u16* moves1 = P.s_moves + (long long)g * MAX_MOVES;
    __syncwarp();                                  // the move row was written by all lanes of this warp just now
    int pick = 0x7fffffff;
    for (int i = lane; i < n1; i += 32)
      if (moves1[i] == reply) pick = i;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) pick = min(pick, __shfl_xor_sync(0xffffffffu, pick, off));
    if (pick < n1) {                               // always, unless the pools were tampered with: then evaluate as usual
      kind = reply_child_warp(P, g, g, child, pick, lane, s_gen[threadIdx.x >> 5]);
      int reused = 1;
      if (kind == KIND_EVAL_LEAF) {
        __syncwarp();
        if (adopt_evaluation_warp(P, g, child, twin, lane)) {
          kind = KIND_EVAL_REUSED;
          reused = 2;
        }
      }
      if (lane != 0) return;
      atomicAdd((unsigned long long*)&P.counters[2], (unsigned long long)reused);
      P.s_node[g] = child;
      P.s_kind[g] = kind;
      if (kind == KIND_EVAL_LEAF)                  // (defensive) the twin's evaluation did not fit: run it
        P.s_row[g] = take_slot_row(P, list_b, n_b, lane_slot(P, g), g);
      return;
    }
  }
  if (lane != 0) return;
  P.s_node[g] = child;
  P.s_kind[g] = kind;
  if (kind == KIND_NEED_REPLY) P.s_row[g] = take_slot_row(P, P.eval_list, P.eval_n, lane_slot(P, g), g);
}

// ---- wave mode: K in-flight simulations per game (the reference's --threads K, mctree.py:173-176) -----------
// One WARP per game runs the wave's selects one after the other (each sees the virtual losses and the
// expansions of the earlier ones, exactly as in the schedule described at select_descend_wave); slot j of
// game g is scratch index g*K + j.  The wave ends early when a select would enter a node whose reply is still
// being evaluated.
__global__ void __launch_bounds__(TREE_BLOCK) k_wave_begin(Pools P, int n_sims) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= P.G) return;
  P.g_sims_left[g] = game_running(P, g) ? n_sims : 0;
  P.s_wave_n[g] = 0;
}

__global__ void __launch_bounds__(TREE_BLOCK) k_select_wave(Pools P) {
  const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (g >= P.G) return;
  const int left = game_running(P, g) ? P.g_sims_left[g] : 0;
  const int kmax = min(P.K, left);
  const int ks = lane_slot(P, g);
  int used = 0;
  for (int j = 0; j < kmax; ++j) {
    int node = 0;
    const int what = select_descend_wave(P, g, WarpScan<true>{P, g, lane}, &node);
    if (what == 2) break;
    const int slot = g * P.K + used;
    // wave_take_slot (tree_core.cuh) with the expansion done by the whole warp
    int kind = KIND_TERMINAL, leaf = node;
    if (what != 1) kind = expand_child_warp(P, g, slot, node, lane, &leaf);
    if (lane == 0) {
      P.s_node[slot] = leaf;
      P.s_kind[slot] = kind;
      if (kind != KIND_IDLE) vloss_add(P, g, leaf, 1);
      if (kind == KIND_NEED_REPLY) P.s_row[slot] = take_slot_row(P, P.eval_list, P.eval_n, ks, slot);
      __threadfence_block();
    }
    __syncwarp();
    ++used;
  }
  if (lane == 0) {
    P.s_wave_n[g] = used;
    P.g_sims_left[g] = left - used;
  }
}

// simulate + backprop of the wave, in slot order (value += v is a float64 sum: the order is part of the result)
__global__ void __launch_bounds__(TREE_BLOCK) k_finalize_wave(Pools P, PolicyView pv, const float* __restrict__ value,
                                                              const int16_t* __restrict__ label_of) {
  const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (g == 0 && lane == 0)
    atomicAdd((unsigned long long*)&P.counters[1],
              (unsigned long long)(*P.eval_n + (P.n_slots > 1 ? P.eval_n[SLOT_N_STRIDE] : 0)));
  if (g >= P.G) return;
  const int used = P.s_wave_n[g];
  for (int j = 0; j < used; ++j) {
    const int slot = g * P.K + j;
    const int node = P.s_node[slot];
    const int kind = P.s_kind[slot];
    if (kind == KIND_IDLE) continue;          // node pool overflow (flagged in P.err)
    NodeRec& n = P.nodes[(long long)g * P.NN + node];
    double v;
    if (kind == KIND_EVAL_LEAF) {
      const int row = P.s_row[slot];
      const long long ebase = (long long)g * P.EA + n.edge0;
      const int L = n.n_legal;
      for (int i = lane; i < L; i += 32) {
        const u16 m = P.e_move[ebase + i];
        P.e_prior[ebase + (L - 1 - i)] = policy_at(pv, row, label_of[(int)mv_promo(m) * 4096 + mv_from(m) * 64 + mv_to(m)]);
      }
      const float vf = value[row];
      v = (double)vf;
      if (lane == 0) {
        n.v = vf;          // kept for the next move's search (evaluation reuse)
        n.evald = 1;
      }
    } else {
      v = (double)n.result;
    }
    if (lane == 0) {
      backup(P, g, node, v);
      vloss_add(P, g, node, -1);
      P.s_kind[slot] = KIND_IDLE;             // nothing in flight any more (k_select_expand finishes what it finds)
    }
  }
  if (lane == 0 && used > 0) atomicAdd((unsigned long long*)&P.counters[0], (unsigned long long)used);
}

// largest number of simulations any game still has to run (the host loops on it)
__global__ void __launch_bounds__(256) k_wave_left(Pools P, int* out) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  int v = (g < P.G && game_running(P, g)) ? P.g_sims_left[g] : 0;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, off));
  if ((threadIdx.x & 31) == 0 && v > 0) atomicMax(out, v);
}

// rows of batch A (positions after our move) -> opponent reply, node state, batch B.
// One WARP per row: the lanes gather the legal-masked policy in parallel and reduce to the FIRST maximum
// (agentdistributed.py:56-58), then play the reply and build the node together (mctree.py:245-249).
// blockIdx.y = network slot: the reply is predicted by the searching side's network, and the leaf goes to its batch B.
__global__ void __launch_bounds__(TREE_BLOCK, 7) k_reply(Pools P, PolicyView pv, const int16_t* __restrict__ label_of,
                                                      int* list_b, int* n_b) {
  __shared__ u16 s_gen[TREE_WARPS][MAX_MOVES];
  const int ks = blockIdx.y;
  const int r0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int n_a = P.eval_n[SLOT_N_STRIDE * ks];
  if (r0 == 0 && lane == 0) atomicAdd((unsigned long long*)&P.counters[1], (unsigned long long)n_a);
  if (r0 >= n_a) return;
  const int r = ks * P.slot_stride + r0;
  const int slot = P.eval_list[r];
  const int g = slot / P.K;
  const int child = P.s_node[slot];
  const u16* moves1 = P.s_moves + (long long)slot * MAX_MOVES;
  const int n1 = P.s_nmoves[slot];
  // (issued now, used by reply_child_warp after the gather below: the record's lines are on their way meanwhile)
  asm volatile("prefetch.global.L2 [%0];" ::"l"(&P.nodes[(long long)g * P.NN + child]));
  asm volatile("prefetch.global.L2 [%0];" ::"l"((const char*)&P.nodes[(long long)g * P.NN + child] + 128));
  float best_p = -CUDART_INF_F;
  int best_i = 0x7fffffff;
  for (int i = lane; i < n1; i += 32) {
    const u16 m = moves1[i];
    const float p = policy_at(pv, r, label_of[(int)mv_promo(m) * 4096 + mv_from(m) * 64 + mv_to(m)]);
    if (p > best_p) {
      best_p = p;
      best_i = i;
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const float op = __shfl_xor_sync(0xffffffffu, best_p, off);
    const int oi = __shfl_xor_sync(0xffffffffu, best_i, off);
    if (op > best_p || (op == best_p && oi < best_i)) {
      best_p = op;
      best_i = oi;
    }
  }
  const int kind = reply_child_warp(P, g, slot, child, best_i, lane, s_gen[threadIdx.x >> 5]);
  if (lane != 0) return;
  P.s_kind[slot] = kind;
  if (kind == KIND_EVAL_LEAF) P.s_row[slot] = take_slot_row(P, list_b, n_b, ks, slot);
}

// the last simulation of a crl_mcts_simulate call has no following k_select_expand to finish it: this does
__global__ void __launch_bounds__(TREE_BLOCK) k_finalize(Pools P, PolicyView pv, const float* __restrict__ value,
                                                         const int16_t* __restrict__ label_of) {
  const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (g >= P.G) return;
  finalize_pending(P, g, lane, pv, value, label_of);
}

// Tree(root): build node 0 of every running game and queue it for evaluation
__global__ void __launch_bounds__(TREE_BLOCK) k_root_init(Pools P, const u8* __restrict__ mask, int use_prev) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= P.G) return;
  P.s_kind[g] = KIND_IDLE;
  if (!game_running(P, g)) {
    P.g_nnodes[g] = 0;          // no tree this move: root statistics of a finished / parked lane read as empty, not as
    P.g_prev_root[g] = -1;      // whatever an earlier search left in this pool
    return;
  }
  if (mask && !mask[g]) return;
  P.s_node[g] = 0;
  if (P.n_slots > 1)                           // the side to move at the root searches with its slot
    P.g_slot[g] = P.g_players[(meta_turn(P.g_cur[8LL * P.G + g]) ? 0 : P.G) + g];
  if (!root_init(P, g, use_prev != 0)) {       // priors taken over from the previous tree: no evaluation
    atomicAdd((unsigned long long*)&P.counters[2], 1ull);
    return;
  }
  P.s_row[g] = take_slot_row(P, P.eval_list, P.eval_n, lane_slot(P, g), g);
}

// blockIdx.y = network slot (its rows start at row blockIdx.y * slot_stride)
__global__ void __launch_bounds__(TREE_BLOCK) k_root_priors(Pools P, PolicyView pv,
                                                            const int16_t* __restrict__ label_of) {
  const int r0 = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = P.eval_n[SLOT_N_STRIDE * blockIdx.y];
  if (r0 == 0) atomicAdd((unsigned long long*)&P.counters[1], (unsigned long long)n);
  if (r0 >= n) return;
  const int r = blockIdx.y * P.slot_stride + r0;
  const int g = P.eval_list[r];
  store_priors_of(P, g, 0, [&](int label) { return policy_at(pv, r, label); }, label_of);
}

// AgentDistributed.best_move(real_game=True): argmax of the legal-masked policy of the current position
__global__ void __launch_bounds__(TREE_BLOCK) k_policy_move(Pools P, PolicyView pv,
                                                            const int16_t* __restrict__ label_of,
                                                            u16* __restrict__ picks) {
  const int r0 = blockIdx.x * blockDim.x + threadIdx.x;
  if (r0 >= P.eval_n[SLOT_N_STRIDE * blockIdx.y]) return;
  const int r = blockIdx.y * P.slot_stride + r0;
  const int g = P.eval_list[r];
  const NodeRec& root = P.nodes[(long long)g * P.NN];
  const u16* moves = P.e_move + (long long)g * P.EA + root.edge0;
  u16 mv = MOVE_NONE;
  if (root.n_legal > 0)
    mv = moves[argmax_legal_of([&](int label) { return policy_at(pv, r, label); }, label_of, moves, root.n_legal)];
  picks[g] = mv;
  game_move(P, g, mv);
  P.g_prev_root[g] = -1;
}

// ---- game records -------------------------------------------------------------------------------------
// lanes != null: game i goes to lane lanes[i] (scattered refill) and all games share start_aos[0..8]
__global__ void __launch_bounds__(TREE_BLOCK) k_games_replay(Pools P, int first, int n, const int* __restrict__ lanes,
                                                             const u64* __restrict__ start_aos,
                                                             const u16* __restrict__ moves,
                                                             const int* __restrict__ n_moves, int stride,
                                                             u8* __restrict__ accepted, u64* __restrict__ records,
                                                             int* __restrict__ n_records) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int g = lanes ? lanes[i] : first + i;
  Board b = load_rec(lanes ? start_aos : start_aos + 9LL * i);
  // a fresh record starts with an empty move stack (Board(fen) / Game())
  b.meta = meta_pack(meta_turn(b.meta), meta_castle(b.meta), meta_ep(b.meta), meta_halfmove(b.meta),
                     meta_fullmove(b.meta), 0, 0);
  store_soa(P.g_cur, P.G, g, b);
  P.g_nmoves[g] = 0;
  P.g_active[g] = 1;
  P.g_nnodes[g] = 0;
  P.g_prev_root[g] = -1;
  game_refresh(P, g, nullptr, nullptr);
  // optional: the record after every ACCEPTED move (AoS, record j of game i at records[(i*(stride+1) + j)*9]);
  // record 0 is the start position.  This is what Board.copy() + pop() walks back through (netencoder.py:58-67).
  int nrec = 0;
  u64* rec = records ? records + (long long)i * (stride + 1) * 9 : nullptr;
  if (rec) store_rec(rec + 9LL * nrec++, b);
  const int m = n_moves ? n_moves[i] : 0;
  for (int k = 0; k < m; ++k) {
    int ok = game_move(P, g, moves[(long long)i * stride + k]);
    if (accepted) accepted[(long long)i * stride + k] = (u8)ok;
    if (rec && ok) store_rec(rec + 9LL * nrec++, load_soa(P.g_cur, P.G, g));
  }
  if (n_records) n_records[i] = nrec;
}

// what game.Game exposes about the current position: legal moves (python-chess order) and get_result
__global__ void __launch_bounds__(TREE_BLOCK) k_game_info(Pools P, int first, int n, u16* __restrict__ legal,
                                                          int* __restrict__ n_legal) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Board b = load_soa(P.g_cur, P.G, first + i);
  StoreSink sink{legal + (long long)i * MAX_MOVES, 0};
  generate_legal(b, sink);
  n_legal[i] = sink.n;
}

// one optional move per game (MOVE_NONE = none), through Game.move's legality check
__global__ void __launch_bounds__(TREE_BLOCK) k_game_moves(Pools P, const u16* __restrict__ mv,
                                                           u8* __restrict__ accepted) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= P.G) return;
  int ok = 0;
  if (P.g_active[g] && mv[g] != MOVE_NONE) ok = game_move(P, g, mv[g]);
  if (ok) P.g_prev_root[g] = -1;             // the position no longer is a node of the last tree
  if (accepted) accepted[g] = (u8)ok;
}

// move lists of the listed lanes (finished games on their way to gameplays.json): one block per lane
__global__ void __launch_bounds__(TREE_BLOCK) k_gather_moves(Pools P, const int* __restrict__ lanes, int n, int cap,
                                                             u16* __restrict__ out, int* __restrict__ n_out) {
  const int i = blockIdx.x;
  if (i >= n) return;
  const int g = lanes[i];
  const int m = P.g_nmoves[g];
  if (threadIdx.x == 0) n_out[i] = m;
  const u16* src = P.g_moves + (long long)g * MAX_GAME_PLIES;
  for (int k = threadIdx.x; k < min(m, cap); k += blockDim.x) out[(long long)i * cap + k] = src[k];
}

// search_move's return value (mctree.py:178-198) for the chosen root child of every game
__global__ void __launch_bounds__(TREE_BLOCK) k_commit(Pools P, const int* __restrict__ pick,
                                                       u16* __restrict__ out_moves, int apply) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= P.G) return;
  u16 m0 = MOVE_NONE, m1 = MOVE_NONE;
  const int k = pick[g];
  const NodeRec& root = P.nodes[(long long)g * P.NN];
  const bool has_tree = P.g_active[g] && P.g_nnodes[g] > 0;      // (a lane without a running game got no tree this move)
  if (has_tree && k >= 0 && k < root.n_exp) {
    const NodeRec& c = P.nodes[(long long)g * P.NN + P.e_child[(long long)g * P.EA + root.edge0 + k]];
    if (c.reply != MOVE_NONE) {
      m0 = c.move;             // move_stack[-2] = our move, [-1] = the opponent's reply
      m1 = c.reply;
    } else if (P.g_nmoves[g] >= 1) {
      m0 = P.g_moves[(long long)g * MAX_GAME_PLIES + P.g_nmoves[g] - 1];   // previous ply (reference quirk)
      m1 = c.move;
    }                          // else: IndexError in the reference -> both stay the null move
  }
  out_moves[2 * g] = m0;
  out_moves[2 * g + 1] = m1;
  int next_root = -1;
  if (apply && has_tree && k >= 0) {
    const int ok0 = game_move(P, g, m0);       // selfplay.py:77-78: Game.move silently rejects an illegal first move
    const int ok1 = game_move(P, g, m1);
    // the game now stands where the chosen child stands: the next search may take evaluations from this tree
    if (ok0 && ok1 && k < root.n_exp) {
      const int c = P.e_child[(long long)g * P.EA + root.edge0 + k];
      if (P.nodes[(long long)g * P.NN + c].reply == m1 && P.nodes[(long long)g * P.NN + c].move == m0) next_root = c;
    }
  }
  P.g_prev_root[g] = next_root;
}

// ---- launchers ----------------------------------------------------------------------------------------
int launch_games_replay(crl_engine_impl* e, int first, int n, const u64* start_aos, const u16* moves,
                        const int* n_moves, int stride, u8* accepted, u64* records, int* n_records, const int* lanes) {
  LaunchScope ls(e, KC_GAME);
  k_games_replay<<<div_up(n, TREE_BLOCK), TREE_BLOCK, 0, e->stream>>>(e->P, first, n, lanes, start_aos, moves, n_moves,
                                                                      stride, accepted, records, n_records);
  CRL_CUDA(cudaGetLastError());
  return CRL_OK;
}
int launch_game_info(crl_engine_impl* e, int first, int n, u16* legal, int* n_legal) {
  LaunchScope ls(e, KC_GAME);
  k_game_info<<<div_up(n, TREE_BLOCK), TREE_BLOCK, 0, e->stream>>>(e->P, first, n, legal, n_legal);
  CRL_CUDA(cudaGetLastError());
  return CRL_OK;
}
int launch_gather_moves(crl_engine_impl* e, const int* lanes, int n, int cap, u16* out, int* n_out) {
  LaunchScope ls(e, KC_GAME);
  k_gather_moves<<<n, TREE_BLOCK, 0, e->stream>>>(e->P, lanes, n, cap, out, n_out);
  CRL_CUDA(cudaGetLastError());
  return CRL_OK;
}
int launch_game_moves(crl_engine_impl* e, const u16* mv, u8* accepted) {
  LaunchScope ls(e, KC_GAME);
  k_game_moves<<<div_up(e->G, TREE_BLOCK), TREE_BLOCK, 0, e->stream>>>(e->P, mv, accepted);
  CRL_CUDA(cudaGetLastError());
  return CRL_OK;
}


// rows the evaluation kernels are launched for: every lane (times K), or the host's promise (crl_mcts_set_row_bound)
static void set_rows(crl_engine_impl* e, int K) {
  long long rows = (long long)e->G * K;
  if (e->row_bound > 0 && (long long)e->row_bound * K < rows) rows = (long long)e->row_bound * K;
  e->cur_rows = (int)rows;
  e->P.row_cap = (int)rows;
}

static int use_list(crl_engine_impl* e, int which) {
  e->P.eval_list = e->d_list[which];
  e->P.eval_n = e->d_n + which;
  return CRL_OK;
}

// Tree(root) for every running game (or the masked subset): node 0, its legal moves, its priors
// use_prev: a new move search of ALL lanes with evaluation reuse on -- the pools swap roles first, so the tree just
// searched becomes the previous tree the new one looks its twins up in
// the row counters of batches A and B, of every slot the search routes rows to
static int clear_counts(crl_engine_impl* e) {
  CRL_CUDA(cudaMemsetAsync(e->d_n, 0, 2 * sizeof(int), e->stream));
  if (e->search_slots > 1) CRL_CUDA(cudaMemsetAsync(e->d_n + SLOT_N_STRIDE, 0, 2 * sizeof(int), e->stream));
  return CRL_OK;
}

int tree_begin_move(crl_engine_impl* e, const u8* mask_dev, bool use_prev) {
  if (use_prev) {
    std::swap(e->P.nodes, e->P.nodes_prev);
    std::swap(e->P.e_prior, e->P.e_prior_prev);
    std::swap(e->P.e_child, e->P.e_child_prev);
    e->tree_parity ^= 1;
  }
  if (int rc = clear_counts(e)) return rc;
  use_list(e, 0);
  e->P.K = 1;                 // root batch: one row per game
  e->P.reuse = e->reuse ? 1 : 0;
  set_rows(e, 1);
  {
    LaunchScope ls(e, KC_TREE);
    k_root_init<<<div_up(e->G, TREE_BLOCK), TREE_BLOCK, 0, e->stream>>>(e->P, mask_dev, use_prev ? 1 : 0);
    CRL_CUDA(cudaGetLastError());
  }
  int rc = launch_eval_batch(e, 0);
  if (rc != CRL_OK) return rc;
  {
    LaunchScope ls(e, KC_TREE);
    k_root_priors<<<dim3(div_up(e->G, TREE_BLOCK), e->search_slots), TREE_BLOCK, 0, e->stream>>>(e->P, e->pview,
                                                                                                 e->d_label_of);
    CRL_CUDA(cudaGetLastError());
  }
  return CRL_OK;
}

// one lockstep simulation of every running game: the fixed kernel sequence described at the top of this file
static int one_simulation(crl_engine_impl* e) {
  if (int rc = clear_counts(e)) return rc;
  use_list(e, 0);
  e->P.K = 1;
  e->P.reuse = e->reuse ? 1 : 0;
  set_rows(e, 1);
  {
    LaunchScope ls(e, KC_TREE);
    k_select_expand<<<div_up((long long)e->G * 32, TREE_BLOCK), TREE_BLOCK, 0, e->stream>>>(
        e->P, e->pview, e->d_value, e->d_label_of, e->d_list[1], e->d_n + 1);
    CRL_CUDA(cudaGetLastError());
  }
  int rc = launch_eval_batch(e, 1);
  if (rc != CRL_OK) return rc;
  {
    LaunchScope ls(e, KC_TREE);
    k_reply<<<dim3(div_up((long long)e->G * 32, TREE_BLOCK), e->search_slots), TREE_BLOCK, 0, e->stream>>>(
        e->P, e->pview, e->d_label_of, e->d_list[1], e->d_n + 1);
    CRL_CUDA(cudaGetLastError());
  }
  use_list(e, 1);
  return launch_eval_batch(e, 2);      // its results are consumed by the next k_select_expand, or by finish_simulations
}

// simulate + backprop of the last simulation in flight (exact schedule)
static int finish_simulations(crl_engine_impl* e) {
  e->P.K = 1;
  LaunchScope ls(e, KC_TREE);
  k_finalize<<<div_up((long long)e->G * 32, TREE_BLOCK), TREE_BLOCK, 0, e->stream>>>(e->P, e->pview, e->d_value, e->d_label_of);
  CRL_CUDA(cudaGetLastError());
  return CRL_OK;
}

// one WAVE of every running game: up to K selects per game, two evaluation batches of up to G*K rows, backups
static int one_wave(crl_engine_impl* e, int K) {
  if (int rc = clear_counts(e)) return rc;
  use_list(e, 0);
  e->P.K = K;
  e->P.reuse = 0;             // the wave schedule evaluates everything (twins are looked up in the exact schedule only)
  set_rows(e, K);
  {
    LaunchScope ls(e, KC_TREE);
    k_select_wave<<<div_up((long long)e->G * 32, TREE_BLOCK), TREE_BLOCK, 0, e->stream>>>(e->P);
    CRL_CUDA(cudaGetLastError());
  }
  int rc = launch_eval_batch(e, 1);
  if (rc != CRL_OK) return rc;
  {
    LaunchScope ls(e, KC_TREE);
    k_reply<<<dim3(div_up((long long)e->cur_rows * 32, TREE_BLOCK), e->search_slots), TREE_BLOCK, 0, e->stream>>>(
        e->P, e->pview, e->d_label_of, e->d_list[1], e->d_n + 1);
    CRL_CUDA(cudaGetLastError());
  }
  use_list(e, 1);
  rc = launch_eval_batch(e, 2);
  if (rc != CRL_OK) return rc;
  {
    LaunchScope ls(e, KC_TREE);
    k_finalize_wave<<<div_up((long long)e->G * 32, TREE_BLOCK), TREE_BLOCK, 0, e->stream>>>(e->P, e->pview, e->d_value,
                                                                                           e->d_label_of);
    CRL_CUDA(cudaGetLastError());
  }
  return CRL_OK;
}

static int one_step(crl_engine_impl* e, int K) { return K <= 1 ? one_simulation(e) : one_wave(e, K); }

// number of simulations the slowest game still has to run in the current wave-mode call (host sync)
static int wave_left(crl_engine_impl* e, int* out) {
  int* d_left = e->d_n + 2;
  CRL_CUDA(cudaMemsetAsync(d_left, 0, sizeof(int), e->stream));
  {
    LaunchScope ls(e, KC_TREE);
    k_wave_left<<<div_up(e->G, 256), 256, 0, e->stream>>>(e->P, d_left);
    CRL_CUDA(cudaGetLastError());
  }
  CRL_CUDA(cudaMemcpyAsync(out, d_left, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
  CRL_CUDA(cudaStreamSynchronize(e->stream));
  return CRL_OK;
}

// The sequence is identical for every simulation (batch sizes live in device memory), so it is captured once
// into a CUDA graph and replayed: one graph launch instead of ~10 kernel launches per simulation.
// K = 1: n_sims lockstep simulations (the exact threads=1 schedule).  K > 1: waves of up to K simulations per game
// until every running game has done n_sims; games whose waves were cut short need a few extra waves, found by
// polling the device once per batch of waves.
int tree_simulate(crl_engine_impl* e, int n_sims, int K) {
  if (n_sims <= 0) return CRL_OK;
  if (K < 1) K = 1;
  int n_steps = n_sims;
  if (K > 1) {
    LaunchScope ls(e, KC_TREE);
    k_wave_begin<<<div_up(e->G, TREE_BLOCK), TREE_BLOCK, 0, e->stream>>>(e->P, n_sims);
    CRL_CUDA(cudaGetLastError());
    n_steps = (n_sims + K - 1) / K;
  }
  for (;;) {
    int rc = tree_run_steps(e, n_steps, K);
    if (rc != CRL_OK) return rc;
    if (K <= 1) return finish_simulations(e);
    int left = 0;
    rc = wave_left(e, &left);
    if (rc != CRL_OK) return rc;
    if (left <= 0) return CRL_OK;
    n_steps = (left + K - 1) / K;
  }
}

int tree_run_steps(crl_engine_impl* e, int n_sims, int K) {
  const bool graph_ok = e->use_graph && !e->profiling && e->stream != nullptr;
  if (!graph_ok) {
    for (int s = 0; s < n_sims; ++s) {
      int rc = one_step(e, K);
      if (rc != CRL_OK) return rc;
    }
    return CRL_OK;
  }
  // the kernel parameters (pool pointers included) are baked into the captured graph; with evaluation reuse the tree
  // pools swap roles at every move, so there is one graph per parity
  const int par = e->tree_parity & 1;
  // the evaluator configuration of every slot the search routes rows to
  auto slot_key = [e](int k) {
    return (unsigned long long)e->eval_kind[k] + 2ull * (unsigned long long)e->eval_bits[k] +
           64ull * (e->eval_seed[k] * 0x9E3779B97F4A7C15ull) + (net_fp8(e, k) ? 0x4000000000000000ull : 0ull);
  };
  unsigned long long key = 1ull + slot_key(0) + 0x100000000ull * (unsigned long long)K +
                           (e->reuse ? 0x8000000000000000ull : 0ull) +
                           0x9E3779B97F4A7C15ull * (unsigned long long)(e->row_bound > 0 ? e->row_bound : 0);
  if (e->search_slots > 1) key = (key * 0x100000001B3ull) ^ (slot_key(1) * 0xC2B2AE3D27D4EB4Full) ^ 0x2000000000000000ull;
  if (e->sim_graph[par] == nullptr || e->sim_graph_key[par] != key) {
    if (e->sim_graph[par]) {
      cudaGraphExecDestroy(e->sim_graph[par]);
      e->sim_graph[par] = nullptr;
    }
    // run one simulation eagerly first: it creates whatever host-side state the launchers cache (tensor maps)
    int rc = one_step(e, K);
    if (rc != CRL_OK) return rc;
    --n_sims;
    const long long l0 = e->launches;
    long long cls0[KC_COUNT];
    for (int i = 0; i < KC_COUNT; ++i) cls0[i] = e->prof_launches[i];
    cudaGraph_t graph = nullptr;
    CRL_CUDA(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
    e->capturing = true;
    rc = one_step(e, K);
    e->capturing = false;
    cudaError_t ce = cudaStreamEndCapture(e->stream, &graph);
    e->sim_graph_launches = e->launches - l0;
    e->launches = l0;
    for (int i = 0; i < KC_COUNT; ++i) e->prof_launches[i] = cls0[i];
    if (rc != CRL_OK) {
      if (graph) cudaGraphDestroy(graph);
      return rc;
    }
    if (ce != cudaSuccess) return cuda_fail(ce, "cudaStreamEndCapture");
    ce = cudaGraphInstantiate(&e->sim_graph[par], graph, 0);
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) return cuda_fail(ce, "cudaGraphInstantiate");
    e->sim_graph_key[par] = key;
  }
  for (int s = 0; s < n_sims; ++s) CRL_CUDA(cudaGraphLaunch(e->sim_graph[par], e->stream));
  e->launches += (long long)n_sims * e->sim_graph_launches;
  return CRL_OK;
}

int tree_policy_move(crl_engine_impl* e, const u8* mask_dev, u16* picks_dev) {
  CRL_CUDA(cudaMemsetAsync(picks_dev, 0xFF, sizeof(u16) * e->G, e->stream));
  const int bound = e->row_bound;
  e->row_bound = 0;                               // the bound is a promise about the NEXT search, not about this call
  int rc = tree_begin_move(e, mask_dev, false);   // root_init + evaluation of the current positions
  e->row_bound = bound;
  if (rc != CRL_OK) return rc;
  LaunchScope ls(e, KC_TREE);
  k_policy_move<<<dim3(div_up(e->G, TREE_BLOCK), e->search_slots), TREE_BLOCK, 0, e->stream>>>(e->P, e->pview,
                                                                                               e->d_label_of, picks_dev);
  CRL_CUDA(cudaGetLastError());
  return CRL_OK;
}

int tree_commit(crl_engine_impl* e, const int* pick_dev, u16* out_moves_dev, int apply) {
  LaunchScope ls(e, KC_GAME);
  k_commit<<<div_up(e->G, TREE_BLOCK), TREE_BLOCK, 0, e->stream>>>(e->P, pick_dev, out_moves_dev, apply);
  CRL_CUDA(cudaGetLastError());
  return CRL_OK;
}

}  // namespace crl
