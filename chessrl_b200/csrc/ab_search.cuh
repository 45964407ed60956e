// ab_search.cuh -- the fixed-depth alpha-beta opponent (DESIGN.md 3.6): a hand-written static evaluation and a per-thread
// negamax alpha-beta with an explicit stack, on the bitboard rules of chess_core.cuh.
//
// The value it returns is defined independently of move ordering and pruning, so any correct alpha-beta returns the same
// bits as a plain minimax over the same tree (oracle/ab_oracle.py restates the definition):
//
//   s(p)     centipawns for the side to move: its pieces minus the opponent's (table in ab_eval_side)
//   T(p, h)  game_result(b, n_legal, in_check, 0): mate -(AB_MATE - h) for the side to move; stalemate, insufficient
//            material and the fifty-move claim 0.  h = plies from the search root; repetitions are not tracked.
//            With repetitions on (R, crl_games_ab_search_host CRL_AB_REPETITIONS): a position h >= 1 plies below the
//            root that repeats an earlier position of its reversible run (on the search path, the root included, or in
//            the game before the root) scores 0 before anything else, counts as one visited position and generates no
//            moves -- python-chess's board.is_repetition(2) on the game's moves followed by the path.
//   V(p,d,h) = T(p,h) if terminal;  Q(p,q,h) if d = 0;  max over legal m of -V(p.m, d-1, h+1)
//   Q(p,k,h) = T(p,h) if terminal;  s(p) if k = 0;  max over legal m of -Q(p.m, k-1, h+1) if in check (no stand-pat);
//              else max(s(p), max over m in C(p) of -Q(p.m, k-1, h+1)),  C(p) = legal captures (en passant included)
//              plus promotions to a queen
//   root     the first legal move, in generation order, with the largest -V(root.m, D-1, 1); the score is that value.
//
// Within a node captures come first by MVV-LVA, then the other moves in generation order; the ordering changes how many
// positions are visited, never the value.  Every function is CRL_HD: the g++ build in tests/hostsim/ab_hostsim.cpp runs
// the same code as the kernels in kernels_ab.cu, node counts included.
#pragma once
#include "chess_core.cuh"

namespace crl {

enum { AB_MAX_DEPTH = 5, AB_MAX_QDEPTH = 8 };
enum { AB_MAX_PLY = AB_MAX_DEPTH + AB_MAX_QDEPTH };   // plies below the root one search can hold moves for
enum { AB_MATE = 32000, AB_INF = 32767 };

// ---- static evaluation -----------------------------------------------------------------------------------------------
// Per piece of colour c on a square with rank r seen from c (7 - rank for black), file f and
// cd = max(|2f - 7|, |2r - 7|) / 2 (0 on d4/e4/d5/e5 .. 3 on the rim):
//   pawn 100 + 5 (r - 1)          knight 310 + 10 (3 - cd)      bishop 330 + 5 (3 - cd), +30 once for >= 2 bishops
//   rook 500, +20 on r = 6        queen 900 + 2 (3 - cd)
//   king -10 min(r, 2) while the other side has a queen, 5 (3 - cd) otherwise
// Evaluated set-wise: 3 - cd is the number of the three nested squares below (inside the rim, the inner 4x4, the
// centre) that hold the piece, and a sum of ranks is a sum of popcounts of "rank >= k" masks.
static const u64 AB_NOT_RIM = 0x007E7E7E7E7E7E00ULL;
static const u64 AB_INNER = 0x00003C3C3C3C0000ULL;
static const u64 AB_CENTER = 0x0000001818000000ULL;

CRL_HD int ab_centrality(u64 s) { return popc64(s & AB_NOT_RIM) + popc64(s & AB_INNER) + popc64(s & AB_CENTER); }
// sum of the ranks (0..7, rank 1 = 0) of the squares of s
CRL_HD int ab_rank_sum(u64 s) {
  int t = 0;
#pragma unroll
  for (int k = 1; k < 8; ++k) t += popc64(s >> (8 * k));
  return t;
}

CRL_HD int ab_eval_side(const Board& b, int white) {
  const u64 us = b.bb[white ? OCC_W : OCC_B], them = b.bb[white ? OCC_B : OCC_W];
  const u64 p = b.bb[PAWN] & us, n = b.bb[KNIGHT] & us, bi = b.bb[BISHOP] & us, r = b.bb[ROOK] & us,
            q = b.bb[QUEEN] & us, k = b.bb[KING] & us;
  const int np = popc64(p), nb = popc64(bi);
  const int pawn_ranks = white ? ab_rank_sum(p) : 7 * np - ab_rank_sum(p);   // sum of r over our pawns
  int v = 100 * np + 5 * (pawn_ranks - np);
  v += 310 * popc64(n) + 10 * ab_centrality(n);
  v += 330 * nb + 5 * ab_centrality(bi) + (nb >= 2 ? 30 : 0);
  v += 500 * popc64(r) + 20 * popc64(r & (white ? (RANK_1 << 48) : (RANK_1 << 8)));
  v += 900 * popc64(q) + 2 * ab_centrality(q);
  if (b.bb[QUEEN] & them) {
    const u64 back = white ? RANK_1 : RANK_8, second = white ? (RANK_1 << 8) : (RANK_1 << 48);
    v -= 10 * (popc64(k & ~back) + popc64(k & ~back & ~second));          // min(r, 2)
  } else {
    v += 5 * ab_centrality(k);
  }
  return v;
}

// s(p): from the point of view of the side to move
CRL_HD int ab_evaluate(const Board& b) {
  const int white = meta_turn(b.meta);
  return ab_eval_side(b, white) - ab_eval_side(b, !white);
}

// T(p, h) for a position the generator reported n_legal / in_check for; false if the game goes on
CRL_HD bool ab_terminal(const Board& b, int n_legal, int in_check, int h, int* value) {
  const int r = game_result(b, n_legal, in_check, 0);
  if (r == RESULT_NONE) return false;
  *value = (n_legal == 0 && in_check) ? -(AB_MATE - h) : 0;
  return true;
}

// ---- move ordering ----------------------------------------------------------------------------------------------------
// MVV-LVA key of a capture (victim value first, then the cheaper attacker), 0 for a move that captures nothing
CRL_HD int ab_capture_key(const Board& b, u16 mv) {
  const int from = mv_from(mv), to = mv_to(mv);
  const u64 them = b.bb[meta_turn(b.meta) ? OCC_B : OCC_W];
  const int attacker = piece_at(b, from);
  int victim;
  if (them & bit(to)) victim = piece_at(b, to);
  else if (attacker == PAWN && ((from ^ to) & 7)) victim = PAWN;       // en passant: a diagonal pawn move to an empty square
  else return 0;
  return 1 + 8 * victim + (7 - attacker);
}

// Reorders moves[0..n): captures by descending key (ties in generation order), then the other moves in generation order.
// captures_only (quiescence, not in check): keeps C(p) only -- the captures and the non-capturing queen promotions.
// Returns the new count.  keys: scratch of MAX_MOVES words.
CRL_HD int ab_order(const Board& b, u16* moves, int n, bool captures_only, u32* keys) {
  int nc = 0, nq = 0;
  for (int i = 0; i < n; ++i) {
    const u16 m = moves[i];
    const int key = ab_capture_key(b, m);
    if (key) {
      // descending key, then ascending index: insertion sort of (key, 255 - index) words
      const u32 w = ((u32)key << 24) | ((u32)(255 - i) << 16) | m;
      int j = nc++;
      while (j > 0 && keys[j - 1] < w) {
        keys[j] = keys[j - 1];
        --j;
      }
      keys[j] = w;
    } else if (!captures_only || mv_promo(m) == QUEEN) {
      moves[nq++] = m;                                                   // stable compaction of the other moves
    }
  }
  for (int i = nq - 1; i >= 0; --i) moves[nc + i] = moves[i];
  for (int i = 0; i < nc; ++i) moves[i] = (u16)(keys[i] & 0xFFFF);
  return nc + nq;
}

// ---- the search -------------------------------------------------------------------------------------------------------
// One thread's stack: level L holds the position L plies below the searched one.  Every level but the last holds a move
// list; a quiescence leaf (k = 0) only counts its moves.
struct AbStack {
  Board b[AB_MAX_PLY + 1];
  u16 m[AB_MAX_PLY][MAX_MOVES];
  u32 keys[MAX_MOVES];
  int n[AB_MAX_PLY], i[AB_MAX_PLY];
  int alpha[AB_MAX_PLY + 1], beta[AB_MAX_PLY + 1], best[AB_MAX_PLY];
};

// The repetition window of one search with R on (kept apart from AbStack, which the plain search uses as it is).
//   key[L]    transposition key of the position at stack level L, stored for a node that has children a repetition
//             could reach (level L + 4 <= d + q)
//   game[i]   key of the position i plies before the root, i = 0..ngame (game[0]: the root, its key as the game
//             recorded it, en passant included); ngame = min(revlen, ply) of the root record
// A repetition needs the same side to move and a reversible run of at least 4 plies, so a node compares its key with
// the positions 4, 6, .. plies above it, back to its own revlen.  A node whose run is non-empty has no en-passant square,
// so its key is position_key(b, 0) and needs no move generation.
enum { AB_REP_KEYS = 100 };   // game[] entries per lane: a searched root's reversible run is < 100 plies (fifty-move rule)
struct AbPath {
  u64 key[AB_MAX_PLY];
  const u64* game;
  int ngame;
};

// does the node at `level` (h = level + 1 plies below the root, revlen rev >= 4, key `key`) repeat an earlier position?
CRL_HD bool ab_repeats(const AbPath& path, u64 key, int level, int h, int rev) {
  for (int j = 4; j <= rev; j += 2) {
    if (j <= level) {
      if (path.key[level - j] == key) return true;
    } else {
      if (j - h > path.ngame) return false;
      if (path.game[j - h] == key) return true;
    }
  }
  return false;
}

// V(p, d, h0) of st.b[0] (d = 0: Q(p, q, h0)) with a full window; requires d + q <= AB_MAX_PLY.
// *nodes += the positions visited (every position whose legal moves were generated, p included).
// REP: repetitions on, with the window in *path; requires h0 == 1 (st.b[0] is a root child, as in ab_root_child): the
// positions above level 0 are then the root and the game before it, path->game[j - h] in ab_repeats.
template <bool REP = false>
CRL_HD int ab_value(AbStack& st, int d, int q, int h0, unsigned long long* nodes, AbPath* path = nullptr) {
  int level = 0, v = 0;
  bool done = false;                 // v is the value of the node at `level`
  st.alpha[0] = -AB_INF;
  st.beta[0] = AB_INF;
  for (;;) {
    if (!done) {
      // ---- enter the node at `level` ----
      const Board& b = st.b[level];
      const int h = h0 + level;
      const bool qnode = level >= d;
      const int k = qnode ? q - (level - d) : 0;
      *nodes += 1;
      u64 key = 0;
      if constexpr (REP) {
        const int rev = meta_revlen(b.meta);
        if (rev >= 4) {
          key = position_key(b, 0);
          if (ab_repeats(*path, key, level, h, rev)) {
            v = 0;
            done = true;
            continue;
          }
        }
      }
      if (qnode && k == 0) {
        CountSink cs{0};
        const GenInfo gi = generate_legal(b, cs);
        if (!ab_terminal(b, cs.n, gi.in_check, h, &v)) v = ab_evaluate(b);
        done = true;
        continue;
      }
      StoreSink ss{st.m[level], 0};
      const GenInfo gi = generate_legal(b, ss);
      if (ab_terminal(b, ss.n, gi.in_check, h, &v)) {
        done = true;
        continue;
      }
      if constexpr (REP) {
        if (level + 4 <= d + q) path->key[level] = meta_revlen(b.meta) >= 4 ? key : position_key(b, gi.ep_legal);
      }
      int best = -AB_INF;
      const bool stand = qnode && !gi.in_check;
      if (stand) {
        best = ab_evaluate(b);
        if (best >= st.beta[level]) {                                    // stand-pat cut
          v = best;
          done = true;
          continue;
        }
        if (best > st.alpha[level]) st.alpha[level] = best;
      }
      st.n[level] = ab_order(b, st.m[level], ss.n, stand, st.keys);
      st.i[level] = 0;
      st.best[level] = best;
    } else {
      // ---- the node at `level` has value v: back it up ----
      if (level == 0) return v;
      --level;
      const int cv = -v;
      if (cv > st.best[level]) st.best[level] = cv;
      if (cv > st.alpha[level]) st.alpha[level] = cv;
      if (st.alpha[level] >= st.beta[level]) {                          // cut: the node is done
        v = st.best[level];
        continue;
      }
      done = false;
    }
    // ---- the next child of the node at `level` ----
    if (st.i[level] >= st.n[level]) {
      v = st.best[level];                                                // (stand-pat value when no capture is left)
      done = true;
      continue;
    }
    const u16 mv = st.m[level][st.i[level]++];
    st.b[level + 1] = st.b[level];
    make_move(st.b[level + 1], mv);
    st.alpha[level + 1] = -st.beta[level];
    st.beta[level + 1] = -st.alpha[level];
    ++level;
  }
}

// the score of root child `mv` at search depth D: -V(root.mv, D - 1, 1)
template <bool REP = false>
CRL_HD int ab_root_child(AbStack& st, const Board& root, u16 mv, int depth, int qdepth, unsigned long long* nodes,
                         AbPath* path = nullptr) {
  st.b[0] = root;
  make_move(st.b[0], mv);
  return -ab_value<REP>(st, depth - 1, qdepth, 1, nodes, path);
}

CRL_HD bool ab_limits_ok(int depth, int qdepth) {
  return depth >= 1 && depth <= AB_MAX_DEPTH && qdepth >= 0 && qdepth <= AB_MAX_QDEPTH;
}

// ---- the seeded near-best root pick (DESIGN.md 3.7, crl_games_ab_pick_host) -------------------------------------------
// s[0..n), n >= 1: the root children's scores in generation order; best = max s[k]; ply = meta_ply of the root record.
//   the first k with s[k] = best        if margin = 0, ply >= pick_plies or |best| >= AB_MATE - AB_MAX_PLY - 1 (a mate);
//   else C[mix64(salt + ply) mod |C|]   with C = [k : s[k] >= best - margin] in generation order.
// Integer arithmetic only (best - s[k] <= margin cannot overflow: |s[k]| <= AB_INF), so the kernels, the g++ build and
// oracle/ab_oracle.py agree bit for bit.
CRL_HD int ab_pick_index(const int* s, int n, int ply, int margin, int pick_plies, u64 salt) {
  int best = s[0], first = 0;
  for (int k = 1; k < n; ++k)
    if (s[k] > best) {
      best = s[k];
      first = k;
    }
  if (margin == 0 || ply >= pick_plies || best >= AB_MATE - AB_MAX_PLY - 1 || best <= -(AB_MATE - AB_MAX_PLY - 1))
    return first;
  unsigned c = 0;
  for (int k = 0; k < n; ++k) c += best - s[k] <= margin;
  unsigned r = (unsigned)(mix64(salt + (u64)ply) % c);
  for (int k = 0; k < n; ++k)
    if (best - s[k] <= margin && r-- == 0) return k;
  return first;                                                          // (not reached: r < |C|)
}

CRL_HD bool ab_pick_ok(int margin, int pick_plies) { return margin >= 0 && pick_plies >= 0; }

}  // namespace crl
