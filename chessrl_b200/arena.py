"""arena: search-vs-search matches between two networks, on one engine.

The engine holds network A in slot 0 and network B in slot 1 (include/chessrl_b200.h crl_net_select_slot).  Every lane
plays one game; the side to move searches with its own network -- root, predicted replies and leaves
(crl_games_set_players_host) -- so one lockstep step advances every running game by one ply, for about the cost of a
self-play step (DESIGN.md 3.5).  Openings come in pairs: each is played once with A as white and once with B as white.

Either side may instead be the fixed-depth alpha-beta opponent (AlphaBetaPlayer, DESIGN.md 3.6): a yardstick of fixed
strength that needs no weights.  Its moves come from Engine.games_ab_move on the same lanes.

    python -m chessrl_b200.arena A B --games N [--lanes L] [--sims S] [--threads K] [--precision-a bf16|fp8]
        [--precision-b bf16|fp8] [--opening-plies P | --openings FILE] [--max-plies M] [--seed X] [--out match.json]

A and B are weights files (.h5) or model directories (their newest model-<n>.h5); they may be the same file with
different precisions, which measures what fp8 evaluation costs in playing strength.  `alphabeta[:D[:Q[:r]]]` in place
of either names the alpha-beta opponent at depth D and quiescence depth Q (default alphabeta:3:4); a trailing `:r` has it
score repeated positions inside its search as draws (DESIGN.md 3.6, off by default).
"""

from __future__ import annotations

import argparse
import json
import math
import os
import random
import time

import numpy as np

from . import boards as B
from ._lib import EVAL_HASH, EVAL_NET
from .lockstep import SMALL_BATCH_ROWS, pick_moves

Z95 = 1.959963984540054          # two-sided 95 % quantile of the standard normal distribution


class HashPlayer:
    """The deterministic test evaluator as a player (crl_set_evaluator(CRL_EVAL_HASH, seed, policy_bits)): a search
    opponent that needs no weights, and the same evaluator as the oracle's hash_evaluator(seed, policy_bits)."""

    def __init__(self, seed, policy_bits=24):
        self.seed = int(seed)
        self.policy_bits = int(policy_bits)


AB_DEPTH, AB_QDEPTH = 3, 4     # the alpha-beta opponent's defaults (DESIGN.md 3.6: cost and ladder)


class AlphaBetaPlayer:
    """The fixed-depth alpha-beta opponent (include/chessrl_b200.h crl_games_ab_move_host): material and position
    evaluation, `depth` full-width plies (1..5), then up to `qdepth` plies of captures and queen promotions (0..8).
    Deterministic: the same position gives the same move.  It searches on the lanes' own positions and needs no network
    slot.  repetitions: a position inside the search that repeats an earlier one of its reversible run, in the game or
    on the search path, scores 0 (crl_games_ab_search_host CRL_AB_REPETITIONS); the move then depends on the game too."""

    def __init__(self, depth=AB_DEPTH, qdepth=AB_QDEPTH, repetitions=False):
        self.depth = int(depth)
        self.qdepth = int(qdepth)
        self.repetitions = bool(repetitions)
        if not (1 <= self.depth <= 5 and 0 <= self.qdepth <= 8):
            raise ValueError("alpha-beta depth 1..5 and qdepth 0..8, not %d / %d" % (self.depth, self.qdepth))

    SPEC = "alphabeta"

    @classmethod
    def parse(cls, spec):
        """'alphabeta', 'alphabeta:D', 'alphabeta:D:Q' or 'alphabeta:D:Q:r' -> AlphaBetaPlayer; None for any other
        string."""
        parts = spec.split(":")
        if parts[0] != cls.SPEC or len(parts) > 4:
            return None
        try:
            if len(parts) == 4 and parts[3] != "r":
                raise ValueError
            nums = [int(p) for p in parts[1:3]]
        except ValueError:
            raise ValueError("alpha-beta player: 'alphabeta[:D[:Q[:r]]]', not %r" % (spec,))
        return cls(*nums, repetitions=len(parts) == 4)

    def __str__(self):
        return "%s:%d:%d%s" % (self.SPEC, self.depth, self.qdepth, ":r" if self.repetitions else "")

    __repr__ = __str__

    def moves(self, engine, mask):
        """This player's moves in the lanes of `mask` (MOVE_NONE elsewhere)."""
        kw = {"repetitions": True} if self.repetitions else {}
        return engine.games_ab_move(self.depth, self.qdepth, mask=mask.astype(np.uint8), **kw)[0]


def _as_player(x):
    """A ChessModel, an Agent, a weights path, a model directory, 'alphabeta[:D[:Q[:r]]]', a HashPlayer or an
    AlphaBetaPlayer -> HashPlayer, AlphaBetaPlayer or ChessModel."""
    from .model import ChessModel
    from .selfplay import get_model_path
    if isinstance(x, (HashPlayer, AlphaBetaPlayer, ChessModel)):
        return x
    if hasattr(x, "model") and isinstance(x.model, ChessModel):      # an Agent
        return x.model
    if isinstance(x, str):
        ab = AlphaBetaPlayer.parse(x)
        if ab is not None:
            return ab
        return ChessModel(weights=get_model_path(x) if os.path.isdir(x) else x)
    raise ValueError("a ChessModel, an Agent, a weights path, a model directory, a HashPlayer or an AlphaBetaPlayer is "
                     "needed, not %r" % (x,))


def _configure(engine, player, slot, precision):
    if isinstance(player, HashPlayer):
        engine.set_evaluator(EVAL_HASH, player.seed, player.policy_bits, slot=slot)
    else:
        engine.load_weights(player.weights, precision=precision, slot=slot)
        engine.set_evaluator(EVAL_NET, slot=slot)


def elo_of_score(s):
    """Elo difference of an expected score s: -400 log10(1/s - 1); -inf / +inf at 0 / 1."""
    if s <= 0:
        return -math.inf
    if s >= 1:
        return math.inf
    return -400.0 * math.log10(1.0 / s - 1.0)


def elo_interval(wins, losses, draws, z=Z95):
    """(score, elo, elo_low, elo_high) of wins / losses / draws: the trinomial normal approximation of the mean score,
    score +- z * sqrt(var / n), mapped through elo_of_score.  A bound at score 0 or 1 is infinite."""
    n = wins + losses + draws
    if n == 0:
        return 0.5, 0.0, -math.inf, math.inf
    s = (wins + 0.5 * draws) / n
    var = (wins * (1.0 - s) ** 2 + losses * s ** 2 + draws * (0.5 - s) ** 2) / n
    half = z * math.sqrt(var / n)
    return s, elo_of_score(s), elo_of_score(s - half), elo_of_score(s + half)


def summarize(games):
    """played, A wins, B wins, draws, unfinished, A's score and the Elo difference A - B with its 95 % interval.
    Unfinished games (max_plies reached) count as draws in the score and the interval."""
    a_wins = b_wins = draws = unfinished = 0
    for g in games:
        r = g["result"]
        if r is None:
            unfinished += 1
        elif r == 0:
            draws += 1
        elif (r == 1) == g["a_white"]:
            a_wins += 1
        else:
            b_wins += 1
    score, elo, lo, hi = elo_interval(a_wins, b_wins, draws + unfinished)
    return {"played": len(games), "a_wins": a_wins, "b_wins": b_wins, "draws": draws, "unfinished": unfinished,
            "score": score, "elo": elo, "elo_low": lo, "elo_high": hi}


def play_match(a, b, games, sims, lanes=None, inflight=1, precision_a="bf16", precision_b="bf16", openings=None,
               opening_plies=4, max_plies=512, seed=None, device=None, engine=None):
    """`games` games of A against B, each side searching its own moves with `sims` simulations (`inflight` in flight
    per game, the reference's threads) and playing the most visited root child; an AlphaBetaPlayer side plays the move
    of its fixed-depth search instead.  Game 2i and 2i+1 start from opening i,
    with A as white in the first and B as white in the second.  Openings are `openings` (a list of UCI move lists,
    used in turn) or `opening_plies` seeded random legal plies.  A game that reaches `max_plies` plies stops unfinished.
    `engine`: an engine to play on (default: a new Engine with `lanes` lanes on `device`).

    Returns (per-game list in game order, summary).  A game is {'opening', 'a_white', 'moves' (UCI, the opening
    included), 'result' (white's point of view; None if unfinished)}."""
    games = int(games)
    if games <= 0:
        raise ValueError("games must be positive")
    pa, pb = _as_player(a), _as_player(b)
    ab = [p if isinstance(p, AlphaBetaPlayer) else None for p in (pa, pb)]
    searchers = [k for k, p in enumerate((pa, pb)) if ab[k] is None]       # the sides that search with MCTS
    if len(searchers) == 2 and isinstance(pa, HashPlayer) != isinstance(pb, HashPlayer):
        raise ValueError("a match is between two networks or two hash players (one search cannot mix them)")
    # network slot of each searching side: A 0 and B 1 when both search; a single searching side takes slot 0, so that
    # the search runs on one slot, as with one network
    slot_of = {k: (k if len(searchers) == 2 else 0) for k in searchers}
    if lanes is None:
        lanes = games if engine is None else min(games, engine.max_games)
    lanes = max(1, min(games, int(lanes)))
    own = engine is None
    if own:
        from .engine import Engine
        from .selfplay import edge_slots_per_node
        nodes = int(sims) + 1 if searchers else 2
        engine = Engine(max_games=lanes, max_nodes=nodes, device=device, max_inflight=int(inflight),
                        avg_moves=edge_slots_per_node(lanes, nodes, device))
    e = engine
    if e.max_games < lanes:
        raise ValueError("the engine has %d lanes, %d asked for" % (e.max_games, lanes))
    base = random.Random(seed).getrandbits(64)
    fixed = [list(o) for o in openings] if openings else None
    n_open = (games + 1) // 2
    opening_of = [None] * n_open                   # UCI lists, fixed at the first game of each pair
    out = [None] * games
    try:
        for k in searchers:                        # (a load replays on lane 0: configure before the games are set)
            _configure(e, (pa, pb)[k], slot_of[k], (precision_a, precision_b)[k])
        e.set_reuse(False)
        e.games_set(np.tile(B.record_from_fen(), (e.max_games, 1)))
        lane_game = np.full(e.max_games, -1, dtype=np.int64)
        next_game = 0

        def start(lanes_):
            """The next games in these lanes: players, start position, opening."""
            nonlocal next_game
            fresh = []
            for lane in lanes_:
                j = next_game
                next_game += 1
                lane_game[lane] = j
                a_white = j % 2 == 0
                if len(searchers) == 2:
                    e.games_set_players([0 if a_white else 1], [1 if a_white else 0], first=int(lane))
                elif searchers:
                    e.games_set_players([0], [0], first=int(lane))
                i = j // 2
                if opening_of[i] is None and fixed is not None:
                    opening_of[i] = fixed[i % len(fixed)]
                if opening_of[i] is not None:
                    e.games_set(B.record_from_fen()[None, :], [[B.uci_to_move(m) for m in opening_of[i]]], first=int(lane))
                else:
                    fresh.append(int(lane))
            if fresh:                              # seeded random legal plies, drawn per opening
                e.games_restart(fresh)
                rngs = {lane: random.Random("%d:%d" % (base, lane_game[lane] // 2)) for lane in fresh}
                for _ in range(int(opening_plies)):
                    legal, cnt = e.games_legal(0, e.max_games)
                    mv = np.full(e.max_games, B.MOVE_NONE, dtype=np.uint16)
                    for lane in fresh:
                        if cnt[lane] > 0:
                            mv[lane] = legal[lane, rngs[lane].randrange(int(cnt[lane]))]
                    e.games_play(mv)
                for lane, moves in zip(fresh, e.games_moves(fresh)):
                    opening_of[lane_game[lane] // 2] = [B.move_to_uci(m) for m in moves]

        first = list(range(min(lanes, games)))
        start(first)
        live = np.zeros(e.max_games, dtype=bool)
        live[first] = True
        if not live.all():
            e.games_set_active(live.astype(np.uint8))
        rec, plies, results = e.games_get(0, e.max_games)
        while True:
            over = live & ((results != B.RESULT_NONE) | (plies >= max_plies))
            if over.any():                         # harvest, then refill or park
                done = np.nonzero(over)[0]
                for lane, moves in zip(done, e.games_moves(done)):
                    j = int(lane_game[lane])
                    res = None if results[lane] == B.RESULT_NONE else int(results[lane])
                    out[j] = {"opening": list(opening_of[j // 2]), "a_white": j % 2 == 0,
                              "moves": [B.move_to_uci(m) for m in moves], "result": res}
                again = [int(l) for l in done[:max(0, games - next_game)]]
                parked = [int(l) for l in done[len(again):]]
                if again:
                    start(again)
                if parked:
                    live[parked] = False
                    e.games_set_active(live.astype(np.uint8))
                if not live.any():
                    break
                rec, plies, results = e.games_get(0, e.max_games)
                continue                           # a refilled opening may already have ended the game
            # one ply of every running game: the side to move searches with its network and plays its most visited
            # child, or plays its alpha-beta move
            white = (rec[:, 8] & np.uint64(1)).astype(bool)
            a_to_move = white == (lane_game % 2 == 0)
            ab_turn = [live & (a_to_move if k == 0 else ~a_to_move) if ab[k] is not None else None for k in (0, 1)]
            searching = live.copy()
            for t in ab_turn:
                if t is not None:
                    searching &= ~t
            mv = np.full(e.max_games, B.MOVE_NONE, dtype=np.uint16)
            if searching.any():
                parked = not np.array_equal(searching, live)
                if parked:                         # the alpha-beta side's lanes sit out the search
                    e.games_set_active(searching.astype(np.uint8))
                n_run = int(searching.sum())
                small = SMALL_BATCH_ROWS // max(1, int(inflight))
                e.set_row_bound(small if 0 < n_run <= small < e.max_games else 0)
                e.mcts_begin_move()
                e.mcts_simulate(int(sims), int(inflight))
                st = e.root_stats(want=("visits", "moves"))
                picks = pick_moves(st["visits"], st["n_children"], st["root_visits"], plies, searching, noise=False)
                rows = np.nonzero(picks >= 0)[0]
                mv[rows] = st["moves"][rows, picks[rows]]
                if parked:                         # resumed before the play: games_play skips parked lanes
                    e.games_set_active(live.astype(np.uint8))
            for k in (0, 1):
                if ab_turn[k] is not None and ab_turn[k].any():
                    mv = np.where(ab_turn[k], ab[k].moves(e, ab_turn[k]), mv)
            e.games_play(mv)
            rec, plies, results = e.games_get(0, e.max_games)
    finally:
        if own:
            e.close()
    return out, summarize(out)


def _read_openings(path):
    with open(path) as f:
        return [line.split() for line in f if line.strip() and not line.lstrip().startswith("#")]


def _label(arg, precision):
    """How a CLI player is reported: 'alphabeta:D:Q[:r]' (its full parameters) or 'path (precision)'."""
    ab = AlphaBetaPlayer.parse(arg)
    return str(ab) if ab is not None else "%s (%s)" % (arg, precision)


def main(argv=None):
    ap = argparse.ArgumentParser(description="Plays a search-vs-search match between two networks, or a network and the "
                                             "alpha-beta opponent, and prints the score and the Elo difference A - B with "
                                             "its 95 % interval.")
    ap.add_argument("a", help="weights file (.h5) or model directory of player A, or alphabeta[:D[:Q[:r]]]")
    ap.add_argument("b", help="weights file (.h5) or model directory of player B (may be A's), or alphabeta[:D[:Q[:r]]]")
    ap.add_argument("--games", type=int, required=True)
    ap.add_argument("--lanes", type=int, default=None, help="concurrent games (default: one per game)")
    ap.add_argument("--sims", type=int, default=100, help="simulations per move")
    ap.add_argument("--threads", type=int, default=1, help="simulations in flight per game (wave mode for > 1)")
    ap.add_argument("--precision-a", choices=("bf16", "fp8"), default="bf16")
    ap.add_argument("--precision-b", choices=("bf16", "fp8"), default="bf16")
    src = ap.add_mutually_exclusive_group()
    src.add_argument("--opening-plies", type=int, default=4, help="seeded random legal plies per opening")
    src.add_argument("--openings", default=None, help="file with one opening per line, space-separated UCI moves")
    ap.add_argument("--max-plies", type=int, default=512)
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--out", default=None, help="write the games and the summary as JSON")
    args = ap.parse_args(argv)
    t0 = time.time()
    games, summary = play_match(args.a, args.b, args.games, args.sims, lanes=args.lanes, inflight=args.threads,
                                precision_a=args.precision_a, precision_b=args.precision_b,
                                openings=_read_openings(args.openings) if args.openings else None,
                                opening_plies=args.opening_plies, max_plies=args.max_plies, seed=args.seed)
    summary["wall_s"] = round(time.time() - t0, 3)
    label_a, label_b = _label(args.a, args.precision_a), _label(args.b, args.precision_b)
    print("A %s vs B %s: %d games, +%d -%d =%d (%d unfinished), score %.4f, Elo %+.1f [%+.1f, %+.1f], %.1f s"
          % (label_a, label_b, summary["played"], summary["a_wins"], summary["b_wins"], summary["draws"],
             summary["unfinished"], summary["score"], summary["elo"], summary["elo_low"], summary["elo_high"],
             summary["wall_s"]))
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"a": args.a, "b": args.b, "player_a": label_a, "player_b": label_b,
                       "precision_a": args.precision_a, "precision_b": args.precision_b,
                       "sims": args.sims, "threads": args.threads, "summary": summary, "games": games}, f, indent=1)
    return summary


if __name__ == "__main__":
    main()
