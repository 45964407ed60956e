"""gen_data: supervised training games from the fixed-depth alpha-beta player, on the GPU (DESIGN.md 3.7).

The reference starts a network from engine games (gen_data_stockfish.py, then supervised.py on the JSON).  Here both
sides of every game are the alpha-beta player of DESIGN.md 3.6, with a seeded near-best root pick so that games differ:
while fewer than `pick_plies` plies have been played, a side may play any root move scored within `margin` centipawns of
the best one (never when the best score is a mate), chosen by a per-game salt.  Every ply is still a move the search
rates as near-best, so every ply is a fair policy target.  Game j's salt is splitmix64(base + j), with base drawn from
the seed as in arena, so the games depend only on the seed and the parameters -- not on the lanes or the number of GPUs.
With --repetitions the search scores a position that repeats an earlier one of its reversible run as a draw (DESIGN.md
3.6), so a side that is ahead stops repeating moves; it is off by default.  With --scores every game also records the
search's root scores of each ply (DESIGN.md 3.8): the exact value of every legal move, the data of soft policy and score
value targets (supervised --targets search); the games themselves are the same.

    python -m chessrl_b200.gen_data OUT.json --games N [--lanes L] [--depth 3] [--qdepth 4] [--margin CP]
        [--pick-plies P] [--max-plies M] [--seed S] [--repetitions] [--scores]

OUT.json is the DatasetGame format that `supervised` reads; games are appended to what the file holds, in game order.
Under torchrun the games are sharded by rank and gathered to rank 0, which writes the file.
"""

from __future__ import annotations

import argparse
import hashlib
import json
import os
import random
import time

import numpy as np

from . import boards as B

DEPTH, QDEPTH = 3, 4          # the alpha-beta player's defaults (arena.AB_DEPTH / AB_QDEPTH)
# Defaults of the pick (DESIGN.md 3.7): at depth 3 / qdepth 4 they made 4,096 games from the start position 100 %
# distinct (measured on a B200 at 1,000 W, seed 1).
MARGIN, PICK_PLIES = 20, 16
MAX_PLIES = 512
LANES = 4096
ENDS = ("mate", "stalemate", "fifty_moves", "other_draw", "unfinished")
_M64 = (1 << 64) - 1


def splitmix64(x):
    """The splitmix64 finaliser (chessrl_b200/csrc/chess_core.cuh mix64)."""
    z = (x + 0x9E3779B97F4A7C15) & _M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


def game_salts(seed, first, n):
    """The salts of games first..first+n-1: splitmix64(base + j), base = random.Random(seed).getrandbits(64)."""
    base = random.Random(seed).getrandbits(64)
    return np.array([splitmix64((base + j) & _M64) for j in range(first, first + n)], dtype=np.uint64)


def game_end(record, result, n_legal):
    """How a finished game ended, from its final record, its result and its legal move count, in the order
    game_result (chess_core.cuh) tests them: the fifty-move claim, mate or stalemate, then the other draws
    (insufficient material, fivefold repetition).  result None: unfinished."""
    if result is None:
        return "unfinished"
    if B.meta_fields(record[8])["halfmove"] >= 100 and n_legal > 0:
        return "fifty_moves"
    if n_legal == 0:
        return "mate" if result != 0 else "stalemate"
    return "other_draw"


def _key(moves):
    return hashlib.sha1(" ".join(moves).encode()).hexdigest()


def tally(games):
    """Per-game facts the summary needs (small enough to gather across ranks)."""
    return [{"plies": len(g["moves"]), "result": g["result"], "end": g["end"], "key": _key(g["moves"])} for g in games]


def summarize(facts, wall_s):
    """games, plies, mean plies, wall time, games/s, positions/s, the result tally, how games ended and the fraction
    of distinct games (distinct move lists over games)."""
    n = len(facts)
    plies = sum(f["plies"] for f in facts)
    res = [f["result"] for f in facts]
    return {"games": n, "plies": plies, "mean_plies": round(plies / max(1, n), 2), "wall_s": round(wall_s, 3),
            "games_per_s": round(n / max(wall_s, 1e-9), 3), "positions_per_s": round(plies / max(wall_s, 1e-9), 1),
            "white_wins": res.count(1), "black_wins": res.count(-1), "draws": res.count(0),
            "unfinished": res.count(None), "ends": {e: sum(f["end"] == e for f in facts) for e in ENDS},
            "distinct_fraction": round(len({f["key"] for f in facts}) / max(1, n), 6)}


def generate_games(n_games, lanes=None, depth=DEPTH, qdepth=QDEPTH, margin=MARGIN, pick_plies=PICK_PLIES,
                   max_plies=MAX_PLIES, seed=None, first=0, device=None, engine=None, repetitions=False, scores=False):
    """Games first..first+n_games-1 of the alpha-beta player against itself with the seeded near-best pick, `lanes` at
    a time on one engine (default: a new Engine on `device` with no tree).  A game that reaches `max_plies` plies stops
    unfinished.  Every step makes one Engine.games_ab_pick call for all running lanes -- both colours -- and plays the
    picks with one games_play; finished games are harvested, and their lanes start the next game or are parked.
    repetitions: the search scores repeated positions 0 (Engine.games_ab_pick repetitions=True).
    scores: after every pick call one Engine.games_ab_root_scores call records the root scores of the ply each lane is
    about to play; a game then also has 'scores', one int32 array per ply (the scores of its legal moves in generation
    order).  The per-step work is a few array operations over all lanes; the arrays are split per game at the end.

    Returns (games in game order, summary).  A game is {'moves' (UCI), 'result' (white's point of view, None if
    unfinished), 'player_color' (game index even), 'end' (one of ENDS)}."""
    n_games = int(n_games)
    if n_games <= 0:
        raise ValueError("n_games must be positive")
    lanes = max(1, min(n_games, int(lanes or min(n_games, LANES))))
    own = engine is None
    if own:
        from .engine import Engine
        engine = Engine(max_games=lanes, max_nodes=2, avg_moves=218, device=device)
    e = engine
    if e.max_games < lanes:
        raise ValueError("the engine has %d lanes, %d asked for" % (e.max_games, lanes))
    salts = game_salts(seed, first, n_games)
    kw = {"repetitions": True} if repetitions else {}
    out = [None] * n_games
    kept = []                  # with scores: per pick call (game, ply, count, the counts' scores concatenated)
    t0 = time.perf_counter()
    try:
        e.games_set(np.tile(B.record_from_fen(), (e.max_games, 1)))
        lane_game = np.full(e.max_games, -1, dtype=np.int64)
        lane_game[:lanes] = np.arange(lanes)
        salt = np.zeros(e.max_games, dtype=np.uint64)
        salt[:lanes] = salts[:lanes]
        live = np.zeros(e.max_games, dtype=bool)
        live[:lanes] = True
        if not live.all():
            e.games_set_active(live.astype(np.uint8))
        next_game = lanes
        while True:
            rec, plies, results = e.games_get(0, e.max_games)
            over = live & ((results != B.RESULT_NONE) | (plies >= max_plies))
            if over.any():                         # harvest, then refill or park
                done = np.nonzero(over)[0]
                _, n_legal = e.games_legal(0, e.max_games)
                for lane, moves in zip(done, e.games_moves(done)):
                    j = int(lane_game[lane])
                    res = None if results[lane] == B.RESULT_NONE else int(results[lane])
                    out[j] = {"moves": [B.move_to_uci(m) for m in moves], "result": res,
                              "player_color": (first + j) % 2 == 0, "end": game_end(rec[lane], res, int(n_legal[lane]))}
                again = done[:max(0, n_games - next_game)]
                parked = done[len(again):]
                if len(again):
                    lane_game[again] = next_game + np.arange(len(again))
                    salt[again] = salts[lane_game[again]]
                    next_game += len(again)
                    e.games_restart(again)
                if len(parked):
                    live[parked] = False
                    e.games_set_active(live.astype(np.uint8))
                if not live.any():
                    break
                continue
            picks = e.games_ab_pick(depth, qdepth, margin, pick_plies, salt, **kw)[0]
            if scores:
                sc, cnt = e.games_ab_root_scores()
                lanes_s = np.nonzero(cnt > 0)[0]
                c = cnt[lanes_s]
                kept.append((lane_game[lanes_s], plies[lanes_s], c, sc[lanes_s][_COLS[None, :] < c[:, None]]))
            e.games_play(picks)
    finally:
        if own:
            e.close()
    if scores:
        _attach_scores(out, kept)
    return out, summarize(tally(out), time.perf_counter() - t0)


_COLS = np.arange(B.MAX_MOVES)


def _attach_scores(games, kept):
    """games[j]['scores'] = the recorded score arrays of game j, one per ply in ply order."""
    game, ply, cnt, flat = (np.concatenate(part) for part in zip(*kept))     # (every run makes a pick call)
    start = np.zeros(len(cnt) + 1, dtype=np.int64)
    start[1:] = np.cumsum(cnt)
    order = np.lexsort((ply, game))
    bounds = np.searchsorted(game[order], np.arange(len(games) + 1))
    for j, g in enumerate(games):
        rows = order[bounds[j]:bounds[j + 1]]
        assert np.array_equal(ply[rows], np.arange(len(g["moves"]))), j
        g["scores"] = [flat[start[r]:start[r + 1]] for r in rows]


def to_dataset(games):
    """The games as a DatasetGame (each replayed once on the device, as selfplay.LockstepRun.dataset does); recorded
    scores become Game.search_scores."""
    from .dataset import DatasetGame
    from .game import Game
    data = DatasetGame()
    for g in games:
        gm = Game(player_color=g["player_color"])
        gm._sync(extra=g["moves"])
        if "scores" in g:
            gm.search_scores = [s.tolist() for s in g["scores"]]
        data.append(gm)
    return data


def main(argv=None):
    ap = argparse.ArgumentParser(description="Generates supervised training games of the alpha-beta player against "
                                             "itself on the GPU and appends them to a DatasetGame JSON file.")
    ap.add_argument("out", help="JSON file to append the games to (the format supervised reads)")
    ap.add_argument("--games", type=int, required=True)
    ap.add_argument("--lanes", type=int, default=None, help="concurrent games per GPU (default: min(games, %d))" % LANES)
    ap.add_argument("--depth", type=int, default=DEPTH, help="full-width plies of the search (1..5)")
    ap.add_argument("--qdepth", type=int, default=QDEPTH, help="quiescence plies (0..8)")
    ap.add_argument("--margin", type=int, default=MARGIN,
                    help="centipawns below the best root score a picked move may be (0: always the best move)")
    ap.add_argument("--pick-plies", type=int, default=PICK_PLIES, help="plies of each game that use the margin")
    ap.add_argument("--max-plies", type=int, default=MAX_PLIES, help="a game stops here, unfinished (result null)")
    ap.add_argument("--seed", type=int, default=None, help="default: drawn at random and printed")
    ap.add_argument("--repetitions", action="store_true",
                    help="the search scores a position that repeats an earlier one of its reversible run as a draw")
    ap.add_argument("--scores", action="store_true",
                    help="record the search's score of every legal move at every ply (training targets, DESIGN.md 3.8)")
    args = ap.parse_args(argv)
    if args.games <= 0 or args.margin < 0 or args.pick_plies < 0 or args.max_plies <= 0:
        ap.error("--games and --max-plies must be positive, --margin and --pick-plies non-negative")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    import torch
    if torch.cuda.is_available():
        torch.cuda.set_device(local_rank)
    seed = args.seed if args.seed is not None else random.SystemRandom().getrandbits(63)
    lo, hi = 0, args.games
    if world > 1:
        import torch.distributed as dist
        from . import sharding
        sharding.init()
        box = [seed]
        dist.broadcast_object_list(box, src=0)          # one seed for every rank when none is given
        seed = box[0]
        lo, hi = sharding.shard_range(args.games)
    games, wall = [], 0.0
    if hi > lo:
        games, s = generate_games(hi - lo, lanes=args.lanes, depth=args.depth, qdepth=args.qdepth, margin=args.margin,
                                  pick_plies=args.pick_plies, max_plies=args.max_plies, seed=seed, first=lo,
                                  device=local_rank, repetitions=args.repetitions, scores=args.scores)
        wall = s["wall_s"]
    facts = tally(games)
    data = to_dataset(games)
    if world > 1:
        gathered = [None] * world
        scores = [g.search_scores for g in data.games] if args.scores else None
        dist.all_gather_object(gathered, (facts, wall, scores))
        facts = [f for part, _, _ in gathered for f in part]
        wall = max(w for _, w, _ in gathered)              # the ranks generate concurrently
        data = sharding.gather_games(data)
        if args.scores and rank == 0:                      # gather_games keeps rank order, then game order
            lists = [s for _, _, part in gathered for s in part]
            if len(lists) != len(data.games):
                raise RuntimeError("gathered %d games but %d score lists" % (len(data.games), len(lists)))
            for g, s in zip(data.games, lists):
                g.search_scores = s
    summary = summarize(facts, wall)
    summary.update({"seed": seed, "depth": args.depth, "qdepth": args.qdepth, "margin": args.margin,
                    "pick_plies": args.pick_plies, "max_plies": args.max_plies, "repetitions": args.repetitions,
                    "ranks": world})
    if args.scores:
        summary["scores"] = True
    if rank == 0:
        data.save(args.out)
        s = summary
        print("%d games, %d plies (mean %.1f) in %.1f s: %.2f games/s, %.0f positions/s"
              % (s["games"], s["plies"], s["mean_plies"], s["wall_s"], s["games_per_s"], s["positions_per_s"]))
        print("white wins %d, black wins %d, draws %d, unfinished %d; ended by %s; distinct games %.2f %%"
              % (s["white_wins"], s["black_wins"], s["draws"], s["unfinished"],
                 ", ".join("%s %d" % kv for kv in s["ends"].items()), 100.0 * s["distinct_fraction"]))
        print(json.dumps(summary))
    if world > 1:
        sharding.shutdown()
    return summary


if __name__ == "__main__":
    main()
