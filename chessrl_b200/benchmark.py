"""benchmark: the reference's policy-only evaluation loop (benchmark.py:59-143) on lockstep lanes.

The reference plays N games of its agent -- moving by the argmax of the legal-masked policy,
`Agent.best_move(game, real_game=True)` (benchmark.py:88-90, agent.py:39-43) -- against a Stockfish process wrapped
in GameStockfish, and tallies played / won / drawn.  Stockfish is out of scope here (no binary, SURVEY.md 8(f)-4);
the loop itself is kept: the same agent side, the same tally, and an opponent that is a seeded uniformly random mover,
a second network (also policy argmax) or the fixed-depth alpha-beta opponent (arena.AlphaBetaPlayer, DESIGN.md 3.6),
the fixed yardstick that stands in for Stockfish.  `workers` concurrent games become `workers` lockstep lanes of one
engine; every ply of every running game is one batched network evaluation or one batched alpha-beta call.

    python -m chessrl_b200.benchmark modeldir [--games 10] [--workers 2]
        [--opponent random|path/to/weights.h5|alphabeta[:D[:Q[:r]]]]
"""

from __future__ import annotations

import argparse
import os
import random

import numpy as np

from . import boards as B
from ._lib import EVAL_NET
from .arena import AlphaBetaPlayer
from .lib.logger import Logger
from .model import ChessModel
from .selfplay import get_model_path


def _as_model(x):
    if x is None or isinstance(x, ChessModel):
        return x
    if hasattr(x, "model") and isinstance(x.model, ChessModel):      # an Agent
        return x.model
    if isinstance(x, str):
        return ChessModel(weights=x)
    raise ValueError("a ChessModel, an Agent or a path to weights is needed")


def play_policy_games(agent, opponent="random", games=10, lanes=None, seed=None, device=None, max_plies=2000):
    """`games` games, agent (policy argmax) versus `opponent` ("random"; a ChessModel / Agent / weights path that
    also moves by policy argmax; or an AlphaBetaPlayer / 'alphabeta[:D[:Q[:r]]]', searched on the agent's engine).  The
    agent's colour is drawn per game like benchmark.py:70.
    Returns one dict per game in game order: {'color', 'result' (white point of view, None if capped), 'moves'}."""
    from .engine import Engine
    agent_model = _as_model(agent)
    ab = opponent if isinstance(opponent, AlphaBetaPlayer) else (
        AlphaBetaPlayer.parse(opponent) if isinstance(opponent, str) else None)
    opp_model = None if ab is not None or (isinstance(opponent, str) and opponent == "random") else _as_model(opponent)
    rng = random.Random(seed)
    lanes = max(1, min(games, games if lanes is None else int(lanes)))
    a = Engine(max_games=lanes, max_nodes=2, avg_moves=218, device=device)
    a.load_weights(agent_model.weights)
    a.set_evaluator(EVAL_NET)
    b = None
    if opp_model is not None:
        b = Engine(max_games=lanes, max_nodes=2, avg_moves=218, device=device)
        b.load_weights(opp_model.weights)
        b.set_evaluator(EVAL_NET)
    colors = [rng.random() <= .5 for _ in range(games)]
    lane_game = np.arange(lanes)
    lane_color = np.array([colors[g] for g in lane_game], dtype=bool)
    live = np.ones(lanes, dtype=bool)
    next_game = lanes
    out = [None] * games
    start = np.tile(B.record_from_fen(), (lanes, 1))
    for e in (a, b):
        if e is not None:
            e.games_set(start)
    none = np.full(lanes, B.MOVE_NONE, dtype=np.uint16)
    try:
        while live.any():
            rec, plies, results = a.games_get(0, lanes)
            over = live & ((results != B.RESULT_NONE) | (plies >= max_plies))
            if over.any():
                done = np.nonzero(over)[0]
                for lane, moves in zip(done, a.games_moves(done)):
                    res = None if results[lane] == B.RESULT_NONE else int(results[lane])
                    out[lane_game[lane]] = {"color": bool(lane_color[lane]), "result": res,
                                            "moves": [B.move_to_uci(m) for m in moves]}
                again = [int(l) for l in done[:max(0, games - next_game)]]
                parked = [int(l) for l in done[len(again):]]
                for lane in again:
                    lane_game[lane] = next_game
                    lane_color[lane] = colors[next_game]
                    next_game += 1
                live[parked] = False
                for e in (a, b):
                    if e is not None:
                        e.games_restart(again)
                        if parked:
                            e.games_set_active(live.astype(np.uint8))
                if not live.any():
                    break
                rec, plies, results = a.games_get(0, lanes)
            white_to_move = (rec[:, 8] & np.uint64(1)).astype(bool)
            agent_turn = live & (white_to_move == lane_color)
            opp_turn = live & ~agent_turn
            if agent_turn.any():
                picks = a.policy_move(mask=agent_turn.astype(np.uint8))          # evaluates and plays on engine a
                if b is not None:
                    b.games_play(np.where(agent_turn, picks, none))
            if opp_turn.any():
                if b is not None:
                    picks = b.policy_move(mask=opp_turn.astype(np.uint8))
                    a.games_play(np.where(opp_turn, picks, none))
                elif ab is not None:
                    a.games_play(ab.moves(a, opp_turn))
                else:
                    legal, cnt = a.games_legal(0, lanes)
                    mv = none.copy()
                    for lane in np.nonzero(opp_turn)[0]:                        # lane order: reproducible for a seed
                        mv[lane] = legal[lane, rng.randrange(int(cnt[lane]))]
                    a.games_play(mv)
    finally:
        a.close()
        if b is not None:
            b.close()
    return out


def benchmark(model_dir, workers=1, games=10, stockfish_depth=10, log=False, opponent="random", seed=None):
    """Plays `games` games and returns dict(played, won, drawn) like the reference (benchmark.py:103-143).
    `workers` = concurrent games (lockstep lanes here, processes there).  `stockfish_depth` is accepted for signature
    compatibility only: the opponent is `opponent` (see play_policy_games), not Stockfish; the depth-selected fixed
    opponent here is opponent="alphabeta:D[:Q]"."""
    logger = Logger.get_instance()
    if log:
        logger.info("Setting up %d concurrent games." % workers)
    model_path = get_model_path(model_dir)
    if not os.path.exists(model_path):
        logger.error("Model not found. Exiting.")                    # benchmark.py:78-82
        return None
    results = play_policy_games(model_path, opponent=opponent, games=games, lanes=workers, seed=seed)
    won = [1 if (x['color'] is True and x['result'] == 1) or (x['color'] is False and x['result'] == -1) else 0
           for x in results]
    if log:
        print("##################### SUMMARY ###################")
        print("Games played: %d" % games)
        print("Games won: %d" % sum(won))
        print("Games drawn: %d" % len([x for x in results if x['result'] == 0]))
        print("#################################################")
    return dict(played=games, won=sum(won), drawn=len([x for x in results if x['result'] == 0]))


def main(argv=None):
    ap = argparse.ArgumentParser(description="Plays policy-only games with the newest model of a directory and prints the tally.")
    ap.add_argument("model_dir", metavar="modeldir")
    ap.add_argument("--games", type=int, default=10)
    ap.add_argument("--workers", type=int, default=2, help="concurrent games (lockstep lanes)")
    ap.add_argument("--opponent", default="random",
                    help="'random', a path to the opponent's weights, or alphabeta[:D[:Q[:r]]] (fixed-depth alpha-beta)")
    ap.add_argument("--seed", type=int, default=None)
    args = ap.parse_args(argv)
    print(benchmark(args.model_dir, workers=args.workers, games=args.games, log=True, opponent=args.opponent, seed=args.seed))


if __name__ == "__main__":
    main()
