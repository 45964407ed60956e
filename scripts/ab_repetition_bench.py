"""Repetitions in the alpha-beta search (crl_games_ab_search_host CRL_AB_REPETITIONS, DESIGN.md 3.6) on one GPU, in one
process:
  - call cost: 4,096 lanes at (2,2) and (3,4), plain and with repetitions alternating, the median of --calls calls each,
    with node counts.  The lanes hold plain gen_data games (depth 2 / qdepth 2, seed 1) cut at staggered plies, so every
    root has its real history;
  - gen_data at the defaults, 4,096 games, seed 1, plain and with repetitions: speed, results, how games ended, the
    "other draw" games split into insufficient material and fivefold repetition (read from the final position), and
    the fraction of distinct games;
  - a match of alphabeta:3:4:r against alphabeta:3:4, 256 games from 4-ply openings with both colours, at most 300
    plies.
The card's name, power limit and SM clock are read in the same call.  Writes profiles/r07_ab_repetition_bench.json (or
--out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

from chessrl_b200 import arena, gen_data             # noqa: E402
from chessrl_b200 import boards as B                 # noqa: E402
from chessrl_b200.engine import CRL_AB_REPETITIONS, Engine   # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def call_cost(calls):
    games, _ = gen_data.generate_games(4096, depth=2, qdepth=2, seed=1)
    eng = Engine(max_games=4096, max_nodes=2, avg_moves=64)
    try:
        # lane j: game j cut at ply (37 j mod its length) -- staggered, every root with its game before it
        cut = [[B.uci_to_move(m) for m in g["moves"][:(37 * j) % max(1, len(g["moves"]))]] for j, g in enumerate(games)]
        eng.games_set(np.tile(B.record_from_fen(), (4096, 1)), cut)
        _, plies, res = eng.games_get(0, 4096)
        out = {"lanes": 4096, "searched": int((res == B.RESULT_NONE).sum()), "mean_ply": round(float(plies.mean()), 1),
               "shapes": []}
        for d, q in ((2, 2), (3, 4)):
            row = {"depth": d, "qdepth": q, "plain_ms": [], "rep_ms": []}
            for flags in (0, CRL_AB_REPETITIONS):                         # warm-up, scratch allocation
                eng.games_ab_search(d, q, flags)
            for _ in range(calls):
                for flags, key in ((0, "plain_ms"), (CRL_AB_REPETITIONS, "rep_ms")):
                    t0 = time.perf_counter()
                    r = eng.games_ab_search(d, q, flags)                   # returns after a stream synchronise
                    row[key].append(round(1e3 * (time.perf_counter() - t0), 2))
                    row["plain_nodes" if flags == 0 else "rep_nodes"] = int(r[2].sum())
                    row["plain_moves" if flags == 0 else "rep_moves"] = r[0]
            changed = int((row.pop("plain_moves") != row.pop("rep_moves")).sum())
            row.update({"plain_median_ms": float(np.median(row["plain_ms"])),
                        "rep_median_ms": float(np.median(row["rep_ms"])), "moves_changed": changed})
            row["rep_over_plain"] = round(row["rep_median_ms"] / row["plain_median_ms"], 3)
            print(json.dumps(row), flush=True)
            out["shapes"].append(row)
        return out
    finally:
        eng.close()


def draw_split(games):
    """The "other draw" games by their final position: insufficient material, else fivefold repetition."""
    from ab_oracle import chess                      # the oracle's python-chess restatement
    split = {"insufficient_material": 0, "fivefold": 0, "neither": 0}
    for g in games:
        if g["end"] != "other_draw":
            continue
        b = chess.Board()
        for m in g["moves"]:
            b.push(chess.Move.from_uci(m))
        if b.is_insufficient_material():
            split["insufficient_material"] += 1
        elif b.is_fivefold_repetition():
            split["fivefold"] += 1
        else:
            split["neither"] += 1
    return split


def generate(games, repetitions):
    params = dict(depth=gen_data.DEPTH, qdepth=gen_data.QDEPTH, margin=gen_data.MARGIN,
                  pick_plies=gen_data.PICK_PLIES, max_plies=gen_data.MAX_PLIES, seed=1, repetitions=repetitions)
    out, summary = gen_data.generate_games(games, lanes=min(games, gen_data.LANES), **params)
    row = {"params": dict(params, games=games), "summary": summary, "other_draw_split": draw_split(out)}
    print(json.dumps(row), flush=True)
    return row


def match(games):
    t0 = time.time()
    a, b = arena.AlphaBetaPlayer(3, 4, repetitions=True), arena.AlphaBetaPlayer(3, 4)
    _, summary = arena.play_match(a, b, games=games, sims=1, lanes=games, opening_plies=4, max_plies=300, seed=5)
    summary["wall_s"] = round(time.time() - t0, 2)
    row = {"a": str(a), "b": str(b), "summary": summary}
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=7)
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--match-games", type=int, default=256)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_ab_repetition_bench.json"))
    args = ap.parse_args()
    res = {"card": card(), "call_cost": call_cost(args.calls)}
    res["gen_data"] = [generate(args.games, False), generate(args.games, True)]
    res["match"] = match(args.match_games)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
