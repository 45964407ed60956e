"""Cost and strength of the fixed-depth alpha-beta opponent (DESIGN.md section 3.6), in one process, on one GPU:
  - cost: milliseconds per Engine.games_ab_move call, positions visited and positions/s, for depth 1..4 and quiescence
    depth 0 and 4, at 1, 64, 512 and 4,096 lanes, on seeded midgame positions (random playouts of 16..40 plies, the same
    positions for every depth); every shape is called once untimed first, then timed over whole calls that end in a
    device synchronise;
  - a ladder of matches (arena.play_match, 128 games each, openings of 4 seeded random plies, each played with both
    colours): alpha-beta at depth d against depth d + 1 for d = 1, 2, 3, and a random-init test network
    (model.random_pack(0, perturb_bn=True), not trained weights) searching 100 simulations against depths 1..3.
The card's name, power limit and SM clock are read in the same call.  Writes profiles/r05_alphabeta_bench.json (or --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np      # noqa: E402
import torch            # noqa: E402

from chessrl_b200 import arena, boards as B, model   # noqa: E402
from chessrl_b200.engine import Engine               # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def midgames(e, seed, lo=16, hi=40):
    """Seeded random playouts of lo..hi plies in every lane (a lane whose game ends early keeps its final position)."""
    G = e.max_games
    rng = np.random.default_rng(seed)
    e.games_set(np.tile(B.record_from_fen(), (G, 1)))
    target = rng.integers(lo, hi + 1, G)
    for ply in range(hi):
        legal, cnt = e.games_legal()
        mv = np.full(G, B.MOVE_NONE, dtype=np.uint16)
        go = (target > ply) & (cnt > 0)
        pick = (rng.random(G) * np.maximum(cnt, 1)).astype(np.int64)
        mv[go] = legal[np.arange(G), pick][go]
        e.games_play(mv)


def cost(lanes_list, depths, qdepths, min_s):
    rows = []
    for lanes in lanes_list:
        e = Engine(max_games=lanes, max_nodes=2, avg_moves=64)
        midgames(e, seed=lanes)
        _, _, res = e.games_get()
        running = int((res == B.RESULT_NONE).sum())
        for d in depths:
            for q in qdepths:
                e.games_ab_move(d, q)                                   # untimed first call (scratch, modules)
                times, nodes = [], 0
                while sum(times) < min_s and len(times) < 20:
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    _, _, n = e.games_ab_move(d, q)                     # (returns after a stream synchronise)
                    times.append(time.perf_counter() - t0)
                    nodes = int(n.sum())
                ms = 1e3 * float(np.median(times))
                rows.append({"lanes": lanes, "running": running, "depth": d, "qdepth": q, "ms_per_call": round(ms, 3),
                             "calls": len(times), "nodes": nodes, "nodes_per_s": round(nodes / (ms * 1e-3))})
                print(json.dumps(rows[-1]), flush=True)
        e.close()
    return rows


def match(a, b, games, sims, seed):
    t0 = time.time()
    out, summary = arena.play_match(a, b, games=games, sims=sims, lanes=games, opening_plies=4, max_plies=300,
                                    seed=seed)
    summary["wall_s"] = round(time.time() - t0, 2)
    summary["mean_plies"] = round(float(np.mean([len(g["moves"]) for g in out])), 1)
    row = {"a": str(a) if isinstance(a, arena.AlphaBetaPlayer) else "random-init network, %d simulations" % sims,
           "b": str(b), "summary": summary}
    print(json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lanes", type=int, nargs="*", default=[1, 64, 512, 4096])
    ap.add_argument("--depths", type=int, nargs="*", default=[1, 2, 3, 4])
    ap.add_argument("--qdepths", type=int, nargs="*", default=[0, 4])
    ap.add_argument("--min-seconds", type=float, default=1.0, help="timed calls per shape: until this long (<= 20 calls)")
    ap.add_argument("--games", type=int, default=128)
    ap.add_argument("--sims", type=int, default=100)
    ap.add_argument("--no-ladder", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_alphabeta_bench.json"))
    args = ap.parse_args()
    out = {"card": card(), "cost": cost(args.lanes, args.depths, args.qdepths, args.min_seconds), "ladder": []}
    if not args.no_ladder:
        for d in (1, 2, 3):
            out["ladder"].append(match(arena.AlphaBetaPlayer(d, 4), arena.AlphaBetaPlayer(d + 1, 4), args.games, 1, d))
        net = model.ChessModel()
        net.weights = model.random_pack(0, perturb_bn=True)
        for d in (1, 2, 3):
            out["ladder"].append(match(net, arena.AlphaBetaPlayer(d, 4), args.games, args.sims, 10 + d))
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
