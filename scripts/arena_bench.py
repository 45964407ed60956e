"""Cost of a two-network search (DESIGN.md section 3.5) in one process, on one GPU:
  - device-resident simulations/s at 4,096 lanes x 200 simulations (one move search per lane, CUDA graph), with every
    lane on one network (players all slot 0) and with the lanes split half and half between two networks (slot 0 and
    slot 1 each searching for 2,048 lanes), the two configurations alternating on the same engine and positions;
  - the same searches once more with crl_profile on (eager launches, per-launch CUDA events): time and launches by
    kernel class.
Lanes start from seeded random openings of 0..40 plies.  The networks are model.random_pack(0 / 1, perturb_bn=True).
The card's name, power limit and SM clock are read in the same call.  Writes profiles/r04_arena_bench.json (or --out)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np      # noqa: E402
import torch            # noqa: E402

from chessrl_b200 import boards as B, model   # noqa: E402
from chessrl_b200._lib import EVAL_NET        # noqa: E402
from chessrl_b200.engine import Engine        # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def openings(e, seed, max_plies=40):
    G = e.max_games
    rng = np.random.default_rng(seed)
    e.games_set(np.tile(B.record_from_fen(), (G, 1)))
    target = rng.integers(0, max_plies + 1, G)
    for ply in range(max_plies):
        legal, cnt = e.games_legal()
        mv = np.full(G, B.MOVE_NONE, dtype=np.uint16)
        go = (target > ply) & (cnt > 0)
        pick = (rng.random(G) * np.maximum(cnt, 1)).astype(np.int64)
        mv[go] = legal[np.arange(G), pick][go]
        e.games_play(mv)


def search_seconds(e, sims):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e.mcts_begin_move()
    e.mcts_simulate(sims)
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lanes", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_arena_bench.json"))
    args = ap.parse_args()
    G, S = args.lanes, args.sims
    e = Engine(max_games=G, max_nodes=S + 1, avg_moves=96)
    for slot in (0, 1):
        e.load_weights(model.random_pack(slot, perturb_bn=True), slot=slot)
        e.set_evaluator(EVAL_NET, slot=slot)
    openings(e, seed=7)
    half = np.zeros(G, dtype=np.uint8)
    half[G // 2:] = 1
    configs = {"one_network": (np.zeros(G, np.uint8), np.zeros(G, np.uint8)), "two_networks": (half, half)}
    times = {k: [] for k in configs}
    for name, (w, b) in configs.items():          # warm-up: graph capture of both configurations
        e.games_set_players(w, b)
        search_seconds(e, S)
    for _ in range(args.reps):
        for name, (w, b) in configs.items():
            e.games_set_players(w, b)
            times[name].append(search_seconds(e, S))
    res = {"card": card(), "lanes": G, "sims": S, "reps": args.reps, "timing": "host clock around begin_move + "
           "simulate, synchronised; CUDA graph replay; same engine, positions and weights", "configs": {}}
    for name in configs:
        med = statistics.median(times[name])
        res["configs"][name] = {"search_s": times[name], "median_s": med, "sims_per_s": G * S / med}
    res["two_over_one"] = res["configs"]["two_networks"]["median_s"] / res["configs"]["one_network"]["median_s"]
    # kernel-class breakdown: one profiled search per configuration (eager launches, events around every launch)
    for name, (w, b) in configs.items():
        e.games_set_players(w, b)
        e.profile(True)
        search_seconds(e, S)
        prof = e.profile_read()
        e.profile(False)
        res["configs"][name]["profile_ms"] = {k: round(v["ms"], 3) for k, v in prof.items()}
        res["configs"][name]["profile_launches"] = {k: v["launches"] for k, v in prof.items()}
    e.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "configs"}))
    for name, c in res["configs"].items():
        print(name, "median %.3f s, %.0f sims/s" % (c["median_s"], c["sims_per_s"]), c["profile_ms"])


if __name__ == "__main__":
    main()
