"""Generating training games on one GPU (chessrl_b200/gen_data.py, DESIGN.md 3.7), in one process:
  - speed, results, how games ended and the fraction of distinct games of gen_data.generate_games, 4,096 games on 4,096
    lanes, at the defaults (depth 3, qdepth 4) and at depth 2 / qdepth 2, both with the default margin and pick plies;
  - one end-to-end run: the default run's games are written as a DatasetGame file, `supervised` trains a fresh model
    on it for one epoch, and `arena` plays 128 games at 100 simulations of the trained network against the fresh one
    (the same random initialisation) and against alphabeta:1:0.
The card's name, power limit and SM clock are read in the same call.  Writes profiles/r06_gen_data_bench.json (or --out);
the dataset and the weights go to a temporary directory."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from chessrl_b200 import arena, gen_data, supervised   # noqa: E402
from chessrl_b200.selfplay import get_model_path       # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def generate(games, depth, qdepth, seed):
    params = dict(depth=depth, qdepth=qdepth, margin=gen_data.MARGIN, pick_plies=gen_data.PICK_PLIES,
                  max_plies=gen_data.MAX_PLIES, seed=seed)
    out, summary = gen_data.generate_games(games, lanes=min(games, gen_data.LANES), **params)
    row = {"params": dict(params, games=games, lanes=min(games, gen_data.LANES)), "summary": summary}
    print(json.dumps(row), flush=True)
    return out, row


def match(a, b, games, sims, seed):
    t0 = time.time()
    _, summary = arena.play_match(a, b, games=games, sims=sims, lanes=games, opening_plies=4, max_plies=300, seed=seed)
    summary["wall_s"] = round(time.time() - t0, 2)
    print(json.dumps({"b": b, "summary": summary}), flush=True)
    return summary


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--match-games", type=int, default=128)
    ap.add_argument("--sims", type=int, default=100)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_gen_data_bench.json"))
    args = ap.parse_args()
    res = {"card": card(), "generate": []}
    games, row = generate(args.games, gen_data.DEPTH, gen_data.QDEPTH, args.seed)
    res["generate"].append(row)
    res["generate"].append(generate(args.games, 2, 2, args.seed)[1])
    if not args.no_e2e:
        with tempfile.TemporaryDirectory() as tmp:
            data = os.path.join(tmp, "games.json")
            t0 = time.time()
            gen_data.to_dataset(games).save(data)
            e2e = {"dataset": {"games": len(games), "write_s": round(time.time() - t0, 1)}}
            fresh_dir, trained_dir = os.path.join(tmp, "fresh"), os.path.join(tmp, "trained")
            os.makedirs(fresh_dir)
            os.makedirs(trained_dir)
            from chessrl_b200.agent import Agent
            Agent(color=True).save(get_model_path(fresh_dir))         # the fresh model, saved before training
            Agent(color=True).save(get_model_path(trained_dir))       # (the same initialisation)
            t0 = time.time()
            supervised.train(trained_dir, data, epochs=1, batch_size=8)
            e2e["supervised"] = {"epochs": 1, "batch_size": 8, "wall_s": round(time.time() - t0, 1)}
            trained = get_model_path(trained_dir)
            e2e["trained_vs_fresh"] = match(trained, get_model_path(fresh_dir), args.match_games, args.sims, 21)
            e2e["trained_vs_alphabeta_1_0"] = match(trained, "alphabeta:1:0", args.match_games, args.sims, 22)
            res["end_to_end"] = e2e
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
