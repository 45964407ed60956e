"""bf16 against fp8 evaluation (DESIGN.md section 3.1) in one process, the two modes alternating, on one GPU:
  - encode + network positions/s at 4,096 positions,
  - device-resident simulations/s at 4,096 lanes x 200 simulations (one move search per lane),
  - one game x 100 simulations (seconds per search),
  - agreement of the most-visited root child between the two modes on the 4,096-lane search, whose lanes start from
    seeded random openings of 0..40 plies (the same in both modes).
The card's name, power limit and SM clock are read in the same call.  Writes profiles/r03_fp8_bench.json (or --out).
The network is model.random_pack(0, perturb_bn=True); fp8 is calibrated on model.calibration_planes(n=256)."""
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


def sync():
    torch.cuda.synchronize()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--lanes", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_fp8_bench.json"))
    a = ap.parse_args()
    pack = model.random_pack(0, perturb_bn=True)
    G = a.lanes
    wide = Engine(max_games=G, max_nodes=a.sims + 1, avg_moves=96)
    wide.load_weights(pack)
    amax = wide.calibrate(model.calibration_planes(wide, n=256))
    wide.set_evaluator(EVAL_NET)
    one = Engine(max_games=1, max_nodes=101, avg_moves=96)
    one.set_evaluator(EVAL_NET)
    start = np.tile(B.record_from_fen(), (G, 1))
    boards = wide.boards_to_device(start)
    # seeded random openings, one per lane, played through the engine's move generator
    rng = np.random.default_rng(0)
    wide.games_set(start)
    target = rng.integers(0, 41, G)
    for ply in range(40):
        legal, cnt = wide.games_legal()
        _, _, done = wide.games_get()
        mv = np.full(G, B.MOVE_NONE, dtype=np.uint16)
        go = (target > ply) & (cnt > 0) & (done == B.RESULT_NONE)
        mv[go] = legal[np.arange(G), (rng.random(G) * np.maximum(cnt, 1)).astype(np.int64)][go]
        wide.games_play(mv)
    openings = Engine.pack_move_lists(wide.games_moves(np.arange(G)))
    res = {m: {"encode_net_pos_s": [], "sims_s": [], "one_game_100_sims_s": []} for m in ("bf16", "fp8")}
    best = {}

    def load(eng, mode):
        eng.load_weights(pack, precision=mode, calibration=amax if mode == "fp8" else None)

    for rep in range(a.reps + 1):              # rep 0 warms every shape up and is not recorded
        for mode in ("bf16", "fp8"):
            load(wide, mode)
            load(one, mode)
            sync()
            t = time.perf_counter()
            for _ in range(10):
                planes = wide.encode(boards)
                wide.net_forward(planes)
            sync()
            enc = 10 * G / (time.perf_counter() - t)
            wide.games_set(start, openings)
            wide.mcts_begin_move()
            sync()
            t = time.perf_counter()
            wide.mcts_simulate(a.sims)
            sync()
            sims = G * a.sims / (time.perf_counter() - t)
            st = wide.root_stats(want=("visits",))
            best[mode] = np.where(st["n_children"] > 0, np.argmax(st["visits"], axis=1), -1)
            one.games_set(start[:1])
            one.mcts_begin_move()
            sync()
            t = time.perf_counter()
            one.mcts_simulate(100)
            sync()
            single = time.perf_counter() - t
            if rep:
                res[mode]["encode_net_pos_s"].append(enc)
                res[mode]["sims_s"].append(sims)
                res[mode]["one_game_100_sims_s"].append(single)
    out = {"card": card(), "lanes": G, "sims": a.sims, "reps": a.reps, "calibration_amax": [float(x) for x in amax],
           "root_best_child_agreement": float(np.mean((best["bf16"] == best["fp8"])[best["bf16"] >= 0])),
           "lanes_with_children": int(np.sum(best["bf16"] >= 0))}
    for mode in res:
        out[mode] = {k: {"median": statistics.median(v), "all": v} for k, v in res[mode].items()}
    out["speedup_fp8_over_bf16"] = {k: out["fp8"][k]["median"] / out["bf16"][k]["median"]
                                    for k in ("encode_net_pos_s", "sims_s")}
    out["speedup_fp8_over_bf16"]["one_game_100_sims_s"] = (out["bf16"]["one_game_100_sims_s"]["median"]
                                                           / out["fp8"]["one_game_100_sims_s"]["median"])
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("card", "root_best_child_agreement", "speedup_fp8_over_bf16")}))
    wide.close()
    one.close()


if __name__ == "__main__":
    main()
