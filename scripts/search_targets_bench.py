"""Search-score training targets on one GPU (DESIGN.md 3.8), in one process:
  1. gen_data with and without scores: 4,096 games on 4,096 lanes, seed 1, at the defaults (depth 3, qdepth 4) and at
     depth 2 / qdepth 2, the two variants alternated; wall time, positions/s, the time spent in the score export per
     step, the size of the written file, and whether the games are identical;
  2. target building at --bs 8: crl_search_targets on the rows of 8 games against crl_encode of the same rows and the
     fp32 training step, CUDA events over many repetitions;
  3. the end-to-end A/B of DESIGN.md 3.7's protocol on the default games with scores: one epoch, bs 8, fp32, from the
     fresh model (model.random_pack(0)) in three arms -- (a) the played-move targets, (b) search targets with w = 0,
     (c) search targets with the defaults -- then 128 arena games at 100 simulations (4-ply seeded openings, at most 300
     plies) of each arm against the fresh network and against alphabeta:1:0, and of (c) against (a).
The card's name, power limit and SM clock are read in the same call.  Writes profiles/r08_search_targets_bench.json (or
--out).  --stage runs one of the three parts (generate, train, match), passing the dataset and the weights on through
--state, so that each part fits a call of limited length; by default all three run, in a temporary directory."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from chessrl_b200 import arena, gen_data, model, runtime, supervised, training   # noqa: E402
from chessrl_b200.engine import Engine                                         # noqa: E402
from chessrl_b200.selfplay import get_model_path                               # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def emit(row):
    print(json.dumps(row), flush=True)
    return row


def generate(games, depth, qdepth, seed, scores, tmp):
    """One gen_data run on a fresh engine whose score export is timed; the games written to a file."""
    lanes = min(games, gen_data.LANES)
    eng = Engine(max_games=lanes, max_nodes=2, avg_moves=218)
    export = {"calls": 0, "s": 0.0}
    real = eng.games_ab_root_scores

    def timed():
        t0 = time.perf_counter()
        out = real()
        export["s"] += time.perf_counter() - t0
        export["calls"] += 1
        return out
    eng.games_ab_root_scores = timed
    try:
        out, summary = gen_data.generate_games(games, lanes=lanes, depth=depth, qdepth=qdepth, seed=seed, engine=eng,
                                               scores=scores)
    finally:
        eng.close()
    path = os.path.join(tmp, "d%d_q%d_%s.json" % (depth, qdepth, "scores" if scores else "plain"))
    gen_data.to_dataset(out).save(path)
    row = {"depth": depth, "qdepth": qdepth, "scores": scores, "games": games, "lanes": lanes, "seed": seed,
           "summary": summary, "file_bytes": os.path.getsize(path),
           "export_calls": export["calls"], "export_ms_per_call": round(1e3 * export["s"] / max(1, export["calls"]), 3),
           "export_share_of_wall": round(export["s"] / summary["wall_s"], 4)}
    emit({"generate": row})
    return out, row, path


def same_games(a, b):
    return all(x["moves"] == y["moves"] and x["result"] == y["result"] for x, y in zip(a, b)) and len(a) == len(b)


def events(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def target_timing(data_path, bs=8, reps=200):
    from chessrl_b200.dataset import DatasetGame
    ds = DatasetGame()
    ds.load(data_path)
    games = ds.games[:bs]
    eng = runtime.scalar_engine()
    boards, hists, hlens, _, _, _ = training.game_samples(games, [False] * bs)
    n = boards.shape[0]
    bt = eng.boards_to_device(boards)
    ht = torch.from_numpy(np.ascontiguousarray(hists.transpose(1, 2, 0)).view(np.int64)).to(eng.device)
    lt = torch.from_numpy(hlens).to(eng.device)
    cnt = np.array([len(s) for g in games for s in g.search_scores], dtype=np.int32)
    off = np.zeros(n + 1, dtype=np.int32)
    off[1:] = np.cumsum(cnt)
    flat = torch.tensor([v for g in games for s in g.search_scores for v in s], dtype=torch.int32, device=eng.device)
    ot = torch.from_numpy(off).to(eng.device)
    t_targets = events(lambda: eng.search_targets(bt, flat, ot, 50.0), reps)
    t_encode = events(lambda: eng.encode(bt, ht, lt), reps)
    planes, pol, val, probs = training.encode_search_games(games, [False] * bs, training.SearchTargets())
    params = [torch.tensor(w, device=eng.device) for w in model.random_pack(0)]
    tr = []
    for i in training.trainable_indices():
        params[i].requires_grad_(True)
        tr.append(params[i])
    opt = training.KerasAdam(tr)
    with training.arithmetic("fp32"):
        t_step = events(lambda: training.train_step(params, opt, planes, pol, val, probs), 10)
        t_step_played = events(lambda: training.train_step(params, opt, planes, pol, val), 10)
    t0 = time.perf_counter()
    for _ in range(20):
        training.encode_search_games(games, [False] * bs, training.SearchTargets())
    torch.cuda.synchronize()
    t_batch = (time.perf_counter() - t0) / 20 * 1e3
    return emit({"target_timing": {"batch_games": bs, "rows": int(n), "search_targets_ms": round(t_targets, 4),
                                   "encode_ms": round(t_encode, 4), "train_step_fp32_search_ms": round(t_step, 2),
                                   "train_step_fp32_played_ms": round(t_step_played, 2),
                                   "encode_search_games_host_ms": round(t_batch, 2)}})["target_timing"]


def match(a, b, games, sims, seed):
    t0 = time.time()
    _, summary = arena.play_match(a, b, games=games, sims=sims, lanes=games, opening_plies=4, max_plies=300, seed=seed)
    summary["wall_s"] = round(time.time() - t0, 2)
    return summary


def last_val(model_dir):
    log = [json.loads(line) for line in open(os.path.join(model_dir, "train_log.jsonl"))]
    return [r for r in log if "val_loss" in r][-1]


ARMS = {"a_played": dict(targets="played"),
        "b_search_w0": dict(targets="search", temperature=50.0, value_weight=0.0),
        "c_search_default": dict(targets="search", temperature=50.0, value_weight=0.5)}


def stage_generate(args, res, state):
    with tempfile.TemporaryDirectory() as tmp:
        runs = {}
        for depth, qdepth in ((gen_data.DEPTH, gen_data.QDEPTH), (2, 2)):
            for scores in (False, True):
                out, row, path = generate(args.games, depth, qdepth, args.seed, scores, tmp)
                res["generate"].append(row)
                runs[(depth, qdepth, scores)] = (out, path)
            res["generate"].append(emit({"identical_games": {"depth": depth, "qdepth": qdepth, "identical": same_games(
                runs[(depth, qdepth, False)][0], runs[(depth, qdepth, True)][0])}}))
        data = runs[(gen_data.DEPTH, gen_data.QDEPTH, True)][1]
        res["target_timing"] = target_timing(data)
        shutil.copy(data, os.path.join(state, "games.json"))


def stage_train(args, res, state):
    from chessrl_b200.agent import Agent
    res["arms"] = {}
    for name, kw in ARMS.items():
        d = os.path.join(state, name)
        os.makedirs(d, exist_ok=True)
        Agent(color=True).save(get_model_path(d))                 # model.random_pack(0)
        t0 = time.time()
        supervised.train(d, os.path.join(state, "games.json"), epochs=1, batch_size=8, **kw)
        res["arms"][name] = emit({"arm": name, "options": kw, "train_wall_s": round(time.time() - t0, 1),
                                  "validation": last_val(d)})


def stage_match(args, res, state):
    from chessrl_b200.agent import Agent
    fresh_dir = os.path.join(state, "fresh")
    os.makedirs(fresh_dir, exist_ok=True)
    Agent(color=True).save(get_model_path(fresh_dir))             # the same initialisation, untrained
    res["matches"] = {}
    for name in ARMS:
        w = get_model_path(os.path.join(state, name))
        res["matches"][name + "_vs_fresh"] = emit({name + "_vs_fresh": match(
            w, get_model_path(fresh_dir), args.match_games, args.sims, 21)})[name + "_vs_fresh"]
        res["matches"][name + "_vs_alphabeta_1_0"] = emit({name + "_vs_alphabeta_1_0": match(
            w, "alphabeta:1:0", args.match_games, args.sims, 22)})[name + "_vs_alphabeta_1_0"]
    res["matches"]["c_vs_a"] = emit({"c_vs_a": match(get_model_path(os.path.join(state, "c_search_default")),
                                                     get_model_path(os.path.join(state, "a_played")),
                                                     args.match_games, args.sims, 23)})["c_vs_a"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--match-games", type=int, default=128)
    ap.add_argument("--sims", type=int, default=100)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--stage", choices=("generate", "train", "match", "all"), default="all",
                    help="run one part: generate (items 1-2, and the dataset of item 3), train or match (item 3); each "
                         "later part reads what the earlier one left in --state")
    ap.add_argument("--state", default=None, help="directory for the dataset and the weights (default: temporary)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_search_targets_bench.json"))
    args = ap.parse_args()
    res = {"card": card(), "stage": args.stage, "generate": []}
    with tempfile.TemporaryDirectory() as tmp:
        state = args.state or tmp
        os.makedirs(state, exist_ok=True)
        stages = ("generate", "train", "match") if args.stage == "all" else (args.stage,)
        for st in stages:
            {"generate": stage_generate, "train": stage_train, "match": stage_match}[st](args, res, state)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
