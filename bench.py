#!/usr/bin/env python
"""bench.py -- self-play MCTS simulations/sec (BASELINE.json's metric) for the lockstep engine on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--games G] [--sims S] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[3] "lockstep self-play 4,096 games x 200 sims/move on 1 B200",
random-init ChessRL network, synthetic start/midgame positions (half the lanes advanced by 8-60 seeded random
plies generated on the device).  With --gpus N (torchrun) every rank runs its own G games: games are independent,
so the path shards by game with no data-path collective ("scaling": "weak").

A STEP is one move search for all G lanes: a fresh tree per game, S simulations, i.e. G*S simulations.
  value : simulations/s with the games resident in HBM (tree build + S lockstep simulations, CUDA events).
  e2e   : the same metric through the public host API with HOST buffers inside the timed region: game records
          host->device, search, root statistics device->host, the numpy move policy, picks host->device, the chosen
          moves device->host (what selfplay.py does per move).
  roofline     : the dominant kernel (tcgen05 3x3 convolution), algorithmic FLOPs / CUDA-event time inside the step,
                 against the measured bf16 peak in MEASURED_PEAKS.json (sustained figure: timed inside a long step).
  cpu_baseline : the oracle port of the reference path (python-chess restatement + mctree restatement + torch-CPU
                 fp32 network, all host threads) on a bounded sample of the same workload; reported, not the target.
  perft        : secondary metric of BASELINE.json (perft nodes/s over >= 65,536 lockstep boards), bit-exact totals.

--dump-outputs DIR writes what the last timed step of each leg returned, as DIR/<name>.npy (float32 / float64), so that
two builds can be compared output for output; the inputs depend only on the arguments.  See dump_outputs().
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONV_FLOP_PER_POS = 2 * (3 * 3 * 127 * 256 * 64 + 20 * 3 * 3 * 256 * 256 * 64)   # unpadded, SURVEY.md 8(d)
NET_FLOP_PER_POS = 1548038656
KIWI = "r3k2r/p1ppqpb1/bn2pnp1/3PN3/1p2P3/2N2Q1p/PPPBBPPP/R3K2R w KQkq - 0 1"
RULES_NCU_NOTE = ("pipe_alu 66.9 %, pipe_xu 19.8 %, issue slots 63.8 % active, 82.5 warp instructions per board "
                  "(profiles/r02_ncu_rules_kernels.txt)")


def measured_tower_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per k_trunk4 launch from the committed ncu capture
    (profiles/r02_trunk4_dram.json, written by scripts/ncu_trunk_dram.py from the --set full report); None if absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_trunk4_dram.json")) as f:
            d = json.load(f)
        return d
    except Exception:
        return None


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synthetic_games(engine, n_games, seed, lo=8, hi=60, start_fraction=0.5):
    """Start positions for `start_fraction` of the lanes, midgame positions (lo..hi seeded random legal plies) for the
    rest.  The random plies are generated on the device with the engine's own movegen / make-move kernels."""
    import torch
    from chessrl_b200 import boards as B
    gen = torch.Generator(device="cpu").manual_seed(seed)
    target = torch.zeros(n_games, dtype=torch.int64)
    half = int(n_games * start_fraction)
    target[half:] = torch.randint(lo, hi + 1, (n_games - half,), generator=gen)
    boards = engine.boards_to_device(np.tile(B.record_from_fen(), (n_games, 1)))
    rnd = torch.randint(0, 1 << 30, (hi + 1, n_games), generator=gen).to(engine.device)
    target_d = target.to(engine.device)
    lists = torch.full((n_games, hi), B.MOVE_NONE - 65536, dtype=torch.int16, device=engine.device)
    for ply in range(hi):
        moves, counts, _ = engine.movegen(boards)
        alive = (counts > 0) & (target_d > ply)
        idx = (rnd[ply] % counts.clamp(min=1)).to(torch.int64)
        pick = moves.gather(1, idx[:, None])[:, 0]
        pick = torch.where(alive, pick, torch.full_like(pick, -1))        # 0xFFFF = skip
        engine.make_moves(boards, pick)
        lists[:, ply] = pick
        target_d = torch.where(alive, target_d, torch.zeros_like(target_d))   # a finished line stops
    lists_h = lists.cpu().numpy().view(np.uint16)
    move_lists = [[int(m) for m in row if m != B.MOVE_NONE] for row in lists_h]
    start = np.tile(B.record_from_fen(), (n_games, 1))
    return start, move_lists


def perft_metric(engine):
    """perft of the start position and Kiwipete (published totals, bit-exact):
      depth 5 over >= 65,536 lockstep boards (BASELINE configs[1]) and two plies deeper over >= 1 Mi boards, each as ONE
      crl_perft_root_host call (device-side breadth-first plies with atomic placement, then a depth-first walk per lane;
      no host round trip in between), timed with CUDA events around the call, with and without leaf bulk counting;
      plus the replicated variant: 65,536 copies of the root, every lane runs perft(3) in lockstep."""
    import torch
    from chessrl_b200 import boards as B
    out = {}

    def timed_root(fen, depth, want, bulk, min_frontier, reps=3):
        rec = B.record_from_fen(fen)
        best, info = None, None
        for rep in range(reps + 1):                     # the first call sizes the engine's frontier buffers
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            total, lanes, plies = engine.perft_root(rec, depth, bulk=bulk, min_frontier=min_frontier)
            b.record()
            torch.cuda.synchronize()
            assert total == want, (fen, depth, total, want)
            if rep:
                ms = a.elapsed_time(b)
                best = ms if best is None else min(best, ms)
            info = (lanes, plies)
        return best, info

    total_nodes, total_ms = 0, 0.0
    for name, fen, want in (("start", B.STARTING_FEN, 4865609), ("kiwipete", KIWI, 193690690)):
        ms, (lanes, plies) = timed_root(fen, 5, want, True, 1 << 20)       # >= 65,536 boards: 197,281 / 4,085,603 lanes
        ms_nb, _ = timed_root(fen, 5, want, False, 1 << 20)
        out[name] = {"nodes": want, "depth": 5, "ms": round(ms, 4), "nodes_per_s": want / ms * 1e3, "lanes": lanes,
                     "breadth_first_plies": plies, "leaf_bulk_counting": True,
                     "headline": "one crl_perft_root_host call: device-side frontier expansion + per-lane walk, leaf bulk counting",
                     "no_bulk_ms": round(ms_nb, 4), "no_bulk_nodes_per_s": want / ms_nb * 1e3}
        # replicated variant (SURVEY.md 8(d) config 2): 65,536 copies of the root, every lane runs perft(3) in lockstep
        rep = engine.boards_to_device(np.tile(B.record_from_fen(fen), (65536, 1)))
        per_lane = {"start": 8902, "kiwipete": 97862}[name]
        for bulk in (True, False):
            engine.perft(rep, 3, bulk=bulk)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            nodes_r = engine.perft(rep, 3, bulk=bulk)
            b.record()
            torch.cuda.synchronize()
            assert bool((nodes_r == per_lane).all())
            out[name]["replicated_65536_lanes_perft3_%s_nodes_per_s" % ("bulk" if bulk else "no_bulk")] = \
                65536 * per_lane / a.elapsed_time(b) * 1e3
        total_nodes += want
        total_ms += ms
    out["nodes_per_s"] = total_nodes / total_ms * 1e3
    # sustained throughput: two plies deeper (depth 5 is over in a fraction of a millisecond).  The breadth-first
    # frontier is grown all the way to the last-but-one ply (start: 119,060,324 boards, Kiwipete: 193,690,690 -- 8.6 / 13.9
    # GB of HBM) so that the walk is one count-only move generation per lane: every lane does the same amount of work and
    # warps stay converged -- about 3x the throughput of 65,536-board frontiers with three plies per lane
    # (scripts/perft_root_probe.py --deep).
    deep_nodes, deep_ms = 0, 0.0
    for name, fen, depth, want in (("start_d7", B.STARTING_FEN, 7, 3195901860), ("kiwipete_d6", KIWI, 6, 8031647685)):
        ms, (lanes, plies) = timed_root(fen, depth, want, True, 1 << 26, reps=2)
        ms_nb, _ = timed_root(fen, depth, want, False, 1 << 26, reps=1)
        out[name] = {"nodes": want, "depth": depth, "lanes": lanes, "breadth_first_plies": plies, "plies_per_lane": depth - plies,
                     "ms_bulk": round(ms, 3), "nodes_per_s_bulk": want / ms * 1e3,
                     "ms_no_bulk": round(ms_nb, 3), "nodes_per_s_no_bulk": want / ms_nb * 1e3}
        deep_nodes += want
        deep_ms += ms
    out["deep_nodes_per_s"] = deep_nodes / deep_ms * 1e3
    return out


def perft_sharded(engine, rank, world, dist):
    """perft over all ranks, ONE crl_perft_root_shard_host call per rank and root: every rank expands the first plies on
    its own GPU (device-side, no host round trip); the first ply whose input frontier holds >= 4,096 boards keeps only
    the children that hash to this rank, which then expands and walks its own boards alone; ONE all_reduce(sum) of an int64
    per root joins the counts (SURVEY.md 8(e)).  The timed region is the whole call -- root in, shard total out -- max over ranks."""
    import torch
    from chessrl_b200 import boards as B
    from chessrl_b200 import sharding
    out = {}
    for name, fen, depth, want in (("start_d6", B.STARTING_FEN, 6, 119060324), ("kiwipete_d5", KIWI, 5, 193690690),
                                   ("start_d7", B.STARTING_FEN, 7, 3195901860), ("kiwipete_d6", KIWI, 6, 8031647685)):
        rec = B.record_from_fen(fen)
        min_frontier = max(1 << 16, ((1 << 20) if depth <= 5 else (1 << 26)) // world)
        best, lanes = None, 0
        for rep in range(4):                                   # the first call sizes the frontier buffers
            dist.barrier()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            mine, lanes, plies = engine.perft_root(rec, depth, bulk=True, min_frontier=min_frontier, shard=rank,
                                                   n_shards=world, shard_min_frontier=1 << 12)
            b.record()
            torch.cuda.synchronize()
            t = torch.tensor([a.elapsed_time(b)], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total = sharding.sum_counts([mine])                            # one all_reduce(sum) of an int64
            assert total == want, (name, total, want)
            if rep > 0:
                best = float(t.item()) if best is None else min(best, float(t.item()))
        out[name] = {"nodes": want, "ms_max_over_ranks": best, "nodes_per_s": want / best * 1e3,
                     "timed": "the whole sharded call on every rank: replicated first plies, own boards (by record hash) from the "
                              "first >= 4,096-board frontier on, walk; max over ranks",
                     "lanes_this_rank": int(lanes), "breadth_first_plies": int(plies), "leaf_bulk_counting": True}
    return out


def whole_games_steady_state(model_pack, lanes, sims, inflight, n_steps, seed, reuse=False):
    """reuse=False: every search evaluates every position (comparable with the per-move `value`); reuse=True: what
    selfplay.py runs by default -- evaluations of the previous move's search of the same game are looked up instead of
    run again (crl_set_reuse; same games move for move, tests/test_gpu_reuse.py), so a simulation costs fewer than two
    network evaluations.
    The path selfplay.py runs (chessrl_b200.selfplay.LockstepRun: harvest finished games -> refill their lanes ->
    one lockstep move for all lanes incl. the host-side move pick) in its steady state, timed by WALL CLOCK.
    Lanes start at staggered phases (0..300 random plies) so games end -- and lanes are harvested and refilled -- at
    their natural rate inside the timed window; the supply of games is unbounded, so there is no drain tail here
    (a finite run's tail is measured by `bench.py --whole-games N`, profiles/)."""
    import torch
    from chessrl_b200._lib import EVAL_NET
    from chessrl_b200.engine import Engine
    from chessrl_b200.selfplay import LockstepRun, edge_slots_per_node
    eng = Engine(max_games=lanes, max_nodes=sims + 1, max_inflight=inflight, avg_moves=edge_slots_per_node(lanes, sims + 1))
    eng.load_weights(model_pack)
    eng.set_evaluator(EVAL_NET)
    start, move_lists = synthetic_games(eng, lanes, seed, lo=0, hi=300, start_fraction=0.0)
    run = LockstepRun(None, None, sims=sims, lanes=lanes, noise=True, seed=seed, threads=inflight, engine=eng, reuse=reuse)
    np.random.seed(seed)
    run.start(start_records=start, move_lists=eng.pack_move_lists(move_lists))
    run.advance()                                                   # warm-up step (graph capture, first refills)
    torch.cuda.synchronize()
    c0, f0, r0, m0 = eng.counters(), run.finished_games, run.refills, run.sp.moves_played
    t0 = time.perf_counter()
    for _ in range(n_steps):
        run.advance()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    c1 = eng.counters()
    sims_done = c1["simulations"] - c0["simulations"]
    out = {"workload": "%d lanes x %d sims/move, %d lockstep moves, unbounded game supply, lanes at staggered phases" %
                       (lanes, sims, n_steps),
           "timing": "wall clock around LockstepRun.advance() x %d (harvest + refill + search + host move pick + commit)" % n_steps,
           "seconds": dt, "simulations_per_s": sims_done / dt, "agent_moves": run.sp.moves_played - m0,
           "games_finished": run.finished_games - f0, "lanes_refilled": run.refills - r0,
           "games_per_s_at_this_phase_mix": (run.finished_games - f0) / dt,
           "lane_occupancy": sims_done / max(1, n_steps * lanes * sims),
           "evaluations_per_simulation": (c1["evaluations"] - c0["evaluations"]) / max(1, sims_done),
           "evaluation_reuse": bool(reuse),
           "reused_evaluations_per_simulation": (c1["reused_evaluations"] - c0["reused_evaluations"]) / max(1, sims_done)}
    eng.close()
    return out


def whole_games_complete_run(model_pack, n_games, lanes, sims, inflight, seed, reuse=True):
    """A complete finite self-play run through chessrl_b200.selfplay.play_games_lockstep, drain tail included."""
    from chessrl_b200 import model
    from chessrl_b200.selfplay import play_games_lockstep
    m = model.ChessModel()
    m.weights = model_pack
    np.random.seed(seed)
    stats = {}
    data = play_games_lockstep(m, n_games, sims=sims, lanes=lanes, noise=True, seed=seed, threads=inflight, stats=stats,
                               reuse=reuse)
    res = [g.get_result() for g in data.games]
    stats.update({"games": len(data), "mean_plies": float(np.mean([len(g) for g in data.games])),
                  "white_wins": res.count(1), "black_wins": res.count(-1), "draws": res.count(0), "unfinished": res.count(None),
                  "simulations_per_s_wall_clock": stats["simulations"] / stats["seconds"],
                  "games_per_s": len(data) / stats["seconds"]})
    return stats


def training_step_leg(pack, n_positions=640, steps=10, warmup=3):
    """SURVEY.md 8(f) rank 1: the training step behind Agent.train (chessrl_b200/training.py: Keras loss, tf.keras Adam,
    BatchNorm in training mode; PyTorch fp32 WITHOUT TF32, like the reference's fp32 TensorFlow -- north_star allows
    PyTorch here) on a synthetic batch the size of 8 games x 80 plies, timed with CUDA events.  Reported against the
    forward + backward arithmetic (3 x the network's forward FLOPs); not a tensor-core path by construction (fp32)."""
    import torch
    from chessrl_b200 import training
    dev = torch.device("cuda", torch.cuda.current_device())
    g = torch.Generator(device=dev).manual_seed(3)
    planes = (torch.rand((n_positions, 8, 8, 128), device=dev, generator=g) < 0.15).to(torch.bfloat16)
    planes[..., 127] = 0
    pol = torch.randint(0, 1968, (n_positions,), device=dev, generator=g)
    val = torch.randint(-1, 2, (n_positions,), device=dev, generator=g).float()
    out = {}
    for precision in training.PRECISIONS:
        params = [torch.tensor(w, device=dev) for w in pack]
        trainable = []
        for i in training.trainable_indices():
            params[i].requires_grad_(True)
            trainable.append(params[i])
        opt = training.KerasAdam(trainable, lr=0.002, epsilon=1e-7)
        with training.arithmetic(precision):
            for _ in range(warmup):
                training.train_step(params, opt, planes, pol, val)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            for _ in range(steps):
                rec = training.train_step(params, opt, planes, pol, val)
            b.record()
            torch.cuda.synchronize()
        ms = a.elapsed_time(b) / steps
        out[precision] = {"ms_per_step": ms, "positions_per_s": n_positions / (ms * 1e-3),
                          "tflops": 3 * NET_FLOP_PER_POS * n_positions / (ms * 1e-3) / 1e12, "last_loss": rec["loss"]}
    return {"workload": "one training step (forward in training mode + backward + Adam) on %d synthetic positions = 8 games x 80 "
                        "plies (PyTorch / cuDNN; SURVEY.md 8f rank 1); fp32 without TF32 is the default and the parity setting, "
                        "tf32 / bf16 autocast are opt-in (CRL_TRAIN_PRECISION)" % n_positions,
            "ms_per_step": out["fp32"]["ms_per_step"], "positions_per_s": out["fp32"]["positions_per_s"],
            "tflops_fp32": out["fp32"]["tflops"], "by_precision": out}


def large_config(pack, world, rank, dist, barrier, K):
    """BASELINE configs[4] (65,536 games x 800 sims/move sharded by game over the ranks) when there are >= 2 ranks;
    on one GPU the >= 65k-concurrent-games claim: 65,536 games x 200 sims/move.  One timed step after a short warm-up."""
    import torch
    from chessrl_b200._lib import EVAL_NET
    from chessrl_b200.engine import Engine
    G2 = 65536 // world
    S2 = 800 if world > 1 else 200
    eng = Engine(max_games=G2, max_nodes=S2 + 1, avg_moves=64, max_inflight=K)
    eng.load_weights(pack)
    eng.set_evaluator(EVAL_NET)
    start, move_lists = synthetic_games(eng, G2, seed=4321 + rank)
    eng.games_set(start, eng.pack_move_lists(move_lists))
    eng.mcts_begin_move()
    eng.mcts_simulate(4, K)                                         # warm-up: graph capture, tensor maps
    barrier()
    c0 = eng.counters()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    eng.mcts_begin_move()
    eng.mcts_simulate(S2, K)
    b.record()
    barrier()
    ms = a.elapsed_time(b)
    c1 = eng.counters()
    sims = float(c1["simulations"] - c0["simulations"])
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        t = torch.tensor([sims], device="cuda", dtype=torch.float64)
        dist.all_reduce(t)
        sims = float(t.item())
    eng.close()
    return {"workload": ("BASELINE configs[4]: 65,536 games x 800 sims/move sharded by game over %d GPUs (%d games per GPU)" % (world, G2))
            if world > 1 else "65,536 concurrent games on ONE GPU x 200 sims/move (north_star: >= 65k concurrent games)",
            "games_total": G2 * world, "games_per_gpu": G2, "sims_per_move": S2, "steps": 1, "ms_per_step_max_over_ranks": ms,
            "simulations": sims, "simulations_per_s": sims / (ms * 1e-3), "tower": "k_trunk4"}


def _time_launch(fn, flush, reps=5):
    """Mean CUDA-event time (ms) of `fn` (one launch), L2 flushed before every timed launch, 3 warm-ups.
    The flush writes a buffer larger than L2 and then READS it back, so the kernel under test does not also pay for
    the write-back of the flush's dirty lines."""
    import torch
    for _ in range(3):
        fn()
    tot = 0.0
    for _ in range(reps):
        flush.fill_(1)
        flush.max()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        tot += a.elapsed_time(b)
    return tot / reps


def kernel_rooflines(engine, peaks, flush, net_loaded):
    """Per-kernel achieved throughput against its roofline (SURVEY.md 8(d) algorithmic bytes / FLOPs per unit),
    each kernel timed alone through the C ABI on device-resident inputs larger than L2 or after an L2 flush."""
    import torch
    from chessrl_b200 import boards as B
    out = {}
    hbm = peaks["hbm_gbs"]
    # ~1M midgame boards: Kiwipete's depth-3 frontier (97,862 boards) replicated 11 times
    fr = engine.boards_to_device(B.record_from_fen(KIWI)[None, :])
    for _ in range(3):
        fr, _ = engine.expand_frontier(fr)
    boards = fr.repeat(1, 11).contiguous()
    n = boards.shape[1]
    moves = torch.empty((n, B.MAX_MOVES), dtype=torch.int16, device=engine.device)
    counts = torch.empty((n,), dtype=torch.int32, device=engine.device)
    from chessrl_b200.engine import _ptr
    from chessrl_b200._lib import check
    ms = _time_launch(lambda: check(engine.lib.crl_movegen(engine.h, _ptr(boards), n, _ptr(moves), _ptr(counts), None)), flush)
    avg_l = float(counts.float().mean().item())
    byt = n * (72 + 2 * avg_l + 4)
    out["movegen"] = {"bound": "INT32 ALU pipe (64-bit bitboard logic on the half-rate integer pipe), then hbm; ncu pipe / issue-slot "
                               "figures of the current build: " + RULES_NCU_NOTE, "boards": n, "avg_legal_moves": avg_l, "us": ms * 1e3,
                      "boards_per_s": n / ms * 1e3, "achieved": byt / ms / 1e6, "peak": hbm, "unit": "GB/s",
                      "frac": byt / ms / 1e6 / hbm, "algorithmic_bytes_per_board": 72 + 2 * avg_l + 4}
    first = moves[:, 0].contiguous()
    work = boards.clone()
    ms = _time_launch(lambda: check(engine.lib.crl_make_moves(engine.h, _ptr(work), n, _ptr(first))), flush)
    out["make_move"] = {"bound": "hbm", "boards": n, "us": ms * 1e3, "moves_per_s": n / ms * 1e3,
                        "achieved": n * 146 / ms / 1e6, "peak": hbm, "unit": "GB/s", "frac": n * 146 / ms / 1e6 / hbm,
                        "algorithmic_bytes_per_move": 146}
    # encode: 32,768 positions with a full 8-position history (580 B in, 16,384 B out per position)
    ne = 32768
    eb = boards[:, :ne].contiguous()
    hist = boards[:8, :8 * ne].reshape(8, 8, ne).contiguous()      # any bitboards do: the kernel's traffic is what counts
    hl = torch.full((ne,), 8, dtype=torch.uint8, device=engine.device)
    planes = torch.empty((ne, 8, 8, 128), dtype=torch.bfloat16, device=engine.device)
    ms = _time_launch(lambda: check(engine.lib.crl_encode(engine.h, _ptr(eb), _ptr(hist), _ptr(hl), ne, _ptr(planes))), flush)
    byt = ne * (580 + 16384)
    out["encode"] = {"bound": "hbm", "positions": ne, "us": ms * 1e3, "positions_per_s": ne / ms * 1e3,
                     "achieved": byt / ms / 1e6, "peak": hbm, "unit": "GB/s", "frac": byt / ms / 1e6 / hbm,
                     "algorithmic_bytes_per_position": 580 + 16384}
    del planes, hist
    if net_loaded:
        # BASELINE configs[2]: encode + network evaluation, 4,096 positions per batch, 3 distinct batches rotated
        nb = 4096
        batches = []
        for k in range(3):
            bb = boards[:, k * nb:(k + 1) * nb].contiguous()
            hh = boards[:8, (3 + 8 * k) * nb:(3 + 8 * k + 8) * nb].reshape(8, 8, nb).contiguous()
            batches.append((bb, hh, torch.full((nb,), 8, dtype=torch.uint8, device=engine.device),
                            torch.empty((nb, 8, 8, 128), dtype=torch.bfloat16, device=engine.device),
                            torch.empty((nb, 1968), dtype=torch.float32, device=engine.device),
                            torch.empty((nb,), dtype=torch.float32, device=engine.device)))

        def one(k):
            bb, hh, ll, pl, po, va = batches[k % 3]
            check(engine.lib.crl_encode(engine.h, _ptr(bb), _ptr(hh), _ptr(ll), nb, _ptr(pl)))
            check(engine.lib.crl_net_forward(engine.h, _ptr(pl), nb, _ptr(po), _ptr(va)))
        for k in range(3):
            one(k)
        torch.cuda.synchronize()
        reps = 30
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for k in range(reps):
            one(k)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / reps
        tf = nb * NET_FLOP_PER_POS / ms / 1e9
        out["encode_plus_net"] = {"bound": "tensor", "workload": "BASELINE configs[2]: 4,096 positions per batch, encode + "
                                  "policy/value network, 3 distinct batches rotated, 30 back-to-back evaluations",
                                  "positions_per_s": nb / ms * 1e3, "ms_per_batch": ms, "achieved": tf,
                                  "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                                  "frac": tf / peaks["bf16_tflops_sustained"]}
    return out


def cpu_perft_baseline():
    """Single-core perft(3) of the start position and Kiwipete on the python-chess restatement (BASELINE.md 3.3)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import chessrl_oracle as O
    chess = O.chess

    def perft(board, d):
        if d == 0:
            return 1
        n = 0
        for m in board.generate_legal_moves():
            board.push(m)
            n += perft(board, d - 1)
            board.pop()
        return n
    out = {}
    for name, fen, want in (("start", None, 8902), ("kiwipete", KIWI, 97862)):
        b = chess.Board(fen) if fen else chess.Board()
        t0 = time.perf_counter()
        got = perft(b, 3)
        dt = time.perf_counter() - t0
        assert got == want, (name, got, want)
        out[name] = {"depth": 3, "nodes": got, "nodes_per_s": got / dt}
    out["cores"] = 1
    out["kind"] = "port (python-chess 0.28.3 restatement, pure Python)"
    return out


def cpu_reference_sims(budget_s, sims_per_move, seed=0, torch_threads=None):
    """The reference path on the host cores: oracle restatement of selfplay.play_game / mctree (threads=1) with the
    torch-CPU fp32 network, 1 game from the start position, `sims_per_move` simulations per move, for about
    `budget_s` seconds.  Returns (simulations, seconds, evals, cores)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import chessrl_oracle as O
    import model_torch
    from chessrl_b200 import model
    torch.set_num_threads(torch_threads or os.cpu_count() or 1)
    pack = model.random_pack(0)

    def evaluate(game):
        with torch.no_grad():
            p, v = model_torch.forward(pack, O.planes(game)[None].astype(np.float32), device="cpu")
        return p[0].numpy(), np.float32(v[0].item())

    agent = O.OAgent(evaluate)
    game = O.OGame()
    np.random.seed(seed)
    sims = 0
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < budget_s and game.get_result() is None:
        tree = O.OSelfPlayTree(game)
        for _ in range(sims_per_move):
            tree.explore_tree(agent)
            sims += 1
            if time.perf_counter() - t0 >= budget_s:
                break
        else:
            pick = int(np.argmax(tree.compute_policy(tree.root, noise=True)))
            stack = tree.root.children[pick].state.board.move_stack
            if len(stack) >= 2:
                game.move(str(stack[-2]))
                game.move(str(stack[-1]))
    dt = time.perf_counter() - t0
    return sims, dt, agent.n_evals, torch.get_num_threads()


def _cpu_worker(job):
    budget_s, sims_per_move, seed = job
    s, t, ev, _ = cpu_reference_sims(budget_s, sims_per_move, seed=seed, torch_threads=1)
    return s, t, ev


def cpu_reference_parallel(budget_s, sims_per_move, procs=None):
    """All host cores: one game per core (one process each, 1 torch thread), the same path as cpu_reference_sims.
    The reference itself plays one game at a time; this is the strongest arrangement of its path on the host.
    Returns (simulations, seconds = slowest worker, evals, processes)."""
    import multiprocessing as mp
    from concurrent.futures import ProcessPoolExecutor
    procs = procs or os.cpu_count() or 1
    with ProcessPoolExecutor(max_workers=procs, mp_context=mp.get_context("spawn")) as ex:
        res = list(ex.map(_cpu_worker, [(budget_s, sims_per_move, i) for i in range(procs)]))
    return sum(r[0] for r in res), max(r[1] for r in res), sum(r[2] for r in res), procs


def cpu_baseline_best(budget_s, sims_per_move=100):
    """Times both arrangements for about budget_s seconds each and returns the faster as the baseline."""
    s1, t1, ev1, c1 = cpu_reference_sims(budget_s, sims_per_move)
    sp, tp, evp, cp = cpu_reference_parallel(budget_s, sims_per_move)
    one = {"value": s1 / t1, "cores": c1, "arrangement": "1 game, torch intra-op threads = all cores (the reference's own "
           "structure: one game at a time)", "simulations": s1, "evaluations": ev1, "seconds": t1}
    par = {"value": sp / tp, "cores": cp, "arrangement": "1 game per core, %d processes x 1 torch thread" % cp,
           "simulations": sp, "evaluations": evp, "seconds": tp}
    best = par if par["value"] >= one["value"] else one
    return best, one, par


def run_reference(args, rank, world):
    if rank != 0:
        return
    per_step = max(1.0, min(20.0, 60.0 / max(1, args.steps + args.warmup)))
    for _ in range(args.warmup):
        cpu_reference_sims(min(per_step, 2.0), args.sims)
    # pick the arrangement once (short probe), then time the steps with it
    best, one, par = cpu_baseline_best(min(per_step, 5.0), args.sims)
    parallel = best is par
    tot_s, tot_t, cores = 0, 0.0, 1
    for _ in range(args.steps):
        if parallel:
            s, t, _, cores = cpu_reference_parallel(per_step, args.sims)
        else:
            s, t, _, cores = cpu_reference_sims(per_step, args.sims)
        tot_s += s
        tot_t += t
    v = tot_s / tot_t
    sample = "%s; games from the start position, %d sims/move, threads=1 schedule, %.0f s of simulations per step" % (
        best["arrangement"], args.sims, per_step)
    line = {"impl": "reference", "metric": "mcts_simulations_per_sec", "value": v, "unit": "simulations/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": tot_t / max(1, args.steps) * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD(args), "note": "reference arm = oracle port of python-chess + mctree + "
                       "torch-CPU fp32 network (python-chess / TensorFlow are not installable offline)"},
            "cpu_baseline": {"value": v, "unit": "simulations/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "simulations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def WORKLOAD(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.games * world == 65536 and args.sims == 800:
        which = "BASELINE configs[4]: 65,536 games x 800 sims/move sharded by game over %d GPU(s)" % world
    elif args.games == 4096 and args.sims == 200:
        which = "BASELINE configs[3] per GPU"
    else:
        which = "a scaled variant of BASELINE configs[3]"
    return "lockstep self-play %d games/GPU x %d sims/move, random-init ChessRL net (%s)" % (args.games, args.sims, which)


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, stats, picks, chosen):
    """Writes the last timed step's results as out_dir/<name>.npy, one row per lane:
      visits, values, priors, moves, replies, results [lanes, 256], n_children, root_visits, root_values [lanes]
        -- Engine.root_stats() after the last device-resident step (the `value` leg);
      e2e_picks [lanes], e2e_chosen [lanes, 2] -- the picks and the (move, reply) words Engine.commit returned in the
        last step of the `e2e` leg.
    Integers are stored as float32 (exact: every value is below 2**24), float64 stays float64.  If all lanes together
    would exceed DUMP_LIMIT_BYTES, a fixed seeded sample of lanes is written instead; lanes.npy lists the lane indices."""
    arrays = {k: stats[k] for k in ("visits", "values", "priors", "moves", "replies", "results", "n_children",
                                    "root_visits", "root_values")}
    arrays["e2e_picks"] = picks
    arrays["e2e_chosen"] = chosen
    arrays = {k: v.astype(np.float64 if v.dtype == np.float64 else np.float32) for k, v in arrays.items()}
    n = len(arrays["root_visits"])
    per_lane = sum(v.nbytes for v in arrays.values()) // n + 8
    lanes = np.arange(n)
    if per_lane * n > DUMP_LIMIT_BYTES:
        lanes = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // per_lane, replace=False))
    arrays = {k: np.ascontiguousarray(v[lanes]) for k, v in arrays.items()}
    arrays["lanes"] = lanes.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)
    sys.stderr.write("bench: wrote %d arrays for %d of %d lanes to %s\n" % (len(arrays), len(lanes), n, out_dir))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--games", type=int, default=4096, help="lockstep games per GPU")
    ap.add_argument("--sims", type=int, default=200, help="simulations per move")
    ap.add_argument("--inflight", type=int, default=1, help="simulations in flight per game (reference --threads); 1 = exact schedule")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-perft", action="store_true")
    ap.add_argument("--no-kernels", action="store_true", help="skip the per-kernel roofline section")
    ap.add_argument("--no-whole-games", action="store_true", help="skip the steady-state whole-game leg")
    ap.add_argument("--wg-steps", type=int, default=10, help="lockstep moves timed in the steady-state whole-game leg")
    ap.add_argument("--no-large", action="store_true", help="skip the configs[4] / 65,536-games leg")
    ap.add_argument("--no-training", action="store_true", help="skip the training-step leg")
    ap.add_argument("--whole-games", type=int, default=0, help="also play this many COMPLETE games (drain included)")
    ap.add_argument("--wg-lanes", type=int, default=None)
    ap.add_argument("--wg-sims", type=int, default=None)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs (root statistics, e2e picks) as DIR/<name>.npy (rank 0's lanes)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from chessrl_b200 import boards as B
    from chessrl_b200 import model
    from chessrl_b200._lib import EVAL_NET
    from chessrl_b200.engine import Engine
    from chessrl_b200.lockstep import pick_moves

    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    peaks = load_peaks()
    G, S = args.games, args.sims

    K = max(1, args.inflight)
    eng = Engine(max_games=G, max_nodes=S + 1, avg_moves=64, max_inflight=K)
    pack = model.random_pack(seed=0)
    if world > 1:
        # weights live on rank 0 and are broadcast over NCCL (the only collective on this path besides timing)
        flat = torch.cat([torch.from_numpy(w.reshape(-1)) for w in pack]).cuda()
        dist.broadcast(flat, 0)
        flat = flat.cpu().numpy()
        o, pk = 0, []
        for w in pack:
            pk.append(flat[o:o + w.size].reshape(w.shape))
            o += w.size
        pack = pk
    eng.load_weights(pack)
    eng.set_evaluator(EVAL_NET)
    start, move_lists = synthetic_games(eng, G, seed=1234 + rank)
    packed = eng.pack_move_lists(move_lists)                                # host buffers (uint16 moves, int32 counts)
    eng.games_set(start, packed)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")     # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def device_step():
        eng.mcts_begin_move()
        eng.mcts_simulate(S, K)

    def e2e_step():
        eng.games_set(start, packed)                                       # host -> device (records + move lists)
        eng.mcts_begin_move()
        eng.mcts_simulate(S, K)
        st = eng.root_stats(want=("visits",))                              # device -> host
        _, plies, results = eng.games_get(0, G)
        picks = pick_moves(st["visits"], st["n_children"], st["root_visits"], plies, results == B.RESULT_NONE, True)
        return picks, eng.commit(picks, apply=False)                       # host -> device, device -> host

    np.random.seed(0)

    def timed(fn, steps, warmup):
        """-> (summed step ms, counter deltas, what the last timed fn() call returned)"""
        for _ in range(warmup):
            flush.fill_(1)
            fn()
        barrier()
        c0 = eng.counters()
        evs = []
        last = None
        for _ in range(steps):
            flush.fill_(1)                                                 # L2 flush between timed iterations
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            last = fn()
            b.record()
            evs.append((a, b))
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        c1 = eng.counters()
        if world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, {k: c1[k] - c0[k] for k in c0}, last

    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_dev, cnt_dev, _ = timed(device_step, args.steps, args.warmup)
    clocks = sampler.stop()
    dev_stats = eng.root_stats() if args.dump_outputs and rank == 0 else None     # the last device step's trees
    wall0 = time.perf_counter()
    ms_e2e, cnt_e2e, (e2e_picks, e2e_chosen) = timed(e2e_step, args.steps, max(1, min(args.warmup, 1)))
    del wall0
    if dev_stats is not None:
        dump_outputs(args.dump_outputs, dev_stats, e2e_picks, e2e_chosen)
    sims_dev = cnt_dev["simulations"]
    sims_e2e = cnt_e2e["simulations"]
    if world > 1:
        t = torch.tensor([sims_dev, sims_e2e, cnt_dev["launches"], cnt_dev["evaluations"]], device="cuda", dtype=torch.float64)
        dist.all_reduce(t)
        sims_dev, sims_e2e, launches_all, evals_all = (float(x) for x in t.tolist())
    else:
        launches_all, evals_all = cnt_dev["launches"], cnt_dev["evaluations"]
    value = sims_dev / (ms_dev * 1e-3)
    e2e_value = sims_e2e / (ms_e2e * 1e-3)

    # ---- roofline of the dominant kernel (conv), measured live with CUDA events around every conv launch ----
    roof = None
    prof = None
    TRAFFIC = measured_tower_traffic()
    if rank == 0:
        eng.profile(True)
        c0 = eng.counters()
        eng.mcts_begin_move()
        eng.mcts_simulate(min(S, 200 * K), K)      # a whole step (capped at 200 waves), so clocks are the sustained ones
        torch.cuda.synchronize()
        prof = eng.profile_read()
        c1 = eng.counters()
        eng.profile(False)
        evals = c1["evaluations"] - c0["evaluations"]
        conv = prof["conv"]
        if conv["launches"] and conv["ms"] > 0:
            flop_per_launch = evals * CONV_FLOP_PER_POS / conv["launches"]
            t_launch = conv["ms"] * 1e-3 / conv["launches"]
            achieved = flop_per_launch / t_launch / 1e12
            v3 = os.environ.get("CRL_TRUNK_V3") == "1"
            roof = {"bound": "tensor", "kernel": ("k_trunk (v3)" if v3 else "k_trunk4") + " (the 21 tcgen05 cta_group::2 implicit-GEMM "
                    "3x3 convolutions of the residual tower as ONE persistent CTA-pair kernel" +
                    ("" if v3 else "; the zero-padded board image of each 64-channel slice is loaded once and serves all nine filter taps "
                     "through shifted shared-memory descriptors") + ")", "achieved": achieved,
                    "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16_tflops_sustained"],
                    "peak_source": peaks["source"] + " bf16_tflops_sustained (kernel timed inside a long step); frac > 1 means the "
                                   "kernel sustains more than cuBLAS did in the driver's 4 s matmul loop on this pod",
                    "peak_burst": peaks["bf16_tflops"], "frac_of_burst": achieved / peaks["bf16_tflops"],
                    "flop_per_launch": flop_per_launch, "us_per_launch": t_launch * 1e6,
                    # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture of
                    # this kernel at 4,096 positions (read from profiles/, not pasted).  Algorithmic minimum: 67.1 MB planes in
                    # + 24.8 MB weights + 1.6 MB head features out = 93.5 MB
                    "traffic": (TRAFFIC or {}).get("dram_bytes_per_launch") if (G == 4096 and K == 1 and not v3) else None,
                    "traffic_unit": "bytes/launch", "traffic_source": (TRAFFIC or {}).get("source"),
                    "traffic_algorithmic": 93.5e6,
                    "share_of_step_ms": {k: round(v["ms"], 3) for k, v in prof.items()}}

    # ---- perft (secondary metric) and CPU baseline, rank 0 only ----
    perft = None
    cpu = None
    kernels = None
    perft_multi = None
    if world > 1 and not args.no_perft:
        small = Engine(max_games=1, max_nodes=8)
        perft_multi = perft_sharded(small, rank, world, dist)
        small.close()
    if rank == 0 and not args.no_perft:
        small = Engine(max_games=1, max_nodes=8)
        perft = perft_metric(small)
        small.close()
        if not args.no_cpu_baseline and world == 1:
            perft["cpu_baseline"] = cpu_perft_baseline()
    if rank == 0 and not args.no_kernels:
        kernels = kernel_rooflines(eng, peaks, flush, True)
    whole = None
    whole_reuse = None
    complete = None
    large = None
    eng.close()                                      # the legs below size their own engines
    if rank == 0 and not args.no_whole_games:
        whole = whole_games_steady_state(pack, args.wg_lanes or G, args.wg_sims or S, K, args.wg_steps, seed=7)
        whole["fraction_of_device_resident_value"] = whole["simulations_per_s"] / (value / world) if (args.wg_lanes or G) == G and (args.wg_sims or S) == S else None
        if K == 1:      # the same loop with evaluation reuse on (selfplay.py's default): same games, fewer evaluations
            whole_reuse = whole_games_steady_state(pack, args.wg_lanes or G, args.wg_sims or S, K, args.wg_steps, seed=7, reuse=True)
            whole_reuse["speedup_over_no_reuse"] = whole_reuse["simulations_per_s"] / whole["simulations_per_s"]
    if rank == 0 and args.whole_games > 0:
        complete = whole_games_complete_run(pack, args.whole_games, args.wg_lanes or G, args.wg_sims or S, K, seed=7)
    train_leg = None
    if rank == 0 and not args.no_training:
        train_leg = training_step_leg(pack)
    if not args.no_large:
        large = large_config(pack, world, rank, dist, barrier, K)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        best, one, par = cpu_baseline_best(12.0)
        cpu = {"value": best["value"], "unit": "simulations/s", "cores": best["cores"], "kind": "port",
               "sample": "%s; start position, 100 sims/move (BASELINE configs[0]), %d simulations / %d network evaluations in "
                         "%.1f s; oracle port (python-chess restatement + mctree restatement + torch-CPU fp32 net)" % (
                             best["arrangement"], best["simulations"], best["evaluations"], best["seconds"]),
               "one_game_all_threads": one["value"], "one_game_per_core": par["value"]}

    if rank == 0:
        bytes_h2d = G * 72 + G * 4 + int(packed[0].nbytes) + G * 4     # records, counts, padded move lists, picks
        bytes_d2h = G * 256 * 4 + 3 * G * 4 + G * 8 + G * 72 + G * 5 + G * 4
        line = {
            "metric": "mcts_simulations_per_sec", "value": value, "unit": "simulations/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD(args), "games_per_gpu": G, "sims_per_move": S,
                       "step": "one move search for all lanes = G*S simulations", "schedule": ("1 in-flight simulation per game (exact threads=1 parity mode)" if K == 1 else
                                    "waves of up to %d in-flight simulations per game (reference --threads %d)" % (K, K)),
                       "l2": "256 MiB buffer written between timed steps; working set (trees + activations) > L2",
                       "parallelism": "games sharded by lane across %d GPU(s), no per-simulation collective" % world},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "simulations/s", "h2d_bytes_per_step": bytes_h2d, "d2h_bytes_per_step": bytes_d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches_all),
            "evaluations_per_simulation": evals_all / max(1.0, sims_dev),
            "net_tflops_in_step": evals_all * NET_FLOP_PER_POS / (ms_dev * 1e-3) / 1e12 / world,
            "roofline": roof, "cpu_baseline": cpu, "perft": perft, "perft_sharded": perft_multi, "kernels": kernels,
            "whole_games": whole, "whole_games_reuse": whole_reuse, "whole_games_complete_run": complete, "large_config": large, "training_step": train_leg,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
