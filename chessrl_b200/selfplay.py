"""selfplay: drop-in for the reference's entry point (selfplay.py:111-167)

    python -m chessrl_b200.selfplay modeldir [--games 1] [--threads 1] [--debug] [--sims 900] [--lanes N] [--no-train]

Plays `--games` self-play games, appends them to <modeldir>/gameplays.json (README.md:77) and trains the model on
them, saving the weights in place.  Unlike the reference, which plays one game at a time in a child process and
talks to a prediction server over TCP, the games run in LOCKSTEP on the GPU (`--lanes` at a time, default all of
them) and the "server" is the batched network evaluation inside the engine.  `--threads` = simulations in flight
per game, like the reference's MCTS thread pool; its default here is 1 (the reference's only deterministic
schedule) instead of 6, K > 1 runs the wave schedule (include/chessrl_b200.h).  `--sims` exposes the
reference's hard-coded 900 simulations per move (selfplay.py:76).  With torchrun the games are sharded by rank,
rank 0 broadcasts the weights and gathers the finished games (NCCL); there is no per-simulation collective.
"""

from __future__ import annotations

import argparse
import os
import random

import numpy as np

from . import boards as B
from .agent import Agent
from .dataset import DatasetGame
from .game import Game
from .lib.logger import Logger


def get_model_path(directory):
    """Newest <directory>/model-<n>.h5 by the reference's rule (selfplay.py:33-56); model-0.h5 if none."""
    path = directory + "/model-0.h5"
    models = [f for f in os.listdir(directory) if f.endswith("h5")]
    if models:
        max_v = max(m.split("-")[1] for m in models)
        path = directory + "/" + [m for m in models if m.endswith(max_v)][0]
    return path


def play_game(agent, max_iters=900):
    """One game through the single-object API, the reference's play_game loop (selfplay.py:59-84)."""
    logger = Logger.get_instance()
    player_color = random.random() >= 0.5
    logger.debug("Player is white: %s" % player_color)
    gam = Game(player_color=player_color)
    agent.color = player_color
    if player_color is False:
        gam.move(agent.best_move(gam, real_game=True))
    while gam.get_result() is None:
        bm, am = agent.best_move(gam, real_game=False, ai_move=True, max_iters=max_iters)
        if not gam.move(bm) | gam.move(am):
            break                                   # the reference would spin forever on two rejected moves
        logger.debug("\tMade move: %s" % bm)
    logger.debug(gam.get_history())
    return gam


def edge_slots_per_node(lanes, nodes, device=None, bytes_per_edge=24, share=0.5):
    """(bytes_per_edge: 24 for the seven edge arrays, 32 with evaluation reuse, which keeps the previous tree's child /
    prior arrays as well.)  Edge-pool sizing for long runs: every tree node reserves one edge slot per legal move of its position, and no
    chess position has more than 218 legal moves, so 218 slots per node can never overflow.  That is what a run gets
    whenever it fits in `share` of the free device memory (4,096 lanes x 901 nodes: 19 GB of a B200's 180 GB);
    otherwise as many as fit (an overflow is then reported as CRL_ENOMEM, never silent)."""
    import torch
    with torch.cuda.device(torch.cuda.current_device() if device is None else device):
        free, _ = torch.cuda.mem_get_info()
    fit = int(share * free / max(1, lanes * nodes * bytes_per_edge))
    return max(48, min(218, fit))


TOWER_ROUND = 592          # positions one round of the persistent tower kernel covers: 74 CTA pairs x 8 boards (DESIGN 3.1)


def default_lanes(n_games):
    """Lanes for a finite run when --lanes is not given.  Two effects pull in opposite directions: a finished game's lane
    is refilled only while games are left, so few games per lane means a long drain at low occupancy (one game per lane:
    ~50 %, four: ~78 %, sixteen: ~94 % -- game lengths have a long tail); and the tower is most efficient on batches that
    are multiples of one round of its persistent grid.  Rule: about four games per lane, a whole number of tower rounds,
    at most seven rounds (4,144 lanes, where the step is tensor-bound anyway); small runs take one lane per game."""
    if n_games <= TOWER_ROUND:
        return max(1, n_games)
    return min(7 * TOWER_ROUND, max(TOWER_ROUND, (n_games // 4) // TOWER_ROUND * TOWER_ROUND))


class LockstepRun:
    """The many-games form of selfplay.py's game loop (selfplay.py:142-163) on one GPU: `lanes` games advance in
    lockstep, a lane whose game ends is refilled with the next game at once (per-GPU slot refill, SURVEY.md 8e) and
    parked when none is left.  n_games=None means an unbounded supply (steady-state measurements: bench.py).

    advance() = harvest finished games -> refill / park their lanes -> one lockstep move for every running game.
    """

    def __init__(self, model, n_games, sims=900, lanes=None, noise=True, device=None, seed=None, max_moves=None,
                 threads=1, evaluator=None, engine=None, reuse=True, net_precision="bf16"):
        import time
        from ._lib import EVAL_HASH, EVAL_NET
        from .engine import Engine
        from .lockstep import LockstepSelfPlay
        self.n_games = n_games
        if lanes is None:
            if n_games is None:
                raise ValueError("an unbounded run needs an explicit lane count")
            lanes = n_games
        self.lanes = lanes = max(1, lanes if n_games is None else min(lanes, n_games))
        self.sims = sims
        threads = max(1, min(int(threads), 64))
        self._own_engine = engine is None
        self.eng = engine if engine is not None else Engine(
            max_games=lanes, max_nodes=sims + 1, device=device, max_inflight=threads,
            avg_moves=edge_slots_per_node(lanes, sims + 1, device, bytes_per_edge=32 if reuse and threads == 1 else 24))
        if evaluator is None:
            if model is not None:
                self.eng.load_weights(model.weights, precision=net_precision)
            elif net_precision != "bf16":
                self.eng.set_net_precision(net_precision)
            self.eng.set_evaluator(EVAL_NET)
        else:
            self.eng.set_evaluator(EVAL_HASH, int(evaluator[1]), int(evaluator[2]))
        self._rng = random.Random(seed)
        self._colors = []                                  # colour of game i, drawn like selfplay.py:62
        # reuse: evaluations of the previous move's search are looked up instead of run again (crl_set_reuse): the games
        # are the same move for move, the network runs less often
        self.sp = LockstepSelfPlay(self.eng, n_games=lanes, sims=sims, noise=noise, inflight=threads, reuse=reuse)
        # the engine's move lists hold 2,048 plies per game: a game that gets there is stored unfinished instead of
        # failing the whole run (the fifty-move claim ends games long before that in practice)
        self.cap = 2040 if max_moves is None else min(2040, 2 * max_moves)
        self.records = []                                  # (moves, colour) by game index; None while running
        self.lane_game = list(range(lanes))
        self.next_game = lanes
        self.steps = 0
        self.refills = 0
        self.finished_games = 0
        self._time = time
        self.t0 = time.perf_counter()
        self.c0 = self.eng.counters()
        self._started = False

    def _color(self, game):
        while len(self._colors) <= game:
            self._colors.append(self._rng.random() >= 0.5)
        return self._colors[game]

    def _record(self, game, moves, color):
        while len(self.records) <= game:
            self.records.append(None)
        self.records[game] = (moves, color)

    def start(self, start_records=None, move_lists=None):
        """First fill of the lanes: games 0..lanes-1 (optionally from given prefixes: staggered phases for benchmarks)."""
        self.sp.start(colors=[self._color(g) for g in range(self.lanes)], start_records=start_records, move_lists=move_lists)
        self._started = True

    def advance(self):
        """Returns False once no game is running (a bounded run is then complete)."""
        if not self._started:
            self.start()
        again, parked = [], []
        for lane, moves, result, color in self.sp.harvest(max_plies=self.cap):
            self._record(self.lane_game[lane], moves, color)
            self.finished_games += 1
            if self.n_games is None or self.next_game < self.n_games:
                self.lane_game[lane] = self.next_game
                again.append(lane)
                self.next_game += 1
            else:
                parked.append(lane)
        self.sp.restart(again, [self._color(self.lane_game[g]) for g in again])   # one batched refill + one opening eval
        self.refills += len(again)
        self.sp.retire(parked)
        if not self.sp.running().any():
            return False
        self.sp.step()
        self.steps += 1
        return True

    def stats(self):
        c1 = self.eng.counters()
        sims = c1["simulations"] - self.c0["simulations"]
        return {"steps": self.steps, "moves": self.sp.moves_played, "seconds": self._time.perf_counter() - self.t0,
                "simulations": sims, "evaluations": c1["evaluations"] - self.c0["evaluations"],
                "reused_evaluations": c1.get("reused_evaluations", 0) - self.c0.get("reused_evaluations", 0), "lanes": self.lanes,
                "games_finished": self.finished_games, "refills": self.refills,
                "lane_occupancy": sims / max(1, self.steps * self.lanes * self.sims)}

    def close(self):
        if self._own_engine:
            self.eng.close()

    def dataset(self):
        out = DatasetGame()
        for rec in self.records:
            if rec is None:
                continue
            moves, color = rec
            gm = Game(player_color=color)
            gm._sync(extra=[B.move_to_uci(m) for m in moves])
            out.append(gm)
        return out


def play_games_lockstep(model, n_games, sims=900, lanes=None, noise=True, device=None, seed=None, max_moves=None,
                        threads=1, evaluator=None, stats=None, reuse=True, net_precision="bf16"):
    """`n_games` games in lockstep, `lanes` at a time; returns a DatasetGame in game-start order.

    The per-move host work is the numpy move policy only.  max_moves caps the agent moves of a game (it is then stored
    unfinished, result None).  evaluator: None = the network with `model`'s weights; ("hash", seed, bits) = the
    deterministic test evaluator.  stats: optional dict that receives steps / moves / simulations / seconds / lane
    occupancy of the run.  reuse: take evaluations from the previous move's tree where it holds the same node (same
    games either way; include/chessrl_b200.h crl_set_reuse).  net_precision: "bf16" (default) or "fp8", the opt-in e4m3
    tower calibrated on model.calibration_planes (DESIGN.md section 3.1; not bit-exact with bf16)."""
    run = LockstepRun(model, n_games, sims=sims, lanes=lanes, noise=noise, device=device, seed=seed, max_moves=max_moves,
                      threads=threads, evaluator=evaluator, reuse=reuse, net_precision=net_precision)
    try:
        while run.advance():
            pass
        if stats is not None:
            stats.update(run.stats())
    finally:
        run.close()
    return run.dataset()


def main(argv=None):
    parser = argparse.ArgumentParser(description="Plays some chess games, stores the result and trains a model.")
    parser.add_argument('model_dir', metavar='modeldir', help="where to store (and load from) the trained model and the logs")
    parser.add_argument('--games', metavar='games', type=int, default=1)
    parser.add_argument('--threads', metavar='threads', type=int, default=1,
                        help="MCTS simulations in flight per game (reference default 6; 1 = its deterministic schedule)")
    parser.add_argument('--debug', action='store_true', default=False, help="Log debug messages on screen. Default false.")
    parser.add_argument('--sims', type=int, default=900, help="MCTS simulations per move (reference: 900)")
    parser.add_argument('--lanes', type=int, default=None,
                        help="games stepped in lockstep per GPU (default: about four games per lane in whole tower rounds)")
    parser.add_argument('--max-moves', type=int, default=None, help="cap on the agent's moves per game (stored unfinished)")
    parser.add_argument('--no-train', action='store_true', default=False)
    parser.add_argument('--no-reuse', action='store_true', default=False,
                        help="evaluate every position of every search (default: evaluations of the previous move's "
                             "search are reused; the games are identical either way)")
    parser.add_argument('--precision', choices=("fp32", "tf32", "bf16"), default=None,
                        help="arithmetic of the training step (default fp32 = the parity setting; see chessrl_b200/training.py)")
    parser.add_argument('--net-precision', choices=("bf16", "fp8"), default="bf16",
                        help="arithmetic of the network's residual tower during self-play (default bf16; fp8 = e4m3 "
                             "tensor cores with calibrated scales, faster but not bit-exact: DESIGN.md section 3.1)")
    args = parser.parse_args(argv)
    if args.precision:
        os.environ["CRL_TRAIN_PRECISION"] = args.precision

    logger = Logger.get_instance()
    logger.set_level(0 if args.debug else 1)
    os.makedirs(args.model_dir, exist_ok=True)
    model_path = get_model_path(args.model_dir)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    import torch
    torch.cuda.set_device(local_rank)
    agent = Agent(True, weights=model_path if os.path.exists(model_path) else None)
    if world > 1:
        from . import sharding
        sharding.init()
        sharding.broadcast_weights(agent.model)
    share = args.games // world + (1 if rank < args.games % world else 0)
    logger.info("rank %d/%d plays %d game(s), %d simulations per move" % (rank, world, share, args.sims))
    stats = {}
    lanes = args.lanes if args.lanes is not None else default_lanes(share)
    data = (play_games_lockstep(agent.model, share, sims=args.sims, lanes=lanes, device=local_rank,
                                threads=args.threads, max_moves=args.max_moves, stats=stats,
                                reuse=not args.no_reuse, net_precision=args.net_precision) if share else DatasetGame())
    if stats:
        full = max(1, stats["steps"] * stats["lanes"] * args.sims)
        logger.info("rank %d: %d games, %d agent moves in %d lockstep steps, %.1f s: %.0f simulations/s, lane occupancy %.1f %%"
                    % (rank, len(data), stats["moves"], stats["steps"], stats["seconds"],
                       stats["simulations"] / max(stats["seconds"], 1e-9), 100.0 * stats["simulations"] / full))
    if world > 1:
        from . import sharding
        data = sharding.gather_games(data)
    if rank == 0:
        data.save(os.path.join(args.model_dir, "gameplays.json"))
        if not args.no_train:
            # The reference trains after EVERY game in a fresh process -- Agent(True, model_path), i.e. a new Adam state,
            # one epoch over that one game (selfplay.py:98-108, 155-162) -- while its PredictWorker keeps the starting
            # weights for the whole run (reload_model is never called).  Playing all games first with the starting
            # weights and then training game by game, each with a fresh optimizer, gives the same sequence of updates.
            for i, g in enumerate(data.games):
                logger.info("\tTraining %d of %d" % (i + 1, len(data)))
                agent.train(DatasetGame([g]), logdir=args.model_dir, epochs=1, validation_split=0, batch_size=1)
            agent.save(model_path)
    if world > 1:
        from . import sharding
        sharding.shutdown()


if __name__ == "__main__":
    main()
