"""BASELINE config 4 parity: lockstep self-play with the REAL network (tcgen05 kernels) against the oracle
SelfPlayTree(threads=1) fed the SAME network outputs -- visit counts, value sums and chosen moves must match
bit-exactly for every sampled game over its first moves.

"Same network outputs" is obtained without any tolerance: the oracle's evaluator encodes the position with the
oracle's own netencoder restatement, and runs it through crl_net_forward (whose rows are independent of batch
composition, see test_gpu_net.py), so both sides see bit-identical policy / value numbers iff the engine's encoder,
history walk, move generator, reply selection and tree logic all agree with the reference's.

Default size keeps the GPU suite short (64 games x 4 moves x 48 sims); CRL_PARITY_SIMS=200 runs BASELINE's size.
"""
import os
import random
import threading

import numpy as np
import pytest

import chessrl_oracle as O
from chessrl_b200 import boards as B
from chessrl_b200 import model
from chessrl_b200._lib import EVAL_NET
from chessrl_b200.engine import Engine
from chessrl_b200.lockstep import compute_policy
from net_oracle import BatchedNetEvaluator

pytestmark = pytest.mark.gpu


def test_lockstep_real_network_matches_oracle_visit_counts():
    n_games = int(os.environ.get("CRL_PARITY_GAMES", "64"))
    n_moves = int(os.environ.get("CRL_PARITY_MOVES", "4"))
    sims = int(os.environ.get("CRL_PARITY_SIMS", "48"))
    import netpacks
    pack = netpacks.lively_pack()          # live value head: with Keras-default init the value is 0.0 for every position
    eng = Engine(max_games=n_games, max_nodes=sims + 1, avg_moves=96)
    eng.load_weights(pack)
    eng.set_evaluator(EVAL_NET)
    net = Engine(max_games=n_games, max_nodes=8)          # serves the oracle's evaluations
    net.load_weights(pack)

    rng = random.Random(3)
    starts = []
    for g in range(n_games):
        og = O.OGame()
        for _ in range(rng.randrange(0, 24)):
            og.move(rng.choice(og.get_legal_moves()))
        starts.append([m.uci() for m in og.board.move_stack])
    eng.games_set(np.tile(B.record_from_fen(), (n_games, 1)), [[B.uci_to_move(m) for m in s] for s in starts])

    # ---- engine: n_moves lockstep searches, statistics recorded after each ----
    recorded = []
    for mv in range(n_moves):
        eng.mcts_begin_move()
        eng.mcts_simulate(sims)
        st = eng.root_stats()
        _, plies, results = eng.games_get(0, n_games)
        picks = np.full(n_games, -1, dtype=np.int32)
        for g in range(n_games):
            k = int(st["n_children"][g])
            if results[g] == B.RESULT_NONE and k:
                picks[g] = int(np.argmax(compute_policy(st["visits"][g, :k], st["root_visits"][g], int(plies[g]), False)))
        out = eng.commit(picks, apply=True)
        recorded.append((st, picks.copy(), out.copy()))

    # the value head must be alive, or "value sums match" would be 0.0 == 0.0 and Q would never steer a visit
    mean_q = []
    for st, _, _ in recorded:
        for g in range(n_games):
            k = int(st["n_children"][g])
            if k:
                mean_q.extend(st["values"][g, :k] / np.maximum(st["visits"][g, :k], 1))
    mean_q = np.asarray(mean_q)
    assert mean_q.max() - mean_q.min() > 0.1 and np.count_nonzero(mean_q) > 0.9 * mean_q.size, (mean_q.min(), mean_q.max())

    # ---- oracle: the same games, one thread each, evaluations batched through crl_net_forward ----
    ev = BatchedNetEvaluator(net, n_games)
    failures = []

    def worker(g):
        try:
            og = O.OGame()
            for m in starts[g]:
                og.move(m)
            agent = O.OAgent(ev)
            for mv in range(n_moves):
                st, picks, out = recorded[mv]
                if og.get_result() is not None:
                    assert picks[g] == -1
                    continue
                tree = O.OSelfPlayTree(og)
                ret = tree.search_move(agent, max_iters=sims, noise=False, ai_move=True)
                kids = tree.root.children
                assert int(st["n_children"][g]) == len(kids)
                assert [c.visits for c in kids] == list(st["visits"][g, :len(kids)])
                assert [float(c.value) for c in kids] == [float(x) for x in st["values"][g, :len(kids)]]
                assert float(tree.root.value) == float(st["root_values"][g])
                assert [B.move_to_uci(out[g, 0]), B.move_to_uci(out[g, 1])] == list(ret)
                og.move(ret[0])
                og.move(ret[1])
        except BaseException as exc:            # noqa: BLE001 - report from the main thread
            failures.append((g, repr(exc)))
        finally:
            ev.done()

    threads = [threading.Thread(target=worker, args=(g,)) for g in range(n_games)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    eng.close()
    net.close()
    assert not failures, failures[:3]
