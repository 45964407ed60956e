"""The oracle's network evaluator for the real-network search parity tests.

The oracle trees (chessrl_oracle.OSelfPlayTree) run in threads, one per game; their evaluation requests are served in
one crl_net_forward batch whenever every live thread is waiting.  Positions are encoded by the oracle's own netencoder
restatement, so the engine and the oracle see bit-identical policy / value numbers iff the engine's encoder, history
walk, move generator, reply selection and tree logic agree with the reference's (and the network's rows do not depend
on the batch they are evaluated in -- test_gpu_evalpath.py)."""
import threading

import numpy as np
import torch

import chessrl_oracle as O


class BatchedNetEvaluator:
    """evaluate(game) -> (policy float32[1968], float32 value) for OAgent; the numbers come from crl_net_forward."""

    def __init__(self, engine, n_threads):
        self.e = engine
        self.live = n_threads
        self.cv = threading.Condition()
        self.pending = []
        self.gen = 0
        self.rows = 0                       # positions evaluated so far

    def _flush(self):
        games = [g for g, _ in self.pending]
        planes = np.stack([O.planes(g) for g in games]).astype(np.float32)
        x = torch.zeros(len(games), 8, 8, 128, dtype=torch.bfloat16, device=self.e.device)
        x[..., :127] = torch.from_numpy(planes).to(self.e.device).to(torch.bfloat16)
        p, v = self.e.net_forward(x)
        p, v = p.cpu().numpy(), v.cpu().numpy()
        for i, (_, slot) in enumerate(self.pending):
            slot.append((p[i].copy(), np.float32(v[i])))
        self.rows += len(games)
        self.pending = []
        self.gen += 1
        self.cv.notify_all()

    def __call__(self, game):
        slot = []
        with self.cv:
            self.pending.append((game, slot))
            if len(self.pending) >= self.live:
                self._flush()
            else:
                gen = self.gen
                while self.gen == gen:
                    self.cv.wait()
        return slot[0]

    def done(self):
        with self.cv:
            self.live -= 1
            if self.live > 0 and len(self.pending) >= self.live:
                self._flush()


def run_oracle_threads(evaluator, n, worker):
    """worker(i) for i < n, each in its own thread, with evaluator.done() after each; returns [(i, repr(exc))]."""
    failures = []

    def body(i):
        try:
            worker(i)
        except BaseException as exc:            # noqa: BLE001 - reported by the caller from the main thread
            failures.append((i, repr(exc)))
        finally:
            evaluator.done()

    threads = [threading.Thread(target=body, args=(i,)) for i in range(n)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    return failures
