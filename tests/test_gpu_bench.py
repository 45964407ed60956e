"""bench.py --dump-outputs: the arrays of the last timed step, in float32 / float64, identical from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

GAMES, SIMS = 16, 8
NAMES = {"visits", "values", "priors", "moves", "replies", "results", "n_children", "root_visits", "root_values",
         "e2e_picks", "e2e_chosen", "lanes"}


def _bench(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
           "--games", str(GAMES), "--sims", str(SIMS), "--no-cpu-baseline", "--no-perft", "--no-kernels",
           "--no-whole-games", "--no-large", "--no-training", "--dump-outputs", str(out_dir)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    return {n[:-4]: np.load(os.path.join(out_dir, n)) for n in os.listdir(out_dir)}


def test_dump_outputs_are_complete_and_reproducible(tmp_path):
    a = _bench(tmp_path / "a")
    b = _bench(tmp_path / "b")
    assert set(a) == NAMES and set(b) == NAMES
    assert sum(v.nbytes for v in a.values()) <= 64 * 10 ** 6
    for k in NAMES:
        assert a[k].dtype in (np.float32, np.float64), k
        assert a[k].shape[0] == GAMES, k
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert (a["lanes"] == np.arange(GAMES)).all()
    live = a["n_children"] > 0
    assert live.any()
    assert (a["root_visits"][live] == SIMS + 1).all() and (a["visits"][live].sum(1) == SIMS).all()
    assert ((a["e2e_picks"] >= -1) & (a["e2e_picks"] < np.maximum(a["n_children"], 1))).all()
