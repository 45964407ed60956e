"""Multi-process path on CPU (gloo, world_size 2): shard ranges, weight broadcast, finished-game gather."""
import os
import socket
import subprocess
import sys
import textwrap

from conftest import ROOT

WORKER = textwrap.dedent("""
    import os, sys, json
    sys.path.insert(0, %r)
    import numpy as np
    import torch.distributed as dist
    from chessrl_b200 import sharding, model
    sharding.init("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    lo, hi = sharding.shard_range(11)
    m = model.ChessModel(seed=rank)              # different weights per rank before the broadcast
    sharding.broadcast_weights(m)
    ref = model.ChessModel(seed=0)
    same = all(np.array_equal(a, b) for a, b in zip(m.weights, ref.weights))
    words = [[(rank * 100 + g) * 1 + k for k in range(3 + g)] for g in range(2 + rank)]
    packed = sharding.pack_games(words, [1 if rank == 0 else None] * len(words), [bool(rank)] * len(words))
    got = sharding.gather_packed(*packed)
    lanes = np.arange(1000, dtype=np.int64) ** 2 %% 977           # per-board node counts of a perft frontier
    total = sharding.sum_counts(lanes[rank::world])               # board i -> rank i mod world, one all_reduce(sum)
    out = {"rank": rank, "range": [lo, hi], "same": bool(same), "perft_total": total}
    if rank == 0:
        out["gathered"] = [[list(map(int, mv)), res, col] for mv, res, col in got]
    with open(os.path.join(%r, "rank%%d.json" %% rank), "w") as f:    # one file per rank: stdout of two ranks interleaves
        json.dump(out, f)
    dist.destroy_process_group()
""")


def _free_port():
    """A loopback port nobody holds right now: a fixed one may be taken by another job on a shared host."""
    with socket.socket(socket.AF_INET, socket.SOCK_STREAM) as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER % (ROOT, str(tmp_path)))
    port = str(_free_port())
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=port)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", port, str(script)]
    p = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=240)
    assert p.returncode == 0, p.stderr[-2000:]
    import json
    res = {}
    for rank in (0, 1):
        with open(tmp_path / ("rank%d.json" % rank)) as f:
            res[rank] = json.load(f)
        assert res[rank]["rank"] == rank
    assert res[0]["range"] == [0, 6] and res[1]["range"] == [6, 11]
    assert res[0]["same"] and res[1]["same"]
    import numpy as np
    want = int((np.arange(1000, dtype=np.int64) ** 2 % 977).sum())
    assert res[0]["perft_total"] == want and res[1]["perft_total"] == want
    g = res[0]["gathered"]
    assert len(g) == 2 + 3                                  # rank 0 sent 2 games, rank 1 sent 3, in rank order
    assert g[0][0] == [0, 1, 2] and g[1][0] == [1, 2, 3, 4]
    assert g[2][0] == [100, 101, 102] and g[4][0] == [102, 103, 104, 105, 106]
    assert [x[1] for x in g] == [1, 1, 2, 2, 2] and [x[2] for x in g] == [False, False, True, True, True]
