"""CPU study (PyTorch, no GPU): how far the opt-in fp8 tower (DESIGN.md section 3.1) moves the network's outputs.

For each pack, the fp8-emulated graph (tests/fp8_emu.py, the numeric definition the GPU tests hold the kernel to) and the
bf16-emulated graph (oracle/model_torch.forward(emulate_bf16_activations=True), today's tower) are compared with the fp32
graph on the same positions: policy and value max |d|, value mean |d|, and how often the legal-masked policy argmax (the
move AgentDistributed.best_move would play) is the fp32 graph's.  fp8 is calibrated the way Engine.load_weights does it by
default, but on the positions themselves: amax_L = max |output| of convolution L of the bf16-emulated graph.
Packs: netpacks.lively_pack() (the GPU tests' pack, very sensitive) and model.random_pack(1, perturb_bn=True) (the
perturbed pack of winograd_numerics.py).  Writes profiles/r03_fp8_numerics.txt (or the path in argv[1])."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import chessrl_oracle as O  # noqa: E402
import fp8_emu  # noqa: E402
import model_torch  # noqa: E402
import netpacks  # noqa: E402
from chessrl_b200 import model  # noqa: E402

N = int(os.environ.get("N", "64"))


def legal_argmax(policy, games):
    idx = O.label_index()
    out = []
    for p, g in zip(policy.numpy(), games):
        legal = [idx[m] for m in (str(x) for x in g.get_legal_moves()) if m in idx]
        out.append(legal[int(np.argmax(p[legal]))] if legal else -1)
    return np.asarray(out)


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    games = netpacks.midgame_games(N, seed=0)
    planes = netpacks.planes_of(games)
    lines = ["fp8 numerics study: %d midgame positions (netpacks.midgame_games(%d, seed=0)), CPU, errors against the "
             "fp32 graph" % (N, N)]
    for name, pack in (("lively pack (netpacks.lively_pack)", netpacks.lively_pack()),
                       ("perturbed pack (model.random_pack(1, perturb_bn=True))", model.random_pack(1, perturb_bn=True))):
        with torch.no_grad():
            p32, v32 = model_torch.forward(pack, planes)
            taps = {}
            p16, v16 = model_torch.forward(pack, planes, emulate_bf16_activations=True, taps=taps)
            amax = [float(a.abs().max()) for a in taps["act"]]
            p8, v8 = fp8_emu.forward(pack, planes, amax)
        best = legal_argmax(p32, games)
        lines.append("== %s" % name)
        for label, (p, v) in (("bf16-emulated", (p16, v16)), ("fp8-emulated", (p8, v8))):
            agree = float(np.mean(legal_argmax(p, games) == best))
            lines.append("  %-14s policy max|d| %.2e  value max|d| %.2e  value mean|d| %.2e  legal argmax agreement %.3f"
                         % (label, (p - p32).abs().max().item(), (v - v32).abs().max().item(), (v - v32).abs().mean().item(),
                            agree))
    text = "\n".join(lines)
    print(text)
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r03_fp8_numerics.txt")
    with open(out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
