#!/bin/bash
# Round 2, second GPU call: two-phase tree kernels, L2 eviction hints, one-block first perft plies, fresh rule-kernel ncu
mkdir -p gpurun_out
T0=$SECONDS
timeout 900 python -m pytest tests -m gpu -q --timeout 300 -x > gpurun_out/pytest_gpu.log 2>&1; echo "== pytest -m gpu: $? at $((SECONDS-T0)) s"; tail -8 gpurun_out/pytest_gpu.log
S="--no-cpu-baseline --no-perft --no-kernels --no-whole-games --no-large"
timeout 300 python bench.py --steps 4 --warmup 3 $S > gpurun_out/bench_hints_on.log 2>&1; echo "== hints on: $?"
timeout 300 python bench.py --games 512 --sims 200 --steps 4 --warmup 3 $S > gpurun_out/bench_512x200.log 2>&1; echo "== 512 lanes: $?"
python - <<'PY'
import json
for f in ("hints_on", "512x200"):
    try:
        d = json.loads(open("gpurun_out/bench_%s.log" % f).read().strip().splitlines()[-1])
        print(f, "value", round(d["value"]), "e2e", round(d["e2e"]["value"]), "roof", round(d["roofline"]["achieved"]), d["roofline"]["share_of_step_ms"], d["clocks"])
    except Exception as ex:
        print(f, "ERR", ex); print(open("gpurun_out/bench_%s.log" % f).read()[-2000:])
PY
timeout 300 python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-whole-games --no-large > gpurun_out/bench_perft.log 2>&1; echo "== perft + kernels: $? at $((SECONDS-T0)) s"
python - <<'PY'
import json
try:
    d = json.loads(open("gpurun_out/bench_perft.log").read().strip().splitlines()[-1])
    p = d["perft"]
    print("perft start", p["start"]["ms"], round(p["start"]["nodes_per_s"] / 1e9, 1), "kiwi", p["kiwipete"]["ms"], round(p["kiwipete"]["nodes_per_s"] / 1e9, 1), "both", round(p["nodes_per_s"] / 1e9, 1), "deep", round(p["deep_nodes_per_s"] / 1e9, 1))
    print("movegen", round(d["kernels"]["movegen"]["boards_per_s"] / 1e9, 2), "G boards/s frac", round(d["kernels"]["movegen"]["frac"], 3))
except Exception as ex:
    print("ERR", ex); print(open("gpurun_out/bench_perft.log").read()[-2000:])
PY
timeout 300 python scripts/perft_probe.py --time > gpurun_out/perft_probe.log 2>&1; echo "== probe $?"; cat gpurun_out/perft_probe.log
B="--games 4096 --sims 6 --steps 1 --warmup 1 $S"
timeout 600 ncu --metrics gpu__time_duration.sum --clock-control none -k regex:'^k_' -c 900 --csv --log-file gpurun_out/launches_step_r02b.csv \
   python bench.py $B > gpurun_out/ncu_launches_r02b.log 2>&1; echo "== launch list: $? at $((SECONDS-T0)) s"
CRL_NO_GRAPH=1 timeout 600 ncu --set full --clock-control none --import-source on -k regex:k_trunk4 -s 4 -c 2 -o gpurun_out/prof_trunk_r02b \
   python bench.py $B > gpurun_out/ncu_trunk_r02b.log 2>&1; echo "== trunk4 full: $? at $((SECONDS-T0)) s"
timeout 900 ncu --set full --clock-control none --import-source on -k regex:'k_(movegen|perft|bfs_ply)' -c 10 -o gpurun_out/prof_rules_r02 python scripts/perft_probe.py > gpurun_out/ncu_rules_r02.log 2>&1; echo "== ncu rules $? at $((SECONDS-T0)) s"
CRL_NO_GRAPH=1 timeout 600 ncu --set full --clock-control none --import-source on -k regex:'k_(select_expand|reply|finalize)$' -s 6 -c 6 -o gpurun_out/prof_tree_r02 \
   python bench.py $B > gpurun_out/ncu_tree_r02.log 2>&1; echo "== tree full: $? at $((SECONDS-T0)) s"
ls -la gpurun_out | tail -14
