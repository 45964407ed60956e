#!/bin/bash
# Round 2, after the fused backup/select head, the statistics-only softmax and the 64-thread row encoder:
# all GPU parity tests, the bench (share_of_step_ms per kernel class), an ncu launch list of a short step.
mkdir -p gpurun_out
T0=$SECONDS
timeout 600 python -m pytest tests -m gpu -q -x --timeout 300 > gpurun_out/pytest_gpu.log 2>&1; echo "== pytest -m gpu: $? at $((SECONDS-T0)) s"; tail -4 gpurun_out/pytest_gpu.log
timeout 60 python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke.log 2>&1; echo "== smoke: $? at $((SECONDS-T0)) s"; tail -1 gpurun_out/smoke.log
timeout 300 python bench.py --steps 5 --warmup 3 --no-cpu-baseline --no-perft --no-kernels --no-large > gpurun_out/bench_sixth.log 2> gpurun_out/bench_sixth.err; echo "== bench: $? at $((SECONDS-T0)) s"
python - <<'PY'
import json
for f in ("bench_sixth",):
    try:
        d = json.loads(open("gpurun_out/%s.log" % f).read().strip().splitlines()[-1])
        print(f, "value", round(d["value"]), "e2e", round(d["e2e"]["value"]), d["clocks"], d["roofline"]["share_of_step_ms"], "launches", d["gpu_launches"])
        for k in ("whole_games", "whole_games_reuse"):
            w = d.get(k)
            if w: print(" ", k, round(w["simulations_per_s"]), w["evaluations_per_simulation"], w.get("reused_evaluations_per_simulation"))
    except Exception as ex:
        print("ERR", f, ex); print(open("gpurun_out/%s.err" % f).read()[-2500:])
PY
S="--no-cpu-baseline --no-perft --no-kernels --no-whole-games --no-large"
CRL_NO_GRAPH=1 timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -s 200 -c 400 --csv --log-file gpurun_out/launches_sixth.csv \
   python bench.py --games 4096 --sims 12 --steps 1 --warmup 1 $S > gpurun_out/ncu_sixth.log 2>&1; echo "== ncu launch list: $? at $((SECONDS-T0)) s"
python scripts/ncu_summarise.py launches gpurun_out/launches_sixth.csv | tail -20
