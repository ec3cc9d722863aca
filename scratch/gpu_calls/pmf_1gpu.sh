#!/bin/bash
# ProbabilisticMF on one B200, outputs under the directory given as $1 (default: out): the whole GPU suite, smoke(),
# bench.py's headline leg, bench_pmf.py at C2 with the sgd_strata sweep that chose the default (DESIGN.md 3.6; its JSON
# line is profiles/bench_pmf_c2.json) and bench_pmf.py's CPU reference arm
OUT=${1:-out}
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/build.log" 2>&1 || tail -20 "$OUT/build.log"
timeout 1500 python -m pytest tests -q -m gpu > "$OUT/tests_gpu.log" 2>&1
tail -4 "$OUT/tests_gpu.log" | cut -c1-400
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
timeout 600 python bench.py --gpus 1 --steps 5 --warmup 3 --no-cpu-baseline > "$OUT/bench_c2.json" 2> "$OUT/bench_c2.err"
tail -1 "$OUT/bench_c2.json" | cut -c1-600
timeout 900 python bench_pmf.py --steps 5 --warmup 1 --epochs 3 --sweep 256,512,1024,2048,4096 \
    > "$OUT/bench_pmf_c2.json" 2> "$OUT/bench_pmf_c2.err"
tail -3 "$OUT/bench_pmf_c2.err" | cut -c1-400
cut -c1-1200 "$OUT/bench_pmf_c2.json"
timeout 900 python bench_pmf.py --impl reference > "$OUT/bench_pmf_c2_reference.json" 2>&1
tail -2 "$OUT/bench_pmf_c2_reference.json" | cut -c1-600
