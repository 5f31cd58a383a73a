#!/usr/bin/env bash
# Same-box A/B of two library builds _ab/lib_<a>.so and _ab/lib_<b>.so (git-ignored; build them first):
#   bash profiles/tapn_ab.sh old new [bench_runs_per_build] [output_dir]
# prints the card and its power limit, then alternates the builds: profiles/tapn_bench.py twice per build, then bench.py
# (default C2 workload) bench_runs_per_build times per build.  Results go to output_dir (default: a new temporary directory).
# The built library is restored at the end.
set -euo pipefail
a=${1:?variant A}; b=${2:?variant B}; runs=${3:-4}; out=${4:-$(mktemp -d)}
mkdir -p "$out"; echo "results: $out"
cp heal_b200/libheal_b200.so "$out/.lib_saved.so"
trap 'cp "$out/.lib_saved.so" heal_b200/libheal_b200.so; rm -f "$out/.lib_saved.so"' EXIT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$out/card.txt"
for v in "$a" "$b" "$a" "$b"; do
    cp "_ab/lib_${v}.so" heal_b200/libheal_b200.so
    python profiles/tapn_bench.py "$v" | tee -a "$out/kernel.jsonl"
done
for i in $(seq 1 "$runs"); do
    for v in "$a" "$b"; do
        cp "_ab/lib_${v}.so" heal_b200/libheal_b200.so
        python bench.py --gpus 1 > "$out/bench_${v}_${i}.json" 2> "$out/bench_${v}_${i}.err"
        echo "== ${v} run ${i}: $(python -c "import json,sys; d=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); print(d['value'], d['latency']['single_frame_ms'], d.get('parity',{}).get('pass'))" "$out/bench_${v}_${i}.json")"
    done
done
