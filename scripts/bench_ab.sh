#!/usr/bin/env bash
# A/B bench of two builds on one GPU, alternating so that both see the same machine state:
#   scripts/bench_ab.sh OTHER_TREE [OUT_DIR] [ROUNDS]
# OTHER_TREE is a second checkout (e.g. `git archive <base> | tar -x -C DIR`) with its library built.
# Per round and build: the default bench line (without the CPU baseline) and its result columns
# (--dump-outputs), then once per build the SF10 join workload. Output: OUT_DIR/{base,this}{i}.json,
# OUT_DIR/dump_{base,this}{i}/, OUT_DIR/joins_{base,this}.jsonl and the card's name and power limit.
set -u
OTHER=$(cd "$1" && pwd)
THIS=$(cd "$(dirname "$0")/.." && pwd)
O=$(mkdir -p "${2:-${TMPDIR:-/tmp}/bench_ab}" && cd "${2:-${TMPDIR:-/tmp}/bench_ab}" && pwd)
ROUNDS=${3:-2}
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$O/gpu.txt" 2>&1
for i in $(seq 1 "$ROUNDS"); do
    for side in base this; do
        tree=$THIS; [ $side = base ] && tree=$OTHER
        (cd "$tree" && timeout 900 python bench.py --no-cpu --dump-outputs "$O/dump_$side$i" > "$O/$side$i.json" 2> "$O/$side$i.err")
        echo "bench $side$i rc=$?"
    done
done
for side in base this; do
    tree=$THIS; [ $side = base ] && tree=$OTHER
    (cd "$tree" && timeout 900 python bench.py --workload joins --sf 10 > "$O/joins_$side.jsonl" 2> "$O/joins_$side.err")
    echo "joins $side rc=$?"
done
