#!/bin/bash
# Step 0 of the one-read-per-sweep pass: correctness of the probe's two MMAs at small ragged shapes, then the time of
# one skeleton pass at config-3 shape (200 000 x 20 000 fp16, k = 64) over slice widths, lags and stage rings.
# Writes <out>/onepass_probe.jsonl and <out>/onepass_probe.log (default <out>: build/onepass_probe_out).
# Build first:  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o build/onepass_probe tools/onepass_probe.cu -lcuda
set -u -o pipefail
OUT=${1:-build/onepass_probe_out}
mkdir -p $OUT
LOG=$OUT/onepass_probe.log
J=$OUT/onepass_probe.jsonl
: > $J
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm,clocks.mem --format=csv | tee $LOG
build/onepass_probe verify 2>&1 | tee -a $LOG || exit 1
N=200000; D=20000; IT=20
t() { build/onepass_probe time $N $D "$@" $IT ${RINGS:-} | tee -a $J; }
# one shared ring (first reads and re-reads in one FIFO), as many stages as fit
for cfg in "512 3" "640 4" "768 5"; do
    set -- $cfg
    t $1 $2 0 0 0
    for L in 1 2 4 8; do t $1 $2 $L 0 1 || exit 1; done
done
# first reads and re-reads in separate rings fed by separate producer warps: "w R sa sb"
for cfg in "512 3 2 2" "384 2 2 2" "384 2 3 1" "640 4 2 1" "256 1 3 2"; do
    set -- $cfg
    RINGS="$3 0" t $1 $2 0 0 0
    for L in 1 2 4; do RINGS="$3 $4" t $1 $2 $L 0 1 || exit 1; done
done
# with the partials' reduction (one pass of the epilogue warps over 1/P of a tile's rows)
RINGS="2 2" t 512 3 2 1 1
nvidia-smi --query-gpu=name,power.limit,clocks.sm,clocks.mem --format=csv | tee -a $LOG
