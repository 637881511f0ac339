#!/bin/bash
# Dependent global-load round trips on the card (tools/micro/latency.cu), with the card's name and power limit.
# Build first (no GPU needed): nvcc -O3 -gencode arch=compute_100a,code=sm_100a tools/micro/latency.cu -o tools/micro/latency
# Result: $OUT_DIR/k1_latency_probe.txt (default: build/, which git ignores).
mkdir -p "${OUT_DIR:-build}"
out=${OUT_DIR:-build}/k1_latency_probe.txt
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > "$out"
tools/micro/latency >> "$out" 2>&1
rc=$?
cat "$out"
exit $rc
