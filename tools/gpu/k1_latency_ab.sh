#!/bin/bash
# A/B of K1's latency-hiding paths on one GPU: the default bench line against `--opt k1_prefetch=0` (the plain paths, same bits),
# alternating, REPS times each, all in one run; the card's name and power limit are recorded with the lines.
#   tools/gpu/k1_latency_ab.sh [REPS] [OTHER_TREE]
# OTHER_TREE (optional): a built checkout of another commit; its bench line runs once with --dump-outputs next to ours, and mix.npy /
# t1_mix.npy of the two must be byte-equal.  Results go to $OUT_DIR/k1_latency_ab (default: build/, which git ignores).
set -u
REPS=${1:-3}
OTHER=${2:-}
OUT=${OUT_DIR:-build}/k1_latency_ab
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > "$OUT/card.txt"
ARGS="--gpus 1 --steps 200 --warmup 20 --no-cpu-baseline"
for r in $(seq 1 "$REPS"); do
    python bench.py $ARGS --dump-outputs "$OUT/dump_on_$r" > "$OUT/on_$r.json" 2> "$OUT/on_$r.err" || tail -3 "$OUT/on_$r.err"
    python bench.py $ARGS --dump-outputs "$OUT/dump_off_$r" --opt k1_prefetch=0 > "$OUT/off_$r.json" 2> "$OUT/off_$r.err" || tail -3 "$OUT/off_$r.err"
done
if [ -n "$OTHER" ]; then
    OUT_ABS=$(cd "$OUT" && pwd)
    (cd "$OTHER" && python bench.py $ARGS --dump-outputs "$OUT_ABS/dump_other") > "$OUT/other.json" 2> "$OUT/other.err" || tail -3 "$OUT/other.err"
fi
python - "$OUT" "$REPS" "$OTHER" <<'PY'
import json, statistics, sys
out, reps, other = sys.argv[1], int(sys.argv[2]), sys.argv[3]
print(open(f"{out}/card.txt").read().strip())
arms = {}
for arm in ("on", "off"):
    rows = [json.load(open(f"{out}/{arm}_{r}.json")) for r in range(1, reps + 1)]
    arms[arm] = rows
    for d in rows:
        oc = {k.split("_")[0]: round(c.get("ms_per_block", float("nan")), 4) for k, c in (d.get("other_configs") or {}).items()}
        print(arm, "value", round(d["value"]), "ms/step", round(d["ms_per_step"], 5), "K1", round(d["kernel_ms"]["K1_render"], 5),
              "K2", round(d["kernel_ms"]["K2_mix_reduce"], 5), "t1 ms/block", round(d["t1_million_voices"]["ms_per_block"], 4),
              "parity", d.get("parity_ok"), "worst", d.get("worst_err_over_tol"), "mix_worst", d.get("mix_worst_err_over_tol"),
              "bit_exact", d.get("bit_exact_rate"), "configs", oc)
med = {a: statistics.median(d["value"] for d in rows) for a, rows in arms.items()}
lo_on, hi_off = min(d["value"] for d in arms["on"]), max(d["value"] for d in arms["off"])
print(f"median value on {med['on']:.0f} off {med['off']:.0f}: {100 * (med['on'] / med['off'] - 1):+.1f} %, ranges overlap: {lo_on <= hi_off}")
dumps = [f"{out}/dump_{a}_{r}" for a in ("on", "off") for r in range(1, reps + 1)] + ([f"{out}/dump_other"] if other else [])
for f in ("mix.npy", "t1_mix.npy"):
    blobs = {d: open(f"{d}/{f}", "rb").read() for d in dumps}
    print(f, "byte-equal over", len(blobs), "runs:", len(set(blobs.values())) == 1)
PY
