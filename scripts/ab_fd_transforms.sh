#!/bin/bash
# Same-box A/B of two built trees of this project on one GPU: A = the parent commit, B = the change.
#   scripts/ab_fd_transforms.sh outputs A_DIR B_DIR OUT_DIR
#       bench.py --dump-outputs on both trees for c4 (the default command), c3, c4 at T = 131072 and c5 HALS at
#       T = 1048576; W.npy, H.npy and loss.npy must be byte-identical, and so must loss.final and
#       value_calibrated_loss.last_checked_prediction_rel_err of the two JSON lines (OUT_DIR/summary.txt)
#   scripts/ab_fd_transforms.sh time A_DIR B_DIR OUT_DIR [ROUNDS]
#       ROUNDS (default 5) alternations of `bench.py --steps 20 --warmup 3 --no-e2e --no-cpu` (ms_per_step,
#       value_direct_loss, value_calibrated_loss; the end-to-end and CPU figures are left out), then one CMF_TRACE=1 run
#       per tree (live per-launch times on stderr).  scripts/ab_fd_summary.py OUT_DIR prints medians and spreads.
set -u
MODE=$1; A=$(cd "$2" && pwd); B=$(cd "$3" && pwd); mkdir -p "$4"; OUT=$(cd "$4" && pwd); ROUNDS=${5:-5}
DUMP=$(mktemp -d); trap 'rm -rf "$DUMP"' EXIT     # the dumped arrays stay out of OUT_DIR
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.txt"

run() {   # tree tag args...
    local tree=$1 tag=$2; shift 2
    (cd "$tree" && timeout 1500 python bench.py "$@" > "$OUT/$tag.json" 2> "$OUT/$tag.err"); echo "$tag rc=$?"
}
if [ "$MODE" = time ]; then
    for r in $(seq 1 "$ROUNDS"); do
        run "$A" "time_A_$r" --steps 20 --warmup 3 --no-e2e --no-cpu
        run "$B" "time_B_$r" --steps 20 --warmup 3 --no-e2e --no-cpu
    done
    for side in A B; do
        tree=$A; [ $side = B ] && tree=$B
        (cd "$tree" && CMF_TRACE=1 timeout 1500 python bench.py --steps 20 --warmup 3 --no-e2e --no-cpu --no-calibrated \
            > "$OUT/trace_$side.json" 2> "$OUT/trace_$side.err"); echo "trace_$side rc=$?"
    done
    exit 0
fi
for side in A B; do
    tree=$A; [ $side = B ] && tree=$B
    run "$tree" "c4_$side" --dump-outputs "$DUMP/dump_c4_$side"
    run "$tree" "c3_$side" --config c3 --no-e2e --no-cpu --dump-outputs "$DUMP/dump_c3_$side"
    run "$tree" "c4T131072_$side" --T 131072 --no-e2e --no-cpu --dump-outputs "$DUMP/dump_c4T131072_$side"
    run "$tree" "c5hals_$side" --config c5 --alg hals --T 1048576 --no-e2e --no-cpu --dump-outputs "$DUMP/dump_c5hals_$side"
done
{
    for w in c4 c3 c4T131072 c5hals; do
        for f in W.npy H.npy loss.npy; do
            if cmp -s "$DUMP/dump_${w}_A/$f" "$DUMP/dump_${w}_B/$f"; then echo "same  $w $f"; else echo "DIFF  $w $f"; fi
        done
    done
    for pair in "c4_A c4_B" "c3_A c3_B" "c4T131072_A c4T131072_B" "c5hals_A c5hals_B"; do
        set -- $pair
        python - "$OUT/$1.json" "$OUT/$2.json" <<'EOF'
import json, sys
a, b = ([json.loads(l) for l in open(p) if l.startswith("{")][-1] for p in sys.argv[1:3])
for key in ("loss.final", "value_calibrated_loss.last_checked_prediction_rel_err"):
    va, vb = a, b
    for k in key.split("."):
        va = va.get(k) if isinstance(va, dict) else None
        vb = vb.get(k) if isinstance(vb, dict) else None
    print("same " if va == vb else "DIFF ", sys.argv[1].rsplit("/", 1)[-1], key, repr(va), repr(vb))
EOF
    done
} | tee "$OUT/summary.txt"
