#!/bin/bash
# Same-call A/B of the Double Sphere headline pass between a base revision and the working tree.  Boxes of the pool differ
# by up to 40 % on FP64-bound kernels, so only figures taken in one call on one card are compared.
#
#   scripts/ab_ds_headline.sh build <rev>   (needs git and nvcc, no GPU) exports <rev> with git archive into build/ab/base,
#                                            builds it there and copies its library to build/ab/libacm_base.so; then builds the tree
#   scripts/ab_ds_headline.sh run           (on the GPU) ROUNDS (default 4) rounds of base / tree alternated, each
#                                            100 M points x REPS (default 200) launches of acm_linearize_async with MODELS=5 (both residual
#                                            kinds: the algebraic one is the control), the SM clock sampled during every timed
#                                            loop; then bench.py --no-e2e --no-extras --no-lm-check once per build with
#                                            --dump-outputs, and the two sets of normal equations compared.
# Output goes to $OUT (default build/ab/out).
set -e
cd "$(dirname "$0")/.."
case "$1" in
build)
    rev=${2:?base revision}
    rm -rf build/ab/base && mkdir -p build/ab/base
    git archive "$rev" | tar -x -C build/ab/base
    python build/ab/base/__graft_entry__.py > build/ab/base.log 2>&1 || { cat build/ab/base.log; exit 1; }
    cp build/ab/base/apex_camera_models_b200/lib/libacm.so build/ab/libacm_base.so
    python __graft_entry__.py
    ;;
run)
    OUT=${OUT:-build/ab/out}; mkdir -p "$OUT"
    base=$PWD/build/ab/libacm_base.so; tree=$PWD/apex_camera_models_b200/lib/libacm.so
    [ -f "$base" ] && [ -f "$tree" ] || { echo "build both libraries first: $0 build <rev>"; exit 1; }
    nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/card.txt"
    for r in $(seq 1 "${ROUNDS:-4}"); do
        for b in base tree; do
            lib=$base; [ $b = tree ] && lib=$tree
            echo -n "round $r $b: " | tee -a "$OUT/ab.txt"
            ACM_LIB_PATH=$lib MODELS=5 REPS=${REPS:-200} CLOCKS=1 python scripts/lin_bench.py | tr "\n" "|" | tee -a "$OUT/ab.txt"
            echo | tee -a "$OUT/ab.txt"
        done
    done
    for b in base tree; do
        lib=$base; [ $b = tree ] && lib=$tree
        ACM_LIB_PATH=$lib python bench.py --gpus 1 --no-e2e --no-extras --no-lm-check --dump-outputs "$OUT/ne_$b" > "$OUT/bench_$b.json" 2> "$OUT/bench_$b.err" || true
        echo "bench $b: $(tail -1 "$OUT/bench_$b.json")"
    done
    python - "$OUT" <<'EOF'
import sys, numpy as np
o = sys.argv[1]
a = {k: np.load(f"{o}/ne_base/{k}.npy") for k in ("H", "g", "cost", "n_valid")}
b = {k: np.load(f"{o}/ne_tree/{k}.npy") for k in ("H", "g", "cost", "n_valid")}
s = np.sqrt(np.abs(np.diag(a["H"])))
dH = np.max(np.abs(b["H"] - a["H"]) / np.outer(s, s))
print(f"normal equations tree vs base: H {dH:.2e} (relative to the diagonal scale)  "
      f"g {np.max(np.abs(b['g'] - a['g']) / (s * np.sqrt(2 * a['cost'][0]))):.2e}  "
      f"cost {abs(b['cost'][0] - a['cost'][0]) / a['cost'][0]:.2e}  n_valid {a['n_valid'][0]:.0f} / {b['n_valid'][0]:.0f}")
EOF
    ;;
*)
    sed -n '2,14p' "$0"; exit 1 ;;
esac
