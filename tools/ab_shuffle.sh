#!/bin/bash
# A/B of the shuffle workload between two builds of the library, alternating in one session so that both see the same
# card, clocks and neighbours.
#   tools/ab_shuffle.sh --build REF OUT.so          build git revision REF's library into OUT.so (needs a git checkout)
#   tools/ab_shuffle.sh OUT_DIR A.so B.so [ROUNDS]  ROUNDS (default 4) alternating runs of each build of
#       bench.py --workload shuffle --no-cpu --no-extra --steps 20 --warmup 5, then one run per build with
#       BPP_ACP_TRACE=1 (the prove / verify stage timelines, on stderr).  Writes OUT_DIR/gpu.csv (card, power limit,
#       max SM clock), OUT_DIR/{a,b}_<round>.json, OUT_DIR/{a,b}_trace.err and OUT_DIR/summary.json (median and spread
#       of the headline value, single_stream, e2e and the `fixed` leg per build).
set -e
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
if [ "$1" = "--build" ]; then
  ref=$2; out=$(realpath -m "$3"); tmp=$(mktemp -d)
  git -C "$ROOT" archive "$ref" bulletproof-perm_b200/csrc include | tar -x -C "$tmp"
  make -C "$tmp/bulletproof-perm_b200/csrc" -j8 OUT="$out" OBJDIR="$tmp/obj" > /dev/null
  rm -rf "$tmp"
  echo "built $out from $ref"
  exit 0
fi
out=$(realpath -m "$1"); libs=("$(realpath "$2")" "$(realpath "$3")"); rounds=${4:-4}
mkdir -p "$out"
cd "$ROOT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$out/gpu.csv"
args=(--workload shuffle --no-cpu --no-extra --steps 20 --warmup 5)
for r in $(seq 1 "$rounds"); do
  for i in 0 1; do
    tag=$([ $i = 0 ] && echo a || echo b)
    BPPERM_LIB=${libs[$i]} python bench.py "${args[@]}" | tail -1 > "$out/${tag}_$r.json"
  done
done
for i in 0 1; do
  tag=$([ $i = 0 ] && echo a || echo b)
  BPP_ACP_TRACE=1 BPPERM_LIB=${libs[$i]} python bench.py --workload shuffle --no-cpu --no-extra --no-fixed --steps 3 \
    --warmup 2 > /dev/null 2> "$out/${tag}_trace.err"
done
python - "$out" "$rounds" "${libs[@]}" <<'EOF'
import json, statistics, sys
out, rounds, libs = sys.argv[1], int(sys.argv[2]), sys.argv[3:]
keys = {"value": ("value",), "single_stream": ("single_stream", "value"), "e2e": ("e2e", "value"),
        "fixed": ("fixed", "value"), "fixed_e2e": ("fixed", "e2e", "value")}
summary = {"gpu": open(f"{out}/gpu.csv").read().strip().splitlines()[-1], "libs": libs, "rounds": rounds}
for tag in "ab":
    runs = [json.loads(open(f"{out}/{tag}_{r}.json").read()) for r in range(1, rounds + 1)]
    s = {}
    for name, path in keys.items():
        vals = []
        for run in runs:
            v = run
            for p in path:
                v = v.get(p) if isinstance(v, dict) else None
            if v is not None:
                vals.append(v)
        if vals:
            s[name] = {"median": statistics.median(vals), "min": min(vals), "max": max(vals), "runs": vals}
    summary[tag] = s
for name in summary["a"]:
    if name in summary["b"]:
        summary.setdefault("b_over_a", {})[name] = summary["b"][name]["median"] / summary["a"][name]["median"]
json.dump(summary, open(f"{out}/summary.json", "w"), indent=1)
print(json.dumps({k: summary[k] for k in ("gpu", "b_over_a")}, indent=1))
EOF
