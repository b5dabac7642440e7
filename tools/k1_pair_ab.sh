#!/bin/bash
# A/B of the current tree against an exported one (tools/export_tree.sh <commit> <tag> -> _ab_<tag>/), on one GPU, in one run:
#   1. outputs: bench.py --dump-outputs of both trees with the same arguments, compared bit for bit (np.array_equal);
#   2. speed: bench.py --steps 200 of both trees ALTERNATELY (rounds of ref, new: RUNS for mppi_ode_1m, RUNS_OTHER for the workloads
#      that share its code), median and spread of each.
# The CPU-baseline sample of bench.py is cut to 1000 rollouts: it is host work and does not enter the GPU numbers.
#     bash tools/k1_pair_ab.sh OUT_DIR [_ab_parent]
set -u
cd "$(dirname "$0")/.."
OUT=$(realpath -m "${1:?output directory}"); REF=${2:-_ab_parent}; RUNS=${RUNS:-5}; RUNS_OTHER=${RUNS_OTHER:-3}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.txt"
tree() { [ "$1" = ref ] && echo "$REF" || echo .; }

# ---- 1. outputs ----
for w in "mppi_ode_1m" "mppi_ode_c1" "mppi_ode_1m --rollouts 300000" "mppi_ode_1m_log"; do
  tag=$(echo "$w" | tr ' ' '_' | tr -d '-')
  for t in ref new; do
    (cd "$(tree $t)" && python bench.py --workload $w --steps 5 --warmup 3 --cpu-sample 1000 --dump-outputs "$OUT/dump_${t}_$tag" \
       > "$OUT/dump_${t}_$tag.json" 2> "$OUT/dump_${t}_$tag.err") || echo "bench failed: $t $w"
  done
done
python - "$OUT" <<'EOF' | tee "$OUT/bits.txt"
import glob, os, sys
import numpy as np
out = sys.argv[1]
for ref in sorted(glob.glob(os.path.join(out, "dump_ref_*/"))):
    new = ref.replace("dump_ref_", "dump_new_")
    names = sorted(os.listdir(ref))
    res = {n: bool(os.path.exists(os.path.join(new, n)) and np.array_equal(np.load(os.path.join(ref, n)), np.load(os.path.join(new, n)))) for n in names}
    print(os.path.basename(ref.rstrip("/"))[9:], "IDENTICAL" if res and all(res.values()) else "DIFFERENT", res)
EOF

# ---- 2. speed ----
for w in mppi_ode_1m mppi_ode_1m_log mppi_ode_c1 cem_ode_c2; do
  n=$RUNS_OTHER; [ $w = mppi_ode_1m ] && n=$RUNS
  for i in $(seq "$n"); do
    for t in ref new; do
      (cd "$(tree $t)" && python bench.py --workload $w --steps 200 --cpu-sample 1000 > "$OUT/speed_${w}_${t}_$i.json" 2> "$OUT/speed_${w}_${t}_$i.err") \
        || echo "bench failed: $t $w $i"
    done
  done
done
python - "$OUT" <<'EOF' | tee "$OUT/speed.txt"
import glob, json, os, statistics, sys
out = sys.argv[1]
def med(xs):
    return statistics.median(xs) if xs else float("nan")
for w in ("mppi_ode_1m", "mppi_ode_1m_log", "mppi_ode_c1", "cem_ode_c2"):
    row = {}
    for t in ("ref", "new"):
        ds = []
        for f in sorted(glob.glob(os.path.join(out, f"speed_{w}_{t}_*.json"))):
            lines = open(f).read().strip().splitlines()
            if lines:
                ds.append(json.loads(lines[-1]))
        v = [d["value"] for d in ds]
        row[t] = {"runs": len(v), "value_median": med(v), "value_min": min(v, default=float("nan")), "value_max": max(v, default=float("nan")),
                  "ms_per_step": med([d["ms_per_step"] for d in ds]),
                  "pipelined_ms": med([d["pipelined"]["ms_per_step"] for d in ds if d.get("pipelined")]),
                  "roofline_frac": med([d["roofline"]["frac"] for d in ds if d.get("roofline") and d["roofline"].get("frac") is not None]),
                  "kernel_ms": med([d["roofline"]["kernel_ms"] for d in ds if d.get("roofline") and d["roofline"].get("kernel_ms") is not None])}
    r, n = row["ref"], row["new"]
    print(json.dumps({"workload": w, **row, "gain_value_median": n["value_median"] / r["value_median"] - 1.0,
                      "ref_spread": (r["value_max"] - r["value_min"]) / r["value_median"], "new_spread": (n["value_max"] - n["value_min"]) / n["value_median"]}))
EOF
