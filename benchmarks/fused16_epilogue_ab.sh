#!/bin/bash
# A/B of builds of the fp16 x 2 fused logistic gradient: c5 and c3 steps (20 timed steps each), the builds alternated
# three times.  Arguments: NAME=LIBRARY pairs, e.g.
#   bash benchmarks/fused16_epilogue_ab.sh parent=build/lib_parent/libb200hmc.so new=aehmc_b200/lib/libb200hmc.so
# Prints one line per run: headline value, gradient call inside the step, SM clock.  Each run's JSON line and stderr
# go to AB_OUT (default: a new temporary directory).
out=${AB_OUT:-$(mktemp -d)}
mkdir -p "$out"
echo "# runs in $out"
for rep in 1 2 3; do
  for wl in c5 c3; do
    for pair in "$@"; do
      name=${pair%%=*}; lib=${pair#*=}
      f=$out/${wl}_${name}_${rep}
      B2H_LIB=$lib python bench.py --workload $wl --no-ess --no-cpu --no-secondary > "$f.json" 2> "$f.err"
      python - "$f.json" "$wl" "$name" "$rep" <<'PY'
import json, sys
f, wl, name, rep = sys.argv[1:]
try:
    d = json.loads(open(f).read().strip().splitlines()[-1])
except Exception as e:
    print(wl, name, rep, "FAILED", e); sys.exit()
r = d["roofline"]
print(wl, name, rep, "value", round(d["value"]), "grad_ms", round(r["avg_launch_ms"], 4),
      "sm_mhz", d.get("clocks", {}).get("sm_mhz"), flush=True)
PY
    done
  done
done
