#!/bin/bash
# A/B of libbpltv builds on one GPU, in one job: the card's name and power limit, then `bench.py` alternating the
# builds REPS times (headline only, --no-extras), one full bench line per build with --dump-outputs (the outputs are
# compared byte for byte: strict arithmetic is bit-exact), and tools/time_pdps.py and
# tools/time_pdps_map.py per build and precision, twice, alternating.
#
#   tools/gpu_ab_bench.sh OUT_DIR LIB_A LIB_B [LIB_C ...]      (REPS=3 STEPS=5 WARMUP=3 TIME_ITERS=240 by default)
#
# A library is chosen with BPLTV_LIB, as tools/gpu_ab.sh does.  Results go to OUT_DIR/<lib name>_*.
set -u
out=$1; shift
mkdir -p "$out"
reps=${REPS:-3}; steps=${STEPS:-5}; warmup=${WARMUP:-3}; titers=${TIME_ITERS:-240}
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$out/gpu.csv"
for rep in $(seq 1 "$reps"); do
    for lib in "$@"; do
        n=$(basename "$lib" .so)
        BPLTV_LIB=$lib python bench.py --gpus 1 --steps "$steps" --warmup "$warmup" --no-extras 2>/dev/null | tail -1 > "$out/${n}_headline_$rep.json"
        python - "$out/${n}_headline_$rep.json" "$n" "$rep" <<'PY'
import json, sys
d = json.loads(open(sys.argv[1]).read())
print("%-16s rep %s  value %.2f  clocks %s" % (sys.argv[2], sys.argv[3], d["value"], json.dumps(d.get("clocks"))))
PY
    done
done
for lib in "$@"; do
    n=$(basename "$lib" .so)
    BPLTV_LIB=$lib python bench.py --gpus 1 --steps "$steps" --warmup "$warmup" --dump-outputs "$out/${n}_dump" 2>/dev/null | tail -1 > "$out/${n}_full.json"
    python - "$out/${n}_full.json" "$n" <<'PY'
import json, sys
d = json.loads(open(sys.argv[1]).read())
pick = lambda k: (d.get(k) or {}).get("value") if isinstance(d.get(k), dict) else d.get(k)  # noqa: E731
c5 = d.get("config5") or {}
print("%-16s full  value %.2f  other_arith %s  fp32 %s  e2e %s  config5.loss_only %s" %
      (sys.argv[2], d["value"], pick("per_gpu_value_other_arith"), pick("per_gpu_value_fp32"), pick("e2e"),
       json.dumps(c5.get("loss_only"))))
PY
done
first=$(basename "$1" .so)
for lib in "$@"; do
    n=$(basename "$lib" .so)
    for f in costgrad.npy u_sample.npy; do
        if cmp -s "$out/${first}_dump/$f" "$out/${n}_dump/$f"; then echo "$n $f identical to $first"; else echo "$n $f DIFFERS from $first"; fi
    done
done
for lib in "$@"; do rm -rf "$out/$(basename "$lib" .so)_dump"; done    # 128 MiB each; compared above
for rep in 1 2; do for lib in "$@"; do
    n=$(basename "$lib" .so)
    for prec in 64 32; do
        BPLTV_LIB=$lib BPLTV_PREC=$prec python tools/time_pdps.py "$titers" 2>&1 | sed "s/^/$n rep $rep /" | tee -a "$out/${n}_time_pdps.txt"
        BPLTV_LIB=$lib BPLTV_PREC=$prec python tools/time_pdps_map.py "$titers" 2>&1 | sed "s/^/$n rep $rep /" | tee -a "$out/${n}_time_pdps_map.txt"
    done
done; done
