#!/bin/bash
# A/B of two library builds on the flagship workload, alternated in one run so that both see the same card and neighbours:
#   base = fslr_b200/csrc/libfslr_b200_base.so (build the parent commit there: make -C <parent checkout>/fslr_b200/csrc, copy the .so)
#   new  = fslr_b200/csrc/libfslr_b200.so
# Every C4 run dumps its cluster / n_reads columns; all dumps must be identical.  Logs go to OUT_DIR (default: a new temporary
# directory), the summary to OUT_DIR/summary.txt.  Usage: tests/_ab_ingest.sh [rounds=3] [OUT_DIR]
set -u
ROUNDS=${1:-3}
OUT=${2:-$(mktemp -d)}
echo "logs: $OUT"
DUMPS=$(mktemp -d)
trap 'rm -rf "$DUMPS"' EXIT
mkdir -p $OUT
declare -A LIB=([base]=fslr_b200/csrc/libfslr_b200_base.so [new]=fslr_b200/csrc/libfslr_b200.so)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/gpu.txt
for i in $(seq 1 $ROUNDS); do
  for tag in base new; do
    FSLR_B200_LIB=${LIB[$tag]} timeout 600 python bench.py --config C4 --steps 20 --warmup 5 --no-cpu-baseline --no-python-reference \
      --dump-outputs $DUMPS/${tag}_$i > $OUT/c4_${tag}_$i.log 2>&1 || { echo "C4 $tag $i failed"; tail -20 $OUT/c4_${tag}_$i.log; }
  done
done
for tag in base new; do
  FSLR_B200_LIB=${LIB[$tag]} timeout 600 python bench.py --config C5 --steps 10 --warmup 3 --no-cpu-baseline --no-python-reference \
    > $OUT/c5_$tag.log 2>&1 || { echo "C5 $tag failed"; tail -20 $OUT/c5_$tag.log; }
done
python - "$OUT" "$DUMPS" "$ROUNDS" <<'EOF' | tee $OUT/summary.txt
import glob, json, os, statistics, sys
import numpy as np
out, dumps, rounds = sys.argv[1], sys.argv[2], int(sys.argv[3])
INGEST = ("keep_fillings", "data_order_mask", "query_rank_read_lists", "chrom_sort", "records_bands")
def load(path):
    return json.loads(open(path).read().strip().splitlines()[-1])
res = {}
for tag in ("base", "new"):
    runs = [load(os.path.join(out, "c4_%s_%d.log" % (tag, i))) for i in range(1, rounds + 1)]
    step = [r["ms_per_step"] for r in runs]
    ingest = [sum(r["stage_ms"][k] for k in INGEST) for r in runs]
    e2e = [r["e2e"]["ms_per_step"] for r in runs]
    res[tag] = dict(step=statistics.median(step), ingest=statistics.median(ingest), e2e=statistics.median(e2e),
                    launches=runs[0].get("gpu_launches"))
    print("C4 %-4s ms/step %s  ingest %s  e2e %s  launches %s" % (tag, [round(x, 3) for x in step], [round(x, 3) for x in ingest],
                                                                  [round(x, 2) for x in e2e], res[tag]["launches"]))
    print("   stages (median run):", {k: round(v, 3) for k, v in sorted(runs, key=lambda r: r["ms_per_step"])[rounds // 2]["stage_ms"].items()})
for tag in ("base", "new"):
    r = load(os.path.join(out, "c5_%s.log" % tag))
    print("C5 %-4s ms/step %.3f" % (tag, r["ms_per_step"]))
b, n = res["base"], res["new"]
print("C4 median: step %.3f -> %.3f (%.3f), ingest %.3f -> %.3f, e2e %.2f -> %.2f" % (b["step"], n["step"], n["step"] - b["step"],
                                                                                   b["ingest"], n["ingest"], b["e2e"], n["e2e"]))
ref = None
for d in sorted(glob.glob(os.path.join(dumps, "*"))):
    cols = {f: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}
    if ref is None:
        ref = cols
    assert cols.keys() == ref.keys() and all(np.array_equal(cols[f], ref[f]) for f in cols), "outputs differ: " + d
print("dumps identical:", len(glob.glob(os.path.join(dumps, "*"))), "runs,", sorted(ref))
EOF
