# A/B of the deflate kernel's two schedules on one GPU, in one call (variants from build/variants/,
# built by scripts/build_variants.py; "ser" is -DLZ_PIPELINE=0, "a<N>" the pipeline with N search warps,
# "<name>t" the same with -DLZ_TIMING).  Usage: [OUT=dir] bash scripts/gpu_pipeline_ab.sh ser a22 [a18 a20 ...]
# Logs, card info and the --dump-outputs files go to $OUT (default ab_out).
set -u
OUT=${OUT:-ab_out}
mkdir -p $OUT
OLD=$1; NEW=$2; shift 2
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv | tee $OUT/card.txt
run() {  # variant tag args...
  v=$1; tag=$2; shift 2
  echo "== $v $tag $*"
  timeout 600 python scripts/variant_roundtrip.py $v "$@" 2> $OUT/ab_${v}_${tag}.err | python scripts/print_bench_line.py
}
# output identity: bench --dump-outputs of both builds at the timed size
run $OLD dump --dump-outputs $OUT/dump_$OLD
run $NEW dump --dump-outputs $OUT/dump_$NEW
python - "$OUT" "$OLD" "$NEW" <<'PY'
import sys, os, numpy as np
a, b = (os.path.join(sys.argv[1], "dump_" + x) for x in sys.argv[2:4])
for f in sorted(os.listdir(a)):
    same = np.array_equal(np.load(os.path.join(a, f)), np.load(os.path.join(b, f)))
    print("dump", f, "identical" if same else "DIFFERENT")
PY
# level 6, alternating, three runs each
for r in 1 2 3; do
  run $OLD l6r$r
  run $NEW l6r$r
done
for v in "$@"; do run $v l6; done
# other levels and every data class, old then new
for L in 1 9; do run $OLD l$L --level $L; run $NEW l$L --level $L; done
for C in 1 2 3 4 5; do run $OLD c$C --data-class $C --chunks 16384; run $NEW c$C --data-class $C --chunks 16384; done
run $OLD l12 --level 12 --chunks 4096 --chunk-size 1048576 --steps 1
run $NEW l12 --level 12 --chunks 4096 --chunk-size 1048576 --steps 1
# phase clocks (-DLZ_TIMING builds named <variant>t)
run ${OLD}t timing --chunks 16384
run ${NEW}t timing --chunks 16384
