#!/bin/bash
# Inflate A/B on one B200 (profiles/r06_inflate_ab.md): the card and its power limit, the inflate kernel alone over every variant in
# $V (two passes, the second in reverse order, each on an image of two rounds of its stream count), the role counters of the
# -DFASTF_TPS_PROF=1 builds (*_prof.so), then the headline job alternating between variants with its outputs compared.
# usage: gpu_r06_ab.sh "<variants for the headline A/B>" [rounds of the headline A/B] [final]
#   variants: libraries in $V (default fastf_b200/_build/variants, see build_variants.sh); "default" = the in-tree library
#   final: then `pytest -m gpu` and one full bench.py line of the in-tree library
# Logs go to $FASTF_AB_OUT (default: a new temporary directory, printed first).
OUT="${FASTF_AB_OUT:-$(mktemp -d)}"
mkdir -p "$OUT" && OUT=$(cd "$OUT" && pwd)
echo "logs in $OUT"
V="${FASTF_AB_VARIANTS:-fastf_b200/_build/variants}"
LOG=$OUT/r06_inflate_ab.log
BENCH_LIBS="$1"; ROUNDS="${2:-3}"; FINAL="$3"
DUMPS=$(mktemp -d)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $LOG
python scripts/inflate_ab.py --reps 1 > /dev/null 2> $OUT/ab_err.txt   # generates + caches the image
libs=$(ls $V/*.so | grep -v _prof)
for pass in 1 2; do
  for lib in $libs; do
    FASTF_GPU_LIB=$PWD/$lib timeout 200 python scripts/inflate_ab.py 2>> $OUT/ab_err.txt >> $LOG || echo "FAILED $lib" >> $LOG
  done
  libs=$(echo $libs | tr ' ' '\n' | tac)
done
for lib in $V/*_prof.so; do
  [ -e "$lib" ] || continue
  echo "== $(basename $lib)" >> $LOG
  FASTF_GPU_LIB=$PWD/$lib timeout 200 python scripts/inflate_ab.py --reps 2 2>> $OUT/ab_err.txt >> $LOG || echo "FAILED $lib" >> $LOG
done
BL=$OUT/r06_bench_ab.log
: > $BL
for r in $(seq $ROUNDS); do
  for v in $BENCH_LIBS; do
    lib=$PWD/$V/$v.so; [ "$v" = default ] && lib=$PWD/fastf_b200/_build/libfastf_gpu.so
    d=$DUMPS/${v}_$r
    FASTF_GPU_LIB=$lib python bench.py --steps 3 --warmup 3 --no-cpu-baseline --no-hw-extra --freq-reads 0 --dump-outputs $d > $OUT/bench_${v}_$r.json 2> $OUT/bench_${v}_$r.err
    echo "rc=$?" >> $OUT/bench_${v}_$r.err
    python -c "
import json, sys
d = json.loads(open('$OUT/bench_${v}_$r.json').read().strip().splitlines()[-1])
print('$v round $r', 'value %.1f M reads/s' % (d['value'] / 1e6), 'ms/step %.1f' % d['ms_per_step'], 'inflate %.1f ms' % d['stages']['inflate']['ms'],
      'parse %.1f ms' % d['stages']['parse']['ms'], 'crc %.1f ms' % d['stages']['crc']['ms'], 'roofline.achieved %.1f GB/s' % d['roofline']['achieved'])" >> $BL 2>&1
    tail -1 $OUT/bench_${v}_$r.err | sed "s/^/$v round $r /" >> $BL
    (cd $d && md5sum *.npy | sed "s/^/$v round $r /") >> $OUT/r06_dump_md5.txt
    rm -rf $d
  done
done
rm -rf $DUMPS
cat $LOG $BL $OUT/r06_dump_md5.txt
if [ -n "$FINAL" ]; then
  python -m pytest tests -m gpu -q -rs > $OUT/r06_pytest_gpu.log 2>&1
  tail -15 $OUT/r06_pytest_gpu.log
  python bench.py > $OUT/r06_bench.json 2> $OUT/r06_bench.err
  echo "bench rc=$?"; tail -c 1500 $OUT/r06_bench.json
fi
