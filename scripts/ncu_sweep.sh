#!/bin/bash
# ncu --set full of the collision kernels (after a clean run of the same command); reports and logs go to $OUT
OUT=${OUT:-$(mktemp -d)}
mkdir -p "$OUT"
CMD="python bench.py --steps 2 --warmup 3 --no-cpu --no-e2e --no-c1 --no-c5"
$CMD > "$OUT"/plain_sw.log 2>&1 || { tail -5 "$OUT"/plain_sw.log; exit 1; }
ncu --set full --clock-control none --import-source on -k regex:"pq_slow_kernel" -s 3 -c 1 -o "$OUT"/prof_sweep_edge -f $CMD > "$OUT"/ncu_sw1.log 2>&1
ncu --set full --clock-control none --import-source on -k regex:"dubins_check_kernel|dubins_size_kernel|dubins_emit_kernel|nearest_tpq" -s 9 -c 4 -o "$OUT"/prof_dubins -f $CMD > "$OUT"/ncu_sw2.log 2>&1
tail -2 "$OUT"/ncu_sw1.log "$OUT"/ncu_sw2.log | cut -c1-200
echo "reports in $OUT"
