# development: one ncu capture of the exec kernel on the real-text workload (source-level counters), written to $OUT
OUT=${OUT:-$(mktemp -d)}
mkdir -p "$OUT"
B="--workload realtext --steps 1 --warmup 1 --no-cpu --sustain 0 --no-compress"
python bench.py $B > /dev/null 2>&1 || exit 1
ncu --set full --clock-control none --import-source on -k regex:k_zexec2 -c 1 -o "$OUT/zexec2" -f python bench.py $B > "$OUT/ncu_exec.log" 2>&1
tail -3 "$OUT/ncu_exec.log"
echo "capture: $OUT/zexec2.ncu-rep"
