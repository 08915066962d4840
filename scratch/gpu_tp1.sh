# temporal resolve: smoke, the new GPU tests, the whole suite, the temporal measurement, bench.py of the parent commit and this tree
# alternated. parent_tree/: `git archive` of the parent commit, built with make (not part of the repository)
set -x
export OUT=${OUT:-temporal_out}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -1
timeout 900 python -m pytest tests/test_gpu_temporal.py -q -s -x 2>&1 | grep -E "dB|passed|failed|Error|assert" | tail -30
timeout 1500 python -m pytest tests -q 2>&1 | tail -4
timeout 900 python scratch/temporal_bench.py --out $OUT/r7a_temporal.json 2> $OUT/temporal_bench.err | cut -c1-300
for i in 1 2 3; do
  (cd parent_tree && python bench.py --gpus 1 --steps 5 --warmup 3 2>/dev/null | tail -1 > ../$OUT/bench_parent_$i.json)
  python bench.py --gpus 1 --steps 5 --warmup 3 2>/dev/null | tail -1 > $OUT/bench_new_$i.json
done
python - <<'PY'
import json, glob, os
for f in sorted(glob.glob(os.environ["OUT"] + "/bench_*.json")):
    d = json.loads(open(f).read())
    print(f, round(d["value"], 1), round(d["ms_per_step"], 3))
PY
