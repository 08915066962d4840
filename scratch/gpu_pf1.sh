# pixel filter: the card, build, smoke, the new GPU tests, bench.py of the parent commit and this tree alternated, the filter
# measurement, then the whole suite. parent_tree/: `git archive` of the parent commit, built with make (not part of the repository).
set -x
export OUT=${OUT:-filter_out}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -1
timeout 900 python -m pytest tests/test_gpu_pixel_filter.py -q -x -rs 2>&1 | tail -25
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
timeout 600 python scratch/filter_bench.py --out $OUT/r9a_filter.json 2> $OUT/filter_bench.err | cut -c1-1500
tail -3 $OUT/filter_bench.err
timeout 1800 python -m pytest tests -q -m gpu -rs 2>&1 | tail -15
