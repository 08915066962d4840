# group resolves: the card, smoke, the new GPU tests, the group measurement, bench.py of the parent commit and this tree alternated, and
# the per-kernel SASS diff against the parent. parent_tree/: `git archive` of the parent commit, built with make (not part of the
# repository). Writes into $OUT.
set -x
export OUT=${OUT:-group_out}
mkdir -p $OUT
nvidia-smi -L
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -1
python scratch/sass_diff.py parent_tree/software-raytracer_b200/build software-raytracer_b200/build > $OUT/r8a_sass_diff.txt; tail -1 $OUT/r8a_sass_diff.txt
timeout 600 python -m pytest tests/test_gpu_group_resolve.py -q -rs 2>&1 | tail -15
timeout 300 python scratch/group_resolve_bench.py --out $OUT/r8a_group_resolve.json 2> $OUT/group_bench.err | cut -c1-600
tail -3 $OUT/group_bench.err
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
