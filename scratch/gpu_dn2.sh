# denoised resolve, final defaults: smoke, GPU suite, denoise measurement, bench.py of the parent commit and this tree alternated
# parent_tree/: `git archive` of the parent commit, built with make (not part of the repository)
set -x
export OUT=${OUT:-denoise_out}
mkdir -p $OUT
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -1
timeout 900 python -m pytest tests -m gpu -q -s 2>&1 | grep -E "dB|passed|failed|Error" | tail -12
timeout 900 python scratch/denoise_bench.py --out $OUT/r6a_denoise.json 2> $OUT/denoise_bench.err | cut -c1-400
for i in 1 2 3; do
  (cd parent_tree && python bench.py --gpus 1 --steps 5 --warmup 3 2>/dev/null | tail -1 > ../$OUT/bench_parent_$i.json)
  python bench.py --gpus 1 --steps 5 --warmup 3 2>/dev/null | tail -1 > $OUT/bench_new_$i.json
done
python - <<'PY'
import json, glob, os
for f in sorted(glob.glob(os.environ["OUT"] + "/bench_*.json")):
    d = json.loads(open(f).read())
    print(f, round(d["value"], 1), round(d["ms_per_step"], 3), [(c.get("config"), c.get("ms_per_step") or c.get("p50_ms")) for c in d.get("configs", [])][:5])
PY
