# temporal resolve, final tree: build, smoke, the whole suite (the new GPU tests print their quality figures)
set -x
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -1
timeout 1500 python -m pytest tests -q -s 2>&1 | grep -E " dB|passed|failed|Error" | tail -12
