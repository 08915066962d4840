# group resolves, final tree: the card, build, smoke, the whole suite (GPU and CPU tests)
set -x
nvidia-smi -L
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -1
timeout 1000 python -m pytest tests -q -rs 2>&1 | tail -20
