# pixel filter, final tree: the card, build, smoke, the new GPU tests, then the whole suite (GPU and CPU tests)
set -x
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -1
timeout 900 python -m pytest tests/test_gpu_pixel_filter.py -q -rs 2>&1 | tail -8
timeout 1800 python -m pytest tests -q -rs 2>&1 | tail -15
