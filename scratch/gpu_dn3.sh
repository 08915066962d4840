# denoised resolve: the final tree's denoise tests, the whole GPU suite and smoke()
set -x
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -1
timeout 900 python -m pytest tests -m gpu -q 2>&1 | tail -3
