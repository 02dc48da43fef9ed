cd "$(dirname "$0")"
nvidia-smi --query-gpu=name,power.limit --format=csv
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
python -m pytest tests/test_respaced.py -m gpu -q -p no:cacheprovider 2>&1 | tail -4
