python -m pytest tests -q -m gpu -p no:cacheprovider 2>&1 | tail -6
python -m pytest tests/test_episodes.py -q -m gpu -p no:cacheprovider -k "big_shared or aggregator" 2>&1 | tail -3
echo "== smoke"; python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
echo "== bench"; python bench.py --gpus 1 --steps 500 --warmup 20 2>&1 | tail -1 | cut -c1-200
