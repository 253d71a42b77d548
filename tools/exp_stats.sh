cd /root/repo
timeout 300 python -m pytest tests/test_gpu_parity.py -q -x -k "rollout_matches_stepwise" 2>&1 | tail -2
for gw in 1 2; do for pat in 0 40; do echo "== gw=$gw patience=$pat"; RBG_GEN_WARPS=$gw RBG_GEN_PATIENCE=$pat python tools/persist_stats.py; done; done
