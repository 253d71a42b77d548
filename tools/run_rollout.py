"""Time the fused rollout (rbg_connector_rollout_random) in the stationary regime: per-kernel averages
from the library's own event pairs.  Used for A/B builds and ncu captures.

    [KIND=uniform|dataset] python tools/run_rollout.py [G N B T calls burnin_calls]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import routing_board_generation_b200 as rbg

a = [int(x) for x in sys.argv[1:]]
G, N, B, T, calls, burn = (a + [10, 5, 65536, 20, 25, 8][len(a):])[:6]
kind = os.environ.get('KIND')
if kind == 'dataset':  # rollout_warp_kernel: resets are picks from a stored board set
    gen = rbg.BoardDatasetGeneratorJAX(G, N, board_name="offline_parallel_rw", number_of_boards=int(os.environ.get('BOARDS', '4096')))
else:  # rollout_persist_kernel with its generator warps
    gen = (rbg.UniformRandomGenerator if kind == 'uniform' else rbg.ParallelRandomWalkGenerator)(grid_size=G, num_agents=N)
env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=gen, time_limit=int(os.environ.get('TL', '50'))))
keys = rbg.split(rbg.PRNGKey(0), B)
st, _ = env.reset(keys)
out = None
for _ in range(burn):
    st, out, _ = env.rollout_random(st, T, out=out)
torch.cuda.synchronize()
timing = not os.environ.get('NOTIMING')  # kernel timing serialises the slices (one kernel at a time)
rbg._lib.kernel_timing(timing)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(calls):
    st, out, _ = env.rollout_random(st, T, out=out)
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / calls
n_ro, ms_ro = rbg._lib.kernel_time("rollout")
n_pw, ms_pw = rbg._lib.kernel_time("prw")
n_env, ms_env = rbg._lib.kernel_time("env")
print(f"{G}x{G}/{N} B={B} T={T}: {ms:.4f} ms/call  {B * T / ms / 1e3:.1f} M env-steps/s | rollout kernel {ms_ro / max(n_ro, 1):.4f} ms x{n_ro}"
      f" | refill {ms_pw / max(n_pw, 1):.4f} ms x{n_pw} | env {ms_env / max(n_env, 1):.4f} ms x{n_env} | checksum {int(out.reward.sum() * 100)} {int(st.grid.sum())}")
