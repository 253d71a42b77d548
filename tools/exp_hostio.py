"""e2e step (rbg_connector_step_host_io) under different host thread counts (RBG_HOST_THREADS): one subprocess per setting."""
import os, subprocess, sys
root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
code = r'''
import ctypes as C, sys, time, numpy as np, torch
sys.path.insert(0, %r)
import routing_board_generation_b200 as rbg
L, lib = rbg._lib, rbg._lib.load()
G, N, B = 10, 5, 65536
keys = rbg.split(rbg.PRNGKey(0), B)
env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50))
st, _ = env.reset(keys)
pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
h = dict(obs=pin((B, N, G, G), torch.int32), mask=pin((B, N, 5), torch.uint8), sc=pin((B,), torch.int32), reward=pin((B, N), torch.float32), discount=pin((B, N), torch.float32),
         step_type=pin((B,), torch.int8), nc=pin((B,), torch.int32), rc=pin((B,), torch.float32), tpl=pin((B,), torch.int32))
act = pin((B, N), torch.int32); act.copy_(torch.randint(0, 5, (B, N), dtype=torch.int32))
a = st.agents
s = L.rbg_state(st.grid.data_ptr(), st.step_count.data_ptr(), a.id.data_ptr(), a.start.data_ptr(), a.target.data_ptr(), a.position.data_ptr(), st.key.data_ptr())
t = L.rbg_timestep(*(h[k].data_ptr() for k in ("obs", "mask", "sc", "reward", "discount", "step_type", "nc", "rc", "tpl")))
params = L.rbg_env_params(50, -0.03, 0.1, 0)
step = lambda: L.check(lib.rbg_connector_step_host_io(C.byref(s), act.data_ptr(), B, G, N, C.byref(params), C.byref(t), -1))
for _ in range(32): step()
best = 1e9
for rep in range(3):
    t0 = time.perf_counter()
    for _ in range(20): step()
    best = min(best, (time.perf_counter() - t0) / 20)
L.host_transfer_stats(reset=True)
for _ in range(10): step()
st_ = L.host_transfer_stats()
print("%%.3f ms/step  %%.1f M env-steps/s  threads %%d  d2h MB/step %%.1f" %% (best * 1e3, B / best / 1e6, st_[2], st_[1] / 10 / 1e6))
''' % root
settings = [{}, {"RBG_HOST_THREADS": "8"}, {"RBG_HOST_THREADS": "10"}, {"RBG_HOST_THREADS": "12"}, {"RBG_HOST_THREADS": "16"}]
if len(sys.argv) > 1:
    settings = [dict(kv.split("=") for kv in a.split(",") if kv) for a in sys.argv[1:]]
for env in settings:
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True, timeout=600)
    print(env, r.stdout.strip() or r.stderr[-600:], flush=True)
