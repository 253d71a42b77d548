"""Parity of the CUDA path (through the C-ABI, librbg_b200.so) with the CPU oracle.

Bit-exact everywhere: boards, coordinates, keys, masks, step types and extras are
integers; rewards / discounts / ratio_connections are float32 values produced by
the same two IEEE operations in both implementations (tolerance 0, compared by
bits).  Runs only on a CUDA device (`-m gpu`).
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PRW_CONFIGS = [(2, 1), (3, 2), (5, 3), (7, 8), (9, 9), (10, 5), (14, 7), (16, 16), (17, 17), (20, 10), (32, 16), (40, 32)]


def _np(t):
    import torch

    if t.dtype == torch.uint32:
        return t.view(torch.int32).cpu().numpy().view(np.uint32)
    if t.dtype == torch.bool:
        return t.cpu().numpy().astype(np.uint8)
    return t.cpu().numpy()


def _keys(rbg, orc, seed, B):
    """split(PRNGKey(seed), B) on the device (checked against the oracle)."""
    k = rbg.split(rbg.PRNGKey(seed), B)
    ref = orc.split(orc.PRNGKey(seed), B)
    assert np.array_equal(_np(k), ref)
    return k, ref


def _state_np(st):
    a = st.agents
    return dict(grid=_np(st.grid), step_count=_np(st.step_count), agent_id=_np(a.id), start=_np(a.start), target=_np(a.target), position=_np(a.position), key=_np(st.key))


def _assert_state(st, ref, where=""):
    got = _state_np(st)
    for k in ("grid", "step_count", "agent_id", "start", "target", "position", "key"):
        assert np.array_equal(got[k], ref[k]), f"state.{k} differs {where}"


def _assert_timestep(ts, ref, where=""):
    o = ts.observation
    assert np.array_equal(_np(o.grid), ref["obs"]), f"observation.grid differs {where}"
    assert np.array_equal(_np(o.action_mask), ref["action_mask"]), f"action_mask differs {where}"
    assert np.array_equal(_np(o.step_count), ref["obs_step_count"]), f"observation.step_count differs {where}"
    assert np.array_equal(_np(ts.step_type), ref["step_type"]), f"step_type differs {where}"
    # float32, tolerance 0: same bits
    assert np.array_equal(_np(ts.reward).view(np.uint32), ref["reward"].view(np.uint32)), f"reward differs {where}"
    assert np.array_equal(_np(ts.discount).view(np.uint32), ref["discount"].view(np.uint32)), f"discount differs {where}"
    assert np.array_equal(_np(ts.extras["num_connections"]), ref["num_connections"]), where
    assert np.array_equal(_np(ts.extras["ratio_connections"]).view(np.uint32), ref["ratio_connections"].view(np.uint32)), where
    assert np.array_equal(_np(ts.extras["total_path_length"]), ref["total_path_length"]), where


# ------------------------------------------------------------------- library
def test_library_is_the_cuda_one(rbg):
    lib = rbg._lib.load()
    arch, sms = C.c_int(), C.c_int()
    assert lib.rbg_device_info(C.byref(arch), C.byref(sms)) == 0
    assert arch.value >= 100 and sms.value > 0
    assert lib.rbg_version() == 200


def test_split_keys(rbg, orc):
    for seed, B in ((0, 1), (0, 2), (0, 5), (7, 1024), (3, 4097)):
        _keys(rbg, orc, seed, B)
    k = rbg.split(rbg.PRNGKey(5), 1000, offset=333, count=100)
    assert np.array_equal(_np(k), orc.split(orc.PRNGKey(5), 1000)[333:433])


# -------------------------------------------------------- ParallelRandomWalk
def test_reference_goldens_on_gpu(rbg, goldens):
    """test_parallel_random_walk_board.py:161-186 and notebook cells 4/13, on the CUDA path."""
    g = goldens["prw_5x5_3"]
    heads, targets, solved = rbg.ParallelRandomWalkBoard(5, 5, 3).generate_board(rbg.PRNGKey(0))
    assert _np(heads).tolist() == g["heads"]
    assert _np(targets).tolist() == g["targets"]
    assert _np(solved).tolist() == g["valid_end_grid2"]
    g = goldens["prw_generator_10x10_5_key0"]
    st = rbg.ParallelRandomWalkGenerator(10, 5)(rbg.PRNGKey(0))
    assert _np(st.agents.start).tolist() == g["start"]
    assert _np(st.agents.target).tolist() == g["target"]
    assert _np(st.agents.position).tolist() == g["start"]
    assert _np(st.key).tolist() == g["key"]
    assert int(st.step_count) == 0
    g = goldens["uniform_generator_10x10_5_key0"]
    st = rbg.UniformRandomGenerator(10, 5)(rbg.PRNGKey(0))
    assert _np(st.agents.start).tolist() == g["start"]
    assert _np(st.agents.target).tolist() == g["target"]
    assert _np(st.key).tolist() == g["key"]


def test_reference_runs_on_gpu(rbg):
    """The CUDA path against outputs of the reference's own Python source (tests/golden/reference_runs.json,
    made by tests/tools/make_reference_fixtures.py): collisions, SeedExtension options, generator States."""
    import json
    import os

    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_runs.json")) as f:
        runs = json.load(f)
    for cfg in runs["prw_generate_board"]:
        keys = rbg.split(rbg.PRNGKey(cfg["seed"]), cfg["n"])
        heads, targets, solved = rbg.ParallelRandomWalkBoard(cfg["G"], cfg["G"], cfg["N"]).generate_board(keys)
        assert _np(solved).tolist() == [r["solved"] for r in cfg["boards"]]
        assert _np(heads).tolist() == [r["heads"] for r in cfg["boards"]]
        assert _np(targets).tolist() == [r["targets"] for r in cfg["boards"]]
    gens = {"parallel_random_walk": rbg.ParallelRandomWalkGenerator, "uniform": rbg.UniformRandomGenerator, "seed_extension": rbg.SeedExtensionGenerator}
    for cfg in runs["generator_states"]:
        keys = rbg.split(rbg.PRNGKey(cfg["seed"]), cfg["n"])
        st = gens[cfg["kind"]](cfg["G"], cfg["N"])(keys)
        assert _np(st.grid).tolist() == [r["grid"] for r in cfg["states"]], cfg["kind"]
        assert _np(st.key).tolist() == [r["key"] for r in cfg["states"]]
        assert _np(st.agents.start).tolist() == [r["start"] for r in cfg["states"]]
        assert _np(st.agents.target).tolist() == [r["target"] for r in cfg["states"]]
    for cfg in runs["seedext_solved"]:
        keys = rbg.split(rbg.PRNGKey(cfg["seed"]), cfg["n"])
        board = rbg.SeedExtensionBoard(cfg["G"], cfg["G"], cfg["N"])
        solved = board.return_solved_board(keys, **cfg["options"])
        assert _np(solved).tolist() == [r["solved"] for r in cfg["boards"]], cfg["options"]
        (sr, sc), (er, ec) = board.generate_starts_ends(keys, **cfg["options"])
        assert _np(sr).tolist() == [r["starts"][0] for r in cfg["boards"]] and _np(sc).tolist() == [r["starts"][1] for r in cfg["boards"]]
        assert _np(er).tolist() == [r["ends"][0] for r in cfg["boards"]] and _np(ec).tolist() == [r["ends"][1] for r in cfg["boards"]]


@pytest.mark.parametrize("G,N", PRW_CONFIGS)
def test_prw_generate_matches_oracle(rbg, orc, G, N):
    B = 2048 if G <= 20 else 512
    keys, kref = _keys(rbg, orc, 11 + G, B)
    heads, targets, solved, stats = rbg.ParallelRandomWalkBoard(G, G, N).generate_board_with_stats(keys)
    rh, rt, rs, rstats = orc.prw_generate_batch(kref, G, N)
    assert np.array_equal(_np(solved), rs)
    assert np.array_equal(_np(heads), rh)
    assert np.array_equal(_np(targets), rt)
    assert np.array_equal(_np(stats), rstats)  # while-loop trips and collided moves too
    if G >= 10:
        assert rstats[:, 1].sum() > 0  # the collision branch is exercised


@pytest.mark.parametrize("B", [1, 2, 3, 31, 33, 63, 65, 257])
def test_prw_ragged_batches(rbg, orc, B):
    keys, kref = _keys(rbg, orc, 99, B)
    _, _, solved = rbg.ParallelRandomWalkBoard(10, 10, 5).generate_board(keys)
    assert np.array_equal(_np(solved), orc.prw_generate_batch(kref, 10, 5)[2])


def test_prw_large_batch_10x10(rbg, orc):
    """BASELINE config 1/2 size class: 65 536 boards at 10x10/5 vs the oracle."""
    B = 65536
    keys, kref = _keys(rbg, orc, 0, B)
    heads, targets, solved = rbg.ParallelRandomWalkBoard(10, 10, 5).generate_board(keys)
    rh, rt, rs, _ = orc.prw_generate_batch(kref, 10, 5)
    assert np.array_equal(_np(solved), rs) and np.array_equal(_np(heads), rh) and np.array_equal(_np(targets), rt)


def test_prw_exact_selection_fallback(rbg):
    """The start-cell selection normally filters sort keys by a threshold and ranks the survivors; when
    the filter keeps too few / too many it falls back to an exact N-round selection.  RBG_DEBUG_FLAGS=1
    forces that path (read once per process, hence the subprocess)."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import sys, numpy as np; sys.path.insert(0, %r)\n"
        "import routing_board_generation_b200 as rbg\n"
        "from oracle import oracle as orc\n"
        "for (G, N, B) in ((10, 5, 777), (5, 3, 300), (20, 10, 200)):\n"
        "    k = rbg.split(rbg.PRNGKey(3), B); kr = orc.split(orc.PRNGKey(3), B)\n"
        "    s = rbg.ParallelRandomWalkBoard(G, G, N).generate_board(k)[2].cpu().numpy()\n"
        "    assert np.array_equal(s, orc.prw_generate_batch(kr, G, N)[2]), (G, N)\n"
        "    st = rbg.UniformRandomGenerator(G, N)(k)\n"
        "    assert np.array_equal(st.grid.cpu().numpy(), orc.state_batch('uniform', kr, G, N)['grid'])\n"
        "print('exact ok')\n"
    ) % root
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, RBG_DEBUG_FLAGS="1"), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "exact ok" in r.stdout, r.stderr[-2000:]


def test_prw_empty_batch(rbg):
    import torch

    keys = torch.empty((0, 2), dtype=torch.uint32, device="cuda")
    h, t, s = rbg.ParallelRandomWalkBoard(10, 10, 5).generate_board(keys)
    assert h.shape == (0, 2, 5) and s.shape == (0, 10, 10)


def test_empty_batches_everywhere(rbg):
    """B = 0 through every batched entry point of the mirror: an empty batch has no buffers (torch gives NULL data pointers)."""
    import torch

    keys = torch.empty((0, 2), dtype=torch.uint32, device="cuda")
    for gen in (rbg.ParallelRandomWalkGenerator(10, 5), rbg.UniformRandomGenerator(10, 5), rbg.SeedExtensionGenerator(10, 5), rbg.SequentialRandomWalkGenerator(10, 5)):
        assert gen(keys).grid.shape == (0, 10, 10)
        env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=gen, time_limit=5))
        st, ts = env.reset(keys)
        assert ts.observation.grid.shape == (0, 5, 10, 10)
        st, ts = env.step(st, torch.empty((0, 5), dtype=torch.int32, device="cuda"))
        assert ts.reward.shape == (0, 5)
        st, ts, act = env.rollout_random(st, 3)
        assert ts.observation.grid.shape == (3, 0, 5, 10, 10) and act.shape == (3, 0, 5)
    assert rbg.SeedExtensionBoard(10, 10, 5).return_solved_board(keys).shape == (0, 10, 10)
    assert rbg.engine.validate(torch.empty((0, 10, 10), dtype=torch.int32, device="cuda"), 5).shape == (0,)


@pytest.mark.parametrize("G,N,B", [(20, 10, 131072), (32, 16, 16384)])
def test_prw_full_size_invariants(rbg, G, N, B):
    """BASELINE config 3 per-GPU slice (131 072 boards 20x20/10): every board passes the validity
    rules on the device (wires connect their own start and target, no crossings, solvable)."""
    keys = rbg.split(rbg.PRNGKey(0), 1048576 if G == 20 else B, 0, B)
    heads, targets, solved = rbg.ParallelRandomWalkBoard(G, G, N).generate_board(keys)
    flags = rbg.engine.validate(solved, N)
    # sound: own-cell connectivity, no duplicates, nothing but zero-length wires (lone TARGETs) breaks rules 2 / 4
    assert int((flags & (1 | 8 | 32 | 64 | 128)).abs().max()) == 0
    # heads / targets agree with the codes on the board
    import torch

    b = torch.arange(B, device="cuda")[:, None]
    i = torch.arange(N, device="cuda")[None, :]
    tcode = solved[b, targets[:, 0].long(), targets[:, 1].long()]
    assert bool((tcode == 3 * i + 3).all())
    hcode = solved[b, heads[:, 0].long(), heads[:, 1].long()]
    zero_len = (heads == targets).all(dim=1)
    assert bool(((hcode == 3 * i + 2) | zero_len).all())


# ------------------------------------------------------------- SeedExtension
SE_CONFIGS = [(2, 1), (4, 3), (5, 4), (6, 3), (9, 5), (10, 5), (14, 7), (20, 10), (32, 16), (40, 32)]


@pytest.mark.parametrize("G,N", SE_CONFIGS)
def test_seedext_solved_matches_oracle(rbg, orc, G, N):
    B = 1024 if G <= 20 else 128
    keys, kref = _keys(rbg, orc, 31 + G, B)
    board = rbg.SeedExtensionBoard(G, G, N)
    solved = board.return_solved_board(keys)
    ref, stats = orc.seedext_solved_batch(kref, G, N)
    assert np.array_equal(_np(solved), ref)
    assert (stats[:, 2] == 0).all()  # the BFS never ran dry in the oracle either
    (sr, sc), (er, ec) = board.generate_starts_ends(keys)
    for b in range(0, B, max(1, B // 16)):
        rs, re_ = orc.seedext_starts_ends(kref[b], G, N)
        assert np.array_equal(_np(sr[b]), rs[0]) and np.array_equal(_np(sc[b]), rs[1])
        assert np.array_equal(_np(er[b]), re_[0]) and np.array_equal(_np(ec[b]), re_[1])
    training = board.return_training_board(keys)
    assert np.array_equal(_np(training), ref * ((ref % 3) != 1))
    if G >= 4:
        assert int(rbg.engine.validate(solved, N).abs().max()) == 0


@pytest.mark.parametrize("kw", [dict(randomness=0.5), dict(randomness=1.0), dict(two_sided=False), dict(extension_iterations=2),
                                dict(extension_iterations=0), dict(extension_steps=3), dict(randomness=0.3, two_sided=False, extension_iterations=3, extension_steps=5)])
def test_seedext_options_match_oracle(rbg, orc, kw):
    G, N, B = 10, 5, 512
    keys, kref = _keys(rbg, orc, 77, B)
    solved = rbg.SeedExtensionBoard(G, G, N).return_solved_board(keys, **kw)
    okw = dict(randomness=kw.get("randomness", 0.0), two_sided=kw.get("two_sided", True), iterations=kw.get("extension_iterations", 1), ext_steps=int(kw.get("extension_steps", -1)))
    ref, _ = orc.seedext_solved_batch(kref, G, N, **okw)
    assert np.array_equal(_np(solved), ref)


_SE_SWITCH_CODE = """
import sys, numpy as np
sys.path.insert(0, {root!r})
import routing_board_generation_b200 as rbg
from oracle import oracle as orc
for (G, N, B, kw) in {cases!r}:
    kref = orc.split(orc.PRNGKey(5), B)
    keys = rbg.engine.as_tensor(kref)
    okw = dict(randomness=kw.get("randomness", 0.0), two_sided=kw.get("two_sided", True), iterations=kw.get("extension_iterations", 1), ext_steps=int(kw.get("extension_steps", -1)))
    ref, _ = orc.seedext_solved_batch(kref, G, N, **okw)
    for rep in range(2):  # the second call reuses the cached scratch pool and the second stream
        got = rbg.SeedExtensionBoard(G, G, N).return_solved_board(keys, **kw).cpu().numpy()
        assert np.array_equal(got, ref), (G, N, B, kw, rep, int((got != ref).any(axis=(1, 2)).sum()))
print("ok")
"""


@pytest.mark.parametrize("env_vars", [{"RBG_SE_CTAS_PER_SM": "1"}, {"RBG_SE_OVERLAP": "0"}, {"RBG_SE_CTAS_PER_SM": "1", "RBG_SE_EXT_WARPS": "8", "RBG_SE_REFILL_MIN": "16"},
                                      {"RBG_SE_EXT_WARPS": "1", "RBG_SE_CTAS_PER_SM": "2"}])
def test_seedext_queue_and_overlap_switches(env_vars):
    """The extend kernel is persistent (lanes take boards from a queue: RBG_SE_CTAS_PER_SM=1 makes a 40 000-board batch
    several times what is resident, so every lane is refilled), its chain phase is shared by the CTA (1, 3, 4, 8 warps
    per CTA), and the optimise kernel runs beside it on the list of finished boards (RBG_SE_OVERLAP=0: behind it).  All
    of it must leave the boards bit-identical to the oracle's, with the options that change the sweep loop as well."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cases = [(10, 5, 40000, {}), (14, 7, 9000, {}), (10, 5, 3000, dict(randomness=0.4, extension_iterations=2)), (9, 4, 2500, dict(two_sided=False, extension_steps=4)), (34, 12, 200, {})]
    code = _SE_SWITCH_CODE.format(root=root, cases=cases)
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env_vars), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and r.stdout.strip().startswith("ok"), (r.stdout[-800:], r.stderr[-2000:])


def test_seedext_single_key_and_ragged(rbg, orc):
    k = rbg.PRNGKey(0)
    solved = rbg.SeedExtensionBoard(10, 10, 5).return_solved_board(k)
    assert solved.shape == (10, 10)
    assert np.array_equal(_np(solved), orc.seedext_solved(orc.PRNGKey(0), 10, 5))
    for B in (1, 31, 33, 129):
        keys, kref = _keys(rbg, orc, 13, B)
        assert np.array_equal(_np(rbg.SeedExtensionBoard(10, 10, 5).return_solved_board(keys)), orc.seedext_solved_batch(kref, 10, 5)[0])


def test_seedext_full_size_invariants(rbg):
    """BASELINE config 4: SeedExtension 14x14 / 7 agents, 65 536 boards, all valid on the device."""
    keys = rbg.split(rbg.PRNGKey(0), 65536)
    solved = rbg.SeedExtensionBoard(14, 14, 7).return_solved_board(keys)
    assert int(rbg.engine.validate(solved, 7).abs().max()) == 0
    assert int((solved > 0).sum(dim=(1, 2)).min()) >= 14  # every wire has at least its two pins


def test_seedext_too_many_agents_is_an_error(rbg):
    with pytest.raises(rbg.RbgError):
        rbg.SeedExtensionBoard(6, 6, 10).return_solved_board(rbg.split(rbg.PRNGKey(0), 4))  # lattice has 9 seed cells


# ----------------------------------------------------------- generator State
@pytest.mark.parametrize("kind", ["parallel_random_walk", "uniform"])
@pytest.mark.parametrize("G,N", [(5, 3), (10, 5), (14, 7), (20, 10), (32, 16)])
def test_generator_state_matches_oracle(rbg, orc, kind, G, N):
    B = 1024
    keys, kref = _keys(rbg, orc, 5, B)
    gen = {"parallel_random_walk": rbg.ParallelRandomWalkGenerator, "uniform": rbg.UniformRandomGenerator}[kind](G, N)
    st = gen(keys)
    _assert_state(st, orc.state_batch(kind, kref, G, N))


@pytest.mark.parametrize("G,N", [(6, 3), (10, 5), (14, 7)])
def test_seedext_generator_state_matches_oracle(rbg, orc, G, N):
    keys, kref = _keys(rbg, orc, 5, 512)
    _assert_state(rbg.SeedExtensionGenerator(G, N)(keys), orc.state_batch("seed_extension", kref, G, N))


def test_seedext_connector_autoreset_matches_oracle(rbg, orc):
    n_last = _rollout(rbg, orc, "seed_extension", 10, 5, B=512, steps=40, autoreset=True, time_limit=15)
    assert n_last > 512


@pytest.mark.parametrize("board_name,G,N,K", [("offline_parallel_rw", 10, 5, 1000), ("offline_parallel_rw", 6, 4, 7), ("offline_seed_extension", 8, 4, 37)])
def test_dataset_generator_matches_oracle(rbg, orc, board_name, G, N, K):
    """BoardDatasetGeneratorJAX: K boards from split(PRNGKey(0), K), __call__ picks one with jax's randint."""
    gen = rbg.BoardDatasetGeneratorJAX(G, N, board_name=board_name, number_of_boards=K)
    kref = orc.split(orc.PRNGKey(0), K)
    if board_name == "offline_seed_extension":
        ref = [orc.seedext_starts_ends(kref[b], G, N, randomness=1.0, two_sided=False) for b in range(K)]
        rh = np.stack([r[0] for r in ref])
        rt = np.stack([r[1] for r in ref])
    else:
        rh, rt, _, _ = orc.prw_generate_batch(kref, G, N)
    assert np.array_equal(_np(gen.heads), rh) and np.array_equal(_np(gen.targets), rt)
    keys, k2 = _keys(rbg, orc, 3, 2048)
    _assert_state(gen(keys), orc.dataset_state_batch(k2, G, N, rh, rt))
    picked = {tuple(map(tuple, s)) for s in _np(gen(keys).agents.start)}
    assert len(picked) > min(K, 2048) // 3  # the draw spreads over the stored boards
    one = gen(rbg.PRNGKey(5))
    assert one.grid.shape == (G, G)
    assert np.array_equal(_np(gen.print_board(3)) > 0, _np(gen.print_board(3)) > 0)


def test_dataset_generator_reference_run(rbg):
    """Against the reference's own BoardDatasetGeneratorJAX run on the jax shim (tests/golden/reference_runs.json)."""
    import json
    import os

    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_runs.json")) as f:
        runs = json.load(f)
    for cfg in runs.get("dataset_generator", []):
        gen = rbg.BoardDatasetGeneratorJAX(cfg["G"], cfg["N"], board_name=cfg["board_name"], number_of_boards=cfg["K"])
        assert _np(gen.heads).tolist() == cfg["heads"] and _np(gen.targets).tolist() == cfg["targets"]
        keys = rbg.split(rbg.PRNGKey(cfg["seed"]), cfg["n"])
        st = gen(keys)
        assert _np(st.grid).tolist() == [r["grid"] for r in cfg["states"]]
        assert _np(st.key).tolist() == [r["key"] for r in cfg["states"]]
        assert _np(st.agents.start).tolist() == [r["start"] for r in cfg["states"]]


# ------------------------------------------------------------------ Connector
@pytest.mark.parametrize("kind", ["parallel_random_walk", "uniform"])
@pytest.mark.parametrize("G,N", [(5, 3), (10, 5), (9, 4), (32, 16)])
def test_connector_reset_matches_oracle(rbg, orc, kind, G, N):
    B = 512
    keys, kref = _keys(rbg, orc, 21, B)
    gen = {"parallel_random_walk": rbg.ParallelRandomWalkGenerator, "uniform": rbg.UniformRandomGenerator}[kind](G, N)
    st, ts = rbg.Connector(generator=gen).reset(keys)
    rst, rts = orc.connector_reset_batch(kind, kref, G, N)
    _assert_state(st, rst)
    _assert_timestep(ts, rts)


def _rollout(rbg, orc, kind, G, N, B, steps, autoreset, time_limit=50, seed=3):
    import torch

    keys, kref = _keys(rbg, orc, seed, B)
    gen = {"parallel_random_walk": rbg.ParallelRandomWalkGenerator, "uniform": rbg.UniformRandomGenerator, "seed_extension": rbg.SeedExtensionGenerator,
           "sequential_random_walk": rbg.SequentialRandomWalkGenerator}[kind](G, N)
    env = rbg.Connector(generator=gen, time_limit=time_limit)
    st, ts = env.reset(keys)
    rst, rts = orc.connector_reset_batch(kind, kref, G, N)
    _assert_state(st, rst, "after reset")
    _assert_timestep(ts, rts, "after reset")
    rng = np.random.default_rng(seed)
    n_last = 0
    for t in range(steps):
        if t % 3 == 2:  # unconstrained actions: illegal moves, collisions, out-of-range codes
            act = rng.integers(-1, 7, size=(B, N)).astype(np.int32)
        else:  # the library's random policy (legal moves): long walks, connections
            act = orc.random_actions_batch(rst)
            got = _np(rbg.make_random_policy_connector()(st))
            assert np.array_equal(got, act), f"random policy differs at step {t}"
        if autoreset:
            st, ts = rbg.VmapAutoResetWrapper(env).step(st, torch.from_numpy(act).cuda())
        else:
            st, ts = env.step(st, torch.from_numpy(act).cuda())
        rst, rts = orc.connector_step_batch(rst, act, time_limit=time_limit, autoreset_kind=kind if autoreset else -1)
        _assert_state(st, rst, f"at step {t}")
        _assert_timestep(ts, rts, f"at step {t}")
        n_last += int((rts["step_type"] == 2).sum())
    return n_last


@pytest.mark.parametrize("kind", ["parallel_random_walk", "uniform"])
@pytest.mark.parametrize("G,N", [(5, 3), (10, 5), (7, 6)])
def test_connector_step_matches_oracle(rbg, orc, kind, G, N):
    n_last = _rollout(rbg, orc, kind, G, N, B=1024, steps=30, autoreset=False, time_limit=20)
    assert n_last > 0


@pytest.mark.parametrize("kind", ["parallel_random_walk", "uniform"])
def test_connector_autoreset_matches_oracle(rbg, orc, kind):
    n_last = _rollout(rbg, orc, kind, 10, 5, B=2048, steps=60, autoreset=True, time_limit=25)
    assert n_last > 2048  # every env has been through at least one auto-reset


@pytest.mark.parametrize("kind", ["parallel_random_walk", "uniform", "seed_extension"])
@pytest.mark.parametrize("time_limit", [1, 2, 3])
def test_connector_autoreset_back_to_back_terminations(rbg, orc, kind, time_limit):
    """Every env finishes every `time_limit` steps: the speculative next-episode cache is consumed
    as fast as it can be refilled, so both the cached and the synchronous reset path run."""
    _rollout(rbg, orc, kind, 10, 5, B=700, steps=12, autoreset=True, time_limit=time_limit, seed=17 + time_limit)


def test_workspace_reused_across_generator_kinds(rbg, orc):
    """One auto-reset workspace serving env batches of different generator kinds in turn: speculative
    (next-episode cache, self-clearing counters) -> seed_extension (plain reset lists) -> speculative.
    The library must re-adopt the workspace when the kind changes hands (regression: the
    seed_extension path left its reset count behind and the next batch's lists started mid-buffer)."""
    import torch

    gens = {"parallel_random_walk": rbg.ParallelRandomWalkGenerator, "uniform": rbg.UniformRandomGenerator, "seed_extension": rbg.SeedExtensionGenerator}
    B, G, N = 700, 10, 5
    token = None
    for i, (kind, tl) in enumerate((("uniform", 1), ("seed_extension", 1), ("uniform", 1), ("parallel_random_walk", 2), ("seed_extension", 2), ("parallel_random_walk", 1))):
        env = rbg.Connector(generator=gens[kind](G, N), time_limit=tl)
        if token is not None:
            env._rbg_ws_token = token  # share the first env's workspace
        keys, kref = _keys(rbg, orc, 40 + i, B)
        st, ts = env.reset(keys)
        rst, rts = orc.connector_reset_batch(kind, kref, G, N)
        for t in range(4):
            act = orc.random_actions_batch(rst)
            st, ts = rbg.VmapAutoResetWrapper(env).step(st, torch.from_numpy(act).cuda())
            rst, rts = orc.connector_step_batch(rst, act, time_limit=tl, autoreset_kind=kind)
            _assert_state(st, rst, f"batch {i} ({kind}) step {t}")
            _assert_timestep(ts, rts, f"batch {i} ({kind}) step {t}")
        if token is None:
            token = env._rbg_ws_token


def test_connector_autoreset_two_batches_share_nothing(rbg, orc):
    """Two env batches stepped alternately (different workspaces by shape) stay independent."""
    import torch

    envs, states, refs = [], [], []
    for (G, N, B, seed) in ((10, 5, 512, 1), (8, 4, 384, 2)):
        keys, kref = _keys(rbg, orc, seed, B)
        env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=6))
        st, _ = env.reset(keys)
        rst, _ = orc.connector_reset_batch("parallel_random_walk", kref, G, N)
        envs.append(env), states.append(st), refs.append(rst)
    for t in range(20):
        for i in range(2):
            act = orc.random_actions_batch(refs[i])
            states[i], ts = envs[i].step(states[i], torch.from_numpy(act).cuda())
            refs[i], rts = orc.connector_step_batch(refs[i], act, time_limit=6, autoreset_kind="parallel_random_walk")
            _assert_state(states[i], refs[i], f"batch {i} step {t}")
            _assert_timestep(ts, rts, f"batch {i} step {t}")


def test_connector_autoreset_32x32(rbg, orc):
    _rollout(rbg, orc, "parallel_random_walk", 32, 16, B=256, steps=24, autoreset=True, time_limit=10)


def test_fused_random_step_matches_two_calls(rbg, orc):
    """rbg_connector_step_random == rbg_random_actions + rbg_connector_step."""
    keys, kref = _keys(rbg, orc, 8, 4096)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(10, 5)))
    st, _ = env.reset(keys)
    rst, _ = orc.connector_reset_batch("parallel_random_walk", kref, 10, 5)
    for t in range(55):
        act_ref = orc.random_actions_batch(rst)
        st, ts, act = env.step_random(st)
        assert np.array_equal(_np(act), act_ref)
        rst, rts = orc.connector_step_batch(rst, act_ref, autoreset_kind="parallel_random_walk")
        _assert_state(st, rst, f"at step {t}")
        _assert_timestep(ts, rts, f"at step {t}")


@pytest.mark.parametrize("kind,G,N,B,T,time_limit", [
    ("parallel_random_walk", 10, 5, 3000, 45, 9),     # resets inside every chunk, some envs twice (generator warps)
    ("parallel_random_walk", 32, 16, 96, 12, 9),      # BASELINE configs[4] shape
    ("parallel_random_walk", 10, 5, 1000, 25, 1),     # every step is terminal: the generator warps run constantly
    ("parallel_random_walk", 10, 5, 1000, 25, 2),
    ("parallel_random_walk", 5, 3, 777, 23, 6),       # cells % 4 != 0: scalar path, ragged last warp
    ("parallel_random_walk", 9, 9, 301, 14, 5),       # N > 8: two envs per warp
    ("parallel_random_walk", 12, 20, 130, 14, 7),     # N > 16: one env per warp
    ("parallel_random_walk", 40, 32, 40, 8, 5),       # largest supported shape
    ("parallel_random_walk", 8, 4, 4611, 24, 6),      # ragged last group and ragged last warp
    ("parallel_random_walk", 12, 10, 4099, 22, 7),    # staged views in two alternating buffers (5.7 KB per env)
    ("parallel_random_walk", 6, 12, 310, 21, 4),      # c4 = 9 < 32 lanes, one env per warp
    ("parallel_random_walk", 4, 2, 1300, 21, 3),      # 16 envs per warp, 2 KB of views per step
    ("uniform", 10, 5, 2000, 30, 7),
    ("uniform", 7, 6, 500, 21, 3),
    ("uniform", 8, 8, 4200, 21, 5),                   # Uniform generation in the generator warps
    ("seed_extension", 10, 5, 300, 12, 5),            # no fused kernel for this generator: step-wise path
])
def test_rollout_matches_stepwise_oracle(rbg, orc, kind, G, N, B, T, time_limit):
    """rbg_connector_rollout_random (fused generate + reset + rollout) == T oracle steps."""
    keys, kref = _keys(rbg, orc, 12, B)
    gen = {"parallel_random_walk": rbg.ParallelRandomWalkGenerator, "uniform": rbg.UniformRandomGenerator, "seed_extension": rbg.SeedExtensionGenerator}[kind](G, N)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=gen, time_limit=time_limit))
    st, _ = env.reset(keys)
    rst, _ = orc.connector_reset_batch(kind, kref, G, N)
    st, ts, act = env.rollout_random(st, T)
    for t in range(T):
        a = orc.random_actions_batch(rst)
        assert np.array_equal(_np(act[t]), a), f"actions differ at step {t}"
        rst, rts = orc.connector_step_batch(rst, a, time_limit=time_limit, autoreset_kind=kind)
        _assert_timestep(ts[t], rts, f"at step {t}")
    _assert_state(st, rst, "after the rollout")
    # a second rollout continues from the in-place State (and a warm cache)
    st, ts, act = env.rollout_random(st, 7)
    for t in range(7):
        a = orc.random_actions_batch(rst)
        rst, rts = orc.connector_step_batch(rst, a, time_limit=time_limit, autoreset_kind=kind)
        _assert_timestep(ts[t], rts, f"at step {t} of the second rollout")
    _assert_state(st, rst, "after the second rollout")


@pytest.mark.parametrize("G,N,B,time_limit", [(10, 5, 8200, 6), (10, 5, 4300, 5), (24, 12, 300, 5), (7, 3, 900, 5)])
def test_rollout_step_rollout_matches_oracle(rbg, orc, G, N, B, time_limit):
    """Two fused rollouts of 21 steps, each followed by a step-wise call that shares the auto-reset workspace
    (next-episode cache and group flags) with them: every action, every leaf of every TimeStep and the State
    against the oracle."""
    import torch

    T = 21
    keys, kref = _keys(rbg, orc, 5, B)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=time_limit))
    st, _ = env.reset(keys)
    rst, _ = orc.connector_reset_batch("parallel_random_walk", kref, G, N)
    for rep in range(2):
        st, ts, act = env.rollout_random(st, T)
        for t in range(T):
            a = orc.random_actions_batch(rst)
            assert np.array_equal(_np(act[t]), a), f"actions differ at step {t} of rollout {rep}"
            rst, rts = orc.connector_step_batch(rst, a, time_limit=time_limit, autoreset_kind="parallel_random_walk")
            _assert_timestep(ts[t], rts, f"at step {t} of rollout {rep}")
        _assert_state(st, rst, f"after rollout {rep}")
        st, ts = env.step(st, torch.from_numpy(a).cuda())
        rst, rts = orc.connector_step_batch(rst, a, time_limit=time_limit, autoreset_kind="parallel_random_walk")
        _assert_state(st, rst, f"after the step that follows rollout {rep}")
        _assert_timestep(ts, rts, f"at the step that follows rollout {rep}")


@pytest.mark.parametrize("G,N,B,T,time_limit", [(10, 5, 65536, 45, 50), (32, 16, 8192, 22, 9)])
def test_rollout_full_size_matches_oracle(rbg, orc, G, N, B, T, time_limit):
    """BASELINE configs[1] (65 536 envs, 10x10/5) and configs[4] (32x32/16, 8 192 envs) at FULL size against the
    oracle: every leaf of every TimeStep of the fused rollout (rollout_persist_kernel) and the final State; then the step-by-step path (env_warp_kernel, speculative + synchronous
    reset kernels) continues from that State for a few steps, also against the oracle."""
    import torch

    keys, kref = _keys(rbg, orc, 0, B)
    gen = rbg.ParallelRandomWalkGenerator(G, N)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=gen, time_limit=time_limit))
    st, ts0 = env.reset(keys)
    rst, rts = orc.connector_reset_batch("parallel_random_walk", kref, G, N)
    _assert_state(st, rst, "after reset")
    _assert_timestep(ts0, rts, "after reset")
    chunk = 9 if G == 10 else 11  # an odd chunking of T: the TimeStep stack of a chunk must fit beside the oracle's copy
    resets, t = 0, 0
    out = {k: v.copy() for k, v in rts.items()}
    while t < T:
        n = min(chunk, T - t)
        st, ts, act = env.rollout_random(st, n)
        acts = _np(act)
        for i in range(n):
            a = orc.random_actions_batch(rst)
            assert np.array_equal(acts[i], a), f"actions differ at step {t + i}"
            rst, rts = orc.connector_step_batch(rst, a, time_limit=time_limit, autoreset_kind="parallel_random_walk", inplace=True, out=out)
            _assert_timestep(ts[i], rts, f"at step {t + i}")
            resets += int((rts["step_type"] == 2).sum())
        _assert_state(st, rst, f"after step {t + n}")
        t += n
    assert resets > B // 2, "the run must exercise the auto-reset"
    for i in range(3):
        a = orc.random_actions_batch(rst)
        st, ts1, got = env.step_random(st, inplace=True)
        assert np.array_equal(_np(got), a)
        rst, rts = orc.connector_step_batch(rst, a, time_limit=time_limit, autoreset_kind="parallel_random_walk", inplace=True, out=out)
        _assert_timestep(ts1, rts, f"step-wise step {i} after the rollout")
        _assert_state(st, rst, f"step-wise step {i} after the rollout")


def test_rollout_long_horizon(rbg, orc):
    """1 480 steps over 4 096 envs (6 M env-steps, ~240 k resets) in odd-sized fused chunks: every
    TimeStep leaf of every step and the final State against the oracle."""
    B, G, N, T = 4096, 10, 5, 37
    keys, kref = _keys(rbg, orc, 77, B)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50))
    st, _ = env.reset(keys)
    rst, _ = orc.connector_reset_batch("parallel_random_walk", kref, G, N)
    ts_buf = rbg.engine.alloc_timestep(B, G, N, T)
    resets = 0
    for chunk in range(40):
        st, ts, act = env.rollout_random(st, T, out=ts_buf)
        acts = _np(act)
        obs, mask, rew = _np(ts.observation.grid), _np(ts.observation.action_mask), _np(ts.reward)
        stype, tpl, disc = _np(ts.step_type), _np(ts.extras["total_path_length"]), _np(ts.discount)
        for t in range(T):
            a = orc.random_actions_batch(rst)
            assert np.array_equal(acts[t], a), (chunk, t)
            rst, rts = orc.connector_step_batch(rst, a, time_limit=50, autoreset_kind="parallel_random_walk", inplace=True)
            assert np.array_equal(obs[t], rts["obs"]) and np.array_equal(mask[t], rts["action_mask"]), (chunk, t)
            assert np.array_equal(rew[t].view(np.uint32), rts["reward"].view(np.uint32)) and np.array_equal(disc[t].view(np.uint32), rts["discount"].view(np.uint32)), (chunk, t)
            assert np.array_equal(stype[t], rts["step_type"]) and np.array_equal(tpl[t], rts["total_path_length"]), (chunk, t)
            resets += int((rts["step_type"] == 2).sum())
        _assert_state(st, rst, f"after chunk {chunk}")
    assert resets > 150000


def test_rollout_and_stepwise_calls_interleave(rbg, orc):
    """The fused rollout and the per-step API share one workspace (cache, refill lists)."""
    import torch

    keys, kref = _keys(rbg, orc, 33, 1500)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(10, 5), time_limit=6))
    st, _ = env.reset(keys)
    rst, _ = orc.connector_reset_batch("parallel_random_walk", kref, 10, 5)
    for rnd in range(4):
        for _ in range(5):
            a = orc.random_actions_batch(rst)
            st, ts = env.step(st, torch.from_numpy(a).cuda(), inplace=True)
            rst, rts = orc.connector_step_batch(rst, a, time_limit=6, autoreset_kind="parallel_random_walk")
            _assert_timestep(ts, rts, f"step-wise, round {rnd}")
        st, ts, act = env.rollout_random(st, 11)
        for t in range(11):
            a = orc.random_actions_batch(rst)
            rst, rts = orc.connector_step_batch(rst, a, time_limit=6, autoreset_kind="parallel_random_walk")
            _assert_timestep(ts[t], rts, f"rollout step {t}, round {rnd}")
        _assert_state(st, rst, f"round {rnd}")


def test_multi_to_single_wrapper(rbg, orc):
    keys, kref = _keys(rbg, orc, 8, 64)
    env = rbg.MultiToSingleWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(10, 5)))
    st, ts = env.reset(keys)
    assert ts.reward.shape == (64,) and ts.discount.shape == (64,)
    assert float(ts.discount.min()) == 1.0


def test_reference_env_composition_values(rbg, orc):
    """The composition the reference builds (rl_training/setup_train.py:158-166):
    VmapAutoResetWrapper(MultiToSingleWrapper(Connector(generator))).  reset, step, step_random and
    rollout_random all return the AGGREGATED reward (sum over agents) and discount (max over agents)."""
    import torch

    G, N, B, TL = 8, 4, 700, 6
    keys, kref = _keys(rbg, orc, 15, B)
    env = rbg.VmapAutoResetWrapper(rbg.MultiToSingleWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=TL)))
    st, ts = env.reset(keys)
    rst, rts = orc.connector_reset_batch("parallel_random_walk", kref, G, N)
    assert ts.reward.shape == (B,) and float(ts.reward.abs().max()) == 0.0 and float(ts.discount.min()) == 1.0

    def check(ts, rts, where):
        assert ts.reward.shape == (B,) and ts.discount.shape == (B,), where
        np.testing.assert_allclose(_np(ts.reward), rts["reward"].sum(axis=1, dtype=np.float32), rtol=0, atol=2e-7, err_msg=where)  # float32 sum: order of the N addends is free
        assert np.array_equal(_np(ts.discount), rts["discount"].max(axis=1)), where
        assert np.array_equal(_np(ts.step_type), rts["step_type"]) and np.array_equal(_np(ts.observation.grid), rts["obs"]), where

    seen_mixed = False
    for t in range(14):
        a = orc.random_actions_batch(rst)
        if t % 2:
            st, ts = env.step(st, torch.from_numpy(a).cuda())
        else:
            st, ts, got = env.step_random(st)
            assert np.array_equal(_np(got), a)
        rst, rts = orc.connector_step_batch(rst, a, time_limit=TL, autoreset_kind="parallel_random_walk")
        check(ts, rts, f"step {t}")
        d = rts["discount"]
        seen_mixed |= bool(((d.max(axis=1) == 1) & (d.min(axis=1) == 0)).any())  # max, not min / mean
    assert seen_mixed
    st, ts, act = env.rollout_random(st, 9)
    assert ts.reward.shape == (9, B) and ts.discount.shape == (9, B)
    for t in range(9):
        a = orc.random_actions_batch(rst)
        rst, rts = orc.connector_step_batch(rst, a, time_limit=TL, autoreset_kind="parallel_random_walk")
        check(ts[t], rts, f"rollout step {t}")
    _assert_state(st, rst)


class _CudaFixtureEnv:
    """reset / step of the product package in the terms of tests/test_connector_reference.py."""

    def __init__(self, rbg, m, z):
        self.rbg, self.m = rbg, m
        G, N = m["G"], m["N"]
        g = m["generator"]
        if g.startswith("offline_"):
            gen = rbg.BoardDatasetGeneratorJAX.__new__(rbg.BoardDatasetGeneratorJAX)  # the fixture's own stored boards (the reference's K = 7)
            rbg.Generator.__init__(gen, G, N)
            gen.heads = rbg.engine.as_tensor(z[f"{m['tag']}/dataset_heads"])
            gen.targets = rbg.engine.as_tensor(z[f"{m['tag']}/dataset_targets"])
        else:
            gen = {"parallel_random_walk": rbg.ParallelRandomWalkGenerator, "uniform": rbg.UniformRandomGenerator, "seed_extension": rbg.SeedExtensionGenerator,
                   "sequential_random_walk": rbg.SequentialRandomWalkGenerator}[g](G, N)
        self.env = rbg.Connector(generator=gen, time_limit=m["time_limit"])
        self.vec = rbg.VmapAutoResetWrapper(rbg.MultiToSingleWrapper(self.env) if m.get("aggregate") else self.env)

    @staticmethod
    def _dicts(st, ts):
        d = _state_np(st)
        t = dict(obs=_np(ts.observation.grid), action_mask=_np(ts.observation.action_mask), obs_step_count=_np(ts.observation.step_count), reward=_np(ts.reward),
                 discount=_np(ts.discount), step_type=_np(ts.step_type), num_connections=_np(ts.extras["num_connections"]),
                 ratio_connections=_np(ts.extras["ratio_connections"]), total_path_length=_np(ts.extras["total_path_length"]))
        return d, t

    def reset(self, keys):
        env = self.vec if self.m["kind"] == "vmapped" else self.env
        self.st, ts = env.reset(np.ascontiguousarray(keys))
        return self._dicts(self.st, ts)

    def step(self, _st, action, autoreset):
        import torch

        act = torch.from_numpy(np.ascontiguousarray(action)).cuda()
        self.st, ts = (self.vec if autoreset else self.env).step(self.st, act)
        return self._dicts(self.st, ts)


def test_connector_reference_fixtures_on_gpu(rbg):
    """The CUDA path through the package's public API against tests/golden/connector_reference.npz: TimeSteps of an
    independent second restatement of jumanji's Connector + wrappers driven like the reference drives them
    (tests/tools/make_connector_fixtures.py; N-version agreement, see tests/test_connector_reference.py)."""
    import test_connector_reference as tcr

    z, meta = tcr.load_connector_fixture()
    term = early = 0
    for m in meta:
        if m["kind"] == "vmapped":
            a, b, _ = tcr.run_vmapped(z, m, _CudaFixtureEnv(rbg, m, z))
            term, early = term + a, early + b
        elif m["kind"] == "episodes":
            assert tcr.run_episodes(z, m, _CudaFixtureEnv(rbg, m, z)) > 50
        else:  # demos/board_generator_demo.py:29-97, the private trio
            import torch

            env = rbg.Connector()
            tag = m["tag"]
            for i in range(m["n"]):
                ag = rbg.Agent(id=torch.arange(5, dtype=torch.int32).cuda(), start=torch.from_numpy(z[f"{tag}/s_start"][i].astype(np.int32)).cuda(),
                               target=torch.from_numpy(z[f"{tag}/s_target"][i].astype(np.int32)).cuda(), position=torch.from_numpy(z[f"{tag}/s_position"][i].astype(np.int32)).cuda())
                grid = torch.from_numpy(z[f"{tag}/s_grid"][i].astype(np.int32)).cuda()
                assert np.array_equal(_np(env._obs_from_grid(grid)), z[f"{tag}/t_obs"][i])
                assert np.array_equal(_np(env._get_action_mask_all(ag, grid)), z[f"{tag}/t_action_mask"][i])
                one = rbg.Agent(id=ag.id[2], start=ag.start[2], target=ag.target[2], position=ag.position[2])
                assert np.array_equal(_np(env._get_action_mask(one, grid)), z[f"{tag}/t_action_mask"][i][2])
                ex = env._get_extras(rbg.State(key=torch.zeros(2, dtype=torch.int32).cuda().view(torch.uint32), grid=grid, step_count=torch.zeros((), dtype=torch.int32).cuda(), agents=ag))
                assert int(ex["num_connections"]) == int(z[f"{tag}/t_num_connections"][i]) and int(ex["total_path_length"]) == int(z[f"{tag}/t_total_path_length"][i])
    assert term > 150 and early > 20


@pytest.mark.parametrize("board_name,G,N,K,time_limit", [
    ("offline_parallel_rw", 10, 5, 200, 7),       # rollout_warp_kernel: observation staged in one buffer
    ("offline_seed_extension", 8, 4, 37, 5),
    ("offline_parallel_rw", 5, 3, 3, 2),          # cells % 4 != 0: scalar stores
    ("offline_parallel_rw", 12, 10, 40, 5),       # two alternating staging buffers
    ("offline_parallel_rw", 32, 16, 20, 5),       # direct 128-bit stores
])
def test_connector_with_dataset_generator(rbg, orc, board_name, G, N, K, time_limit):
    """Connector(generator=BoardDatasetGeneratorJAX(...)) as rl_training/setup_train.py:119-133,158 builds it:
    reset, 60 auto-reset steps and a fused rollout against the oracle (the in-kernel reset is a table lookup)."""
    import torch

    B = 300 if G >= 32 else 900  # 32x32/16 emits 64 KB of observation per env-step
    gen = rbg.BoardDatasetGeneratorJAX(G, N, board_name=board_name, number_of_boards=K)
    heads, targets = _np(gen.heads), _np(gen.targets)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=gen, time_limit=time_limit))
    keys, kref = _keys(rbg, orc, 41, B)
    st, ts = env.reset(keys)
    rst = orc.dataset_state_batch(kref, G, N, heads, targets)
    rts = orc.connector_observe_batch(rst)
    _assert_state(st, rst, "after reset")
    _assert_timestep(ts, rts, "after reset")
    rng = np.random.default_rng(1)
    resets = 0
    for t in range(60):
        a = rng.integers(0, 5, size=(B, N)).astype(np.int32) if t % 3 == 2 else orc.random_actions_batch(rst)
        st, ts = env.step(st, torch.from_numpy(a).cuda(), inplace=bool(t % 2))
        rst, rts = orc.connector_step_batch(rst, a, time_limit=time_limit, autoreset_kind="dataset", dataset=(heads, targets))
        _assert_state(st, rst, f"at step {t}")
        _assert_timestep(ts, rts, f"at step {t}")
        resets += int((rts["step_type"] == 2).sum())
    assert resets > 4 * B
    st, ts, act = env.rollout_random(st, 23)
    for t in range(23):
        a = orc.random_actions_batch(rst)
        assert np.array_equal(_np(act[t]), a), f"actions differ at rollout step {t}"
        rst, rts = orc.connector_step_batch(rst, a, time_limit=time_limit, autoreset_kind="dataset", dataset=(heads, targets))
        _assert_timestep(ts[t], rts, f"at rollout step {t}")
    _assert_state(st, rst, "after the rollout")


def test_connector_with_user_defined_generator(rbg, orc):
    """`Generator` is an open ABC in the reference (uniform_generator.py:26-53): any subclass works in Connector.
    This one builds its State with torch ops from the key (two wires on fixed rows, columns from the key bits)."""
    import torch

    G, N, B, TL = 6, 2, 300, 4

    class RowsGenerator(rbg.Generator):
        def __call__(self, key):
            k = rbg.engine.as_keys(key)[0].view(torch.int32).to(torch.int64) & 0xFFFFFFFF
            Bk = k.shape[0]
            c0, c1 = (k[:, 0] % G).int(), (k[:, 1] % G).int()
            start = torch.stack([torch.stack([torch.zeros_like(c0), c0], -1), torch.stack([torch.full_like(c1, 2), c1], -1)], 1)
            target = torch.stack([torch.stack([torch.ones_like(c0) * (G - 1), c1], -1), torch.stack([torch.full_like(c1, 4), c0], -1)], 1)
            grid = torch.zeros((Bk, G, G), dtype=torch.int32, device=k.device)
            b = torch.arange(Bk, device=k.device)
            for i in range(N):
                grid[b, start[:, i, 0].long(), start[:, i, 1].long()] = 2 + 3 * i
                grid[b, target[:, i, 0].long(), target[:, i, 1].long()] = 3 + 3 * i
            newkey = rbg.engine.split_each(rbg.engine.as_keys(key)[0], 2)[:, 0].contiguous()
            return rbg.State(key=newkey, grid=grid, step_count=torch.zeros(Bk, dtype=torch.int32, device=k.device),
                             agents=rbg.Agent(id=torch.arange(N, dtype=torch.int32, device=k.device).expand(Bk, N).contiguous(), start=start.int().contiguous(),
                                              target=target.int().contiguous(), position=start.int().contiguous()))

    gen = RowsGenerator(G, N)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=gen, time_limit=TL))
    keys, kref = _keys(rbg, orc, 43, B)
    st, ts = env.reset(keys)
    rst = {k: v for k, v in _state_np(st).items()}
    rts = orc.connector_observe_batch(rst)
    _assert_timestep(ts, rts, "after reset")
    assert np.array_equal(_np(st.key), np.stack([orc.split(k)[0] for k in kref]))
    resets = 0
    for t in range(13):
        a = orc.random_actions_batch(rst)
        st, ts, got = env.step_random(st)
        assert np.array_equal(_np(got), a)
        prev_key = rst["key"].copy()
        rst, rts = orc.connector_step_batch(rst, a, time_limit=TL)  # plain step, then the wrapper's auto-reset by hand
        last = rts["step_type"] == 2
        if last.any():
            nk = np.stack([orc.split(k)[0] for k in prev_key[last]])
            fresh = _state_np(gen(nk))
            fts = orc.connector_observe_batch(fresh)
            for f in ("grid", "step_count", "agent_id", "start", "target", "position", "key"):
                rst[f][last] = fresh[f]
            for f in ("obs", "action_mask", "obs_step_count"):
                rts[f][last] = fts[f]
        _assert_state(st, rst, f"at step {t}")
        _assert_timestep(ts, rts, f"at step {t}")
        resets += int(last.sum())
    assert resets >= 2 * B


def test_random_policy_is_uniform_over_legal_actions(rbg, orc):
    """make_random_policy_connector (setup_train.py:246) is "distribution-equal", not bit-equal, to upstream's
    masked categorical: chi-square of the sampled actions against the uniform law over each agent's legal
    actions (NOOP included), pooled by number of legal actions; and no illegal action is ever drawn."""
    import torch

    G, N, B = 10, 5, 65536
    keys = rbg.split(rbg.PRNGKey(123), B)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=50))
    st, ts = env.reset(keys)
    for _ in range(6):  # a few steps in, so that masks are diverse
        st, ts, _a = env.step_random(st, inplace=True)
    mask = ts.observation.action_mask  # the mask the policy samples from at the next step
    act = rbg.make_random_policy_connector()(st).long()
    assert bool(mask.gather(2, act[..., None]).all()), "an illegal action was sampled"
    m = mask.reshape(-1, 5).cpu().numpy().astype(bool)
    a = act.reshape(-1).cpu().numpy()
    nlegal = m.sum(axis=1)
    for k in (2, 3, 4, 5):
        sel = nlegal == k
        n = int(sel.sum())
        if n < 5000:
            continue
        # rank of the chosen action among the legal ones must be uniform on {0..k-1}
        rank = (np.cumsum(m[sel], axis=1) - 1)[np.arange(n), a[sel]]
        obs = np.bincount(rank, minlength=k).astype(float)
        chi2 = float(((obs - n / k) ** 2 / (n / k)).sum())
        # 99.99 % quantiles of chi-square with k-1 degrees of freedom: 15.1, 18.4, 21.1, 23.5
        assert chi2 < {2: 15.1, 3: 18.4, 4: 21.1, 5: 23.5}[k], (k, n, obs.tolist(), chi2)
    # different agents / envs / steps draw independently: the action of agent 0 says nothing about agent 1
    both = (nlegal.reshape(B, N)[:, 0] == 5) & (nlegal.reshape(B, N)[:, 1] == 5)
    if both.sum() > 10000:
        tab = np.zeros((5, 5))
        aa = a.reshape(B, N)[both]
        np.add.at(tab, (aa[:, 0], aa[:, 1]), 1)
        exp = tab.sum(1, keepdims=True) * tab.sum(0, keepdims=True) / tab.sum()
        assert float(((tab - exp) ** 2 / exp).sum()) < 45.0  # 16 degrees of freedom, 99.99 % quantile 44.3


def test_state_stepped_twice_keeps_its_boards_pure(rbg, orc):
    """Functional use (inplace=False): the same State stepped again and again while the side stream refills the
    next-episode cache.  A reader must never take a half-rewritten cache entry (seqlock on the tag): every reset
    board is still a pure function of its key."""
    import torch

    G, N, B, TL = 10, 5, 8192, 2
    keys, kref = _keys(rbg, orc, 61, B)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=TL))
    st0, _ = env.reset(keys)
    rst0, _ = orc.connector_reset_batch("parallel_random_walk", kref, G, N)
    a = orc.random_actions_batch(rst0)
    act = torch.from_numpy(a).cuda()
    st1, _ = env.step(st0, act)
    rst1, _ = orc.connector_step_batch(rst0, a, time_limit=TL, autoreset_kind="parallel_random_walk")
    a1 = orc.random_actions_batch(rst1)
    act1 = torch.from_numpy(a1).cuda()
    rst2, rts2 = orc.connector_step_batch(rst1, a1, time_limit=TL, autoreset_kind="parallel_random_walk")  # every env resets here
    assert (rts2["step_type"] == 2).all()
    for rep in range(30):  # st1 over and over, interleaved with steps of its successor that trigger refills of the same entries
        st2, ts2 = env.step(st1, act1)
        _assert_state(st2, rst2, f"rep {rep}")
        _assert_timestep(ts2, rts2, f"rep {rep}")
        a2 = orc.random_actions_batch(rst2)
        st3, _ = env.step(st2, torch.from_numpy(a2).cuda())
        rst3, _ = orc.connector_step_batch(rst2, a2, time_limit=TL, autoreset_kind="parallel_random_walk")
        _assert_state(st3, rst3, f"rep {rep} successor")


def test_unaligned_step_slices_of_a_stacked_rollout(rbg, orc):
    """G*G % 4 != 0: the kernels use scalar accesses and the per-step slices of a stacked rollout are not
    16-byte aligned (5x5/3, B = 1: 75 int32 per step).  The step-wise rollout path (SeedExtension resets) must
    accept them."""
    G, N, B, T, TL = 5, 3, 1, 6, 3
    keys, kref = _keys(rbg, orc, 5, B)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.SeedExtensionGenerator(G, N), time_limit=TL))
    st, _ = env.reset(keys)
    rst, _ = orc.connector_reset_batch("seed_extension", kref, G, N)
    st, ts, act = env.rollout_random(st, T)
    for t in range(T):
        a = orc.random_actions_batch(rst)
        assert np.array_equal(_np(act[t]), a)
        rst, rts = orc.connector_step_batch(rst, a, time_limit=TL, autoreset_kind="seed_extension")
        _assert_timestep(ts[t], rts, f"at step {t}")
    _assert_state(st, rst)


# -------------------------------------------------------------- board validity
def test_validate_matches_reference_verdicts(rbg):
    """rbg_validate against what the reference's own NumPy validity code says about 2 400 generated and corrupted
    boards (tests/golden/validity_reference.npz, made by tests/tools/make_validity_fixtures.py)."""
    import torch
    from test_validity_reference import check_flags_against_reference, load_validity_fixture

    fx = load_validity_fixture()
    n = check_flags_against_reference(fx, lambda boards, N: _np(rbg.engine.validate(torch.from_numpy(boards).cuda(), N)))
    assert n == len(fx["outcome"]) >= 2000


def test_board_statistics_match_reference(rbg, orc):
    """rbg_board_statistics (scored board, count_detours, heatmap_score_diversity) against the outputs of the reference's
    own EvaluateEmptyBoard class (tests/golden/board_stats_reference.npz), then against the oracle on big batches."""
    import torch
    from test_board_stats_reference import check_stats_against_reference, load_stats_fixture

    def cuda_stats(boards, N, ccw):
        s, d, v = rbg.engine.board_statistics(torch.from_numpy(boards).cuda(), count_current_wire=ccw)
        return _np(s), _np(d), _np(v)

    fx = load_stats_fixture()
    assert check_stats_against_reference(fx, cuda_stats) == len(fx["G"]) + len(fx["p_G"])
    ev = rbg.EvaluateEmptyBoard(fx["boards"][0, :5, :5].astype(np.int32))  # the class mirror, single board
    assert np.array_equal(_np(ev.scored_board), fx["scored"][0, :5, :5]) and int(ev.count_detours()) == int(fx["detours"][0, 0])
    assert int(ev.count_detours(True)) == int(fx["detours"][0, 1]) and int(ev.board_statistics["heatmap_score_diversity"]) == int(fx["diversity"][0])
    for (G, N, B) in ((20, 10, 4096), (32, 16, 1024), (40, 32, 256), (3, 2, 1000)):
        boards = orc.prw_generate_batch(orc.split(orc.PRNGKey(9), B), G, N)[2]
        for ccw in (False, True):
            rs, rd, rv = orc.board_statistics_batch(boards, ccw)
            s, d, v = cuda_stats(boards, N, ccw)
            assert np.array_equal(s, rs) and np.array_equal(d, rd) and np.array_equal(v, rv), (G, N, ccw)


def test_validate_matches_oracle_on_corrupted_boards(rbg, orc):
    import torch

    G, N, B = 10, 5, 2048
    keys = orc.split(orc.PRNGKey(4), B)
    boards = orc.prw_generate_batch(keys, G, N)[2]
    rng = np.random.default_rng(0)
    for b in range(0, B, 2):  # corrupt every other board: overwrite 1-3 random cells
        for _ in range(rng.integers(1, 4)):
            boards[b, rng.integers(G), rng.integers(G)] = rng.integers(-1, 3 * N + 2)
    ref = orc.validate_batch(boards, N)
    got = _np(rbg.engine.validate(torch.from_numpy(boards).cuda(), N))
    assert np.array_equal(got, ref)
    assert (ref != 0).sum() > B // 8 and (ref == 0).sum() >= B // 2 - 64
    for (G, N, B) in ((7, 12, 512), (32, 16, 256), (5, 3, 512)):  # dense boards (zero-length wires), big boards, heavier damage
        boards = orc.prw_generate_batch(orc.split(orc.PRNGKey(5), B), G, N)[2]
        for b in range(0, B, 2):
            for _ in range(rng.integers(1, 8)):
                boards[b, rng.integers(G), rng.integers(G)] = rng.integers(0, 3 * N + 1)
        ref = orc.validate_batch(boards, N)
        got = _np(rbg.engine.validate(torch.from_numpy(boards).cuda(), N))
        assert np.array_equal(got, ref), (G, N)


# --------------------------------------------------------------- host variants
def test_host_variants(rbg, orc):
    lib = rbg._lib.load()
    G, N, B = 10, 5, 5000
    kref = orc.split(orc.PRNGKey(6), B)
    heads = np.empty((B, 2, N), np.int32)
    targets = np.empty((B, 2, N), np.int32)
    solved = np.empty((B, G, G), np.int32)
    rc = lib.rbg_prw_generate_host(kref.ctypes.data, B, G, N, heads.ctypes.data, targets.ctypes.data, solved.ctypes.data, -1)
    assert rc == 0, lib.rbg_last_error()
    rh, rt, rs, _ = orc.prw_generate_batch(kref, G, N)
    assert np.array_equal(solved, rs) and np.array_equal(heads, rh) and np.array_equal(targets, rt)


@pytest.mark.parametrize("seed,iters,glo,ghi,bhi", [(2024, 24, 2, 25, 200), (2025, 10, 25, 41, 40)])
def test_random_shapes_sweep(rbg, orc, seed, iters, glo, ghi, bhi):
    """Random (G, N, B) shapes: generators, reset and a short fused rollout against the oracle."""
    rng = np.random.default_rng(seed)
    for it in range(iters):
        G = int(rng.integers(glo, ghi))
        N = int(rng.integers(1, min(32, G * G // 2) + 1))
        B = int(rng.integers(1, bhi))
        keys, kref = _keys(rbg, orc, 100 + it, B)
        heads, targets, solved = rbg.ParallelRandomWalkBoard(G, G, N).generate_board(keys)
        rh, rt, rs, _ = orc.prw_generate_batch(kref, G, N)
        assert np.array_equal(_np(solved), rs) and np.array_equal(_np(heads), rh) and np.array_equal(_np(targets), rt), (G, N, B)
        kind = "uniform" if it % 3 == 0 else "parallel_random_walk"
        gen = (rbg.UniformRandomGenerator if kind == "uniform" else rbg.ParallelRandomWalkGenerator)(G, N)
        tl = int(rng.integers(1, 9))
        env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=gen, time_limit=tl))
        st, ts = env.reset(keys)
        rst, rts = orc.connector_reset_batch(kind, kref, G, N)
        _assert_state(st, rst, (G, N, B))
        _assert_timestep(ts, rts, (G, N, B))
        T = int(rng.integers(1, 12))
        st, tss, act = env.rollout_random(st, T)
        for t in range(T):
            a = orc.random_actions_batch(rst)
            rst, rts = orc.connector_step_batch(rst, a, time_limit=tl, autoreset_kind=kind)
            _assert_timestep(tss[t], rts, (G, N, B, kind, tl, t))
        _assert_state(st, rst, (G, N, B, kind))
        if N <= (G // 2) ** 2:
            sb = rbg.SeedExtensionBoard(G, G, N).return_solved_board(keys)
            assert np.array_equal(_np(sb), orc.seedext_solved_batch(kref, G, N)[0]), ("seed extension", G, N, B)


def test_dlpack_and_numpy_keys(rbg, orc):
    """Keys may come from any DLPack producer (JAX / CuPy arrays in the reference's world) or NumPy;
    results leave as DLPack capsules without a copy."""
    import torch
    from torch.utils import dlpack as tdl

    class Foreign:  # a minimal non-torch DLPack producer
        def __init__(self, t):
            self._t = t

        def __dlpack__(self, stream=None):
            return self._t.__dlpack__()

        def __dlpack_device__(self):
            return self._t.__dlpack_device__()

    kref = orc.split(orc.PRNGKey(9), 300)
    ref = orc.prw_generate_batch(kref, 10, 5)[2]
    board = rbg.ParallelRandomWalkBoard(10, 10, 5)
    dev_keys = torch.from_numpy(kref.view(np.int32)).cuda()
    for keys in (kref, kref.view(np.int32), Foreign(dev_keys), dev_keys, kref.astype(np.int64)):
        assert np.array_equal(_np(board.generate_board(keys)[2]), ref)
    solved = board.generate_board(kref)[2]
    back = tdl.from_dlpack(tdl.to_dlpack(solved))
    assert back.data_ptr() == solved.data_ptr() and np.array_equal(_np(back), ref)
    # single key as a Python list / NumPy vector -> un-batched result, like the reference
    one = board.generate_board([int(kref[0][0]), int(kref[0][1])])[2]
    assert one.shape == (10, 10) and np.array_equal(_np(one), ref[0])


def test_step_host_io_matches_oracle(rbg, orc):
    """rbg_connector_step_host_io: device-resident State, host actions in, host TimeStep out."""
    import torch

    L, lib = rbg._lib, rbg._lib.load()
    G, N, B = 10, 5, 5000
    keys, kref = _keys(rbg, orc, 44, B)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=7))
    st, _ = env.reset(keys)
    rst, _ = orc.connector_reset_batch("parallel_random_walk", kref, G, N)
    h = dict(obs=np.empty((B, N, G, G), np.int32), mask=np.empty((B, N, 5), np.uint8), sc=np.empty(B, np.int32), reward=np.empty((B, N), np.float32), discount=np.empty((B, N), np.float32),
             step_type=np.empty(B, np.int8), nc=np.empty(B, np.int32), rc=np.empty(B, np.float32), tpl=np.empty(B, np.int32))
    a = st.agents
    s = L.rbg_state(st.grid.data_ptr(), st.step_count.data_ptr(), a.id.data_ptr(), a.start.data_ptr(), a.target.data_ptr(), a.position.data_ptr(), st.key.data_ptr())
    t = L.rbg_timestep(*(h[k].ctypes.data for k in ("obs", "mask", "sc", "reward", "discount", "step_type", "nc", "rc", "tpl")))
    params = L.rbg_env_params(7, -0.03, 0.1, 0)
    for step in range(20):
        act = orc.random_actions_batch(rst)
        L.check(lib.rbg_connector_step_host_io(C.byref(s), act.ctypes.data, B, G, N, C.byref(params), C.byref(t), -1))
        rst, rts = orc.connector_step_batch(rst, act, time_limit=7, autoreset_kind="parallel_random_walk")
        assert np.array_equal(h["obs"], rts["obs"]) and np.array_equal(h["mask"], rts["action_mask"]), f"step {step}"
        assert np.array_equal(h["reward"].view(np.uint32), rts["reward"].view(np.uint32)) and np.array_equal(h["step_type"], rts["step_type"])
        assert np.array_equal(h["tpl"], rts["total_path_length"]) and np.array_equal(h["sc"], rts["obs_step_count"])
        _assert_state(st, rst, f"step {step}")


_HOST_IO_CODE = """
import ctypes as C, sys, numpy as np
sys.path.insert(0, {root!r})
import routing_board_generation_b200 as rbg
from oracle import oracle as orc
L, lib = rbg._lib, rbg._lib.load()
G, N, B, TL = {G}, {N}, {B}, {TL}
kref = orc.split(orc.PRNGKey(77), B)
keys = rbg.engine.as_tensor(kref)
env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=TL))
st, _ = env.reset(keys)
rst, _ = orc.connector_reset_batch("parallel_random_walk", kref, G, N)
pad = 3  # the observation buffer starts 12 bytes into its allocation when the vector path is not needed
ob = np.full(B * N * G * G + 8, -1, np.int32)
o0 = pad if (G * G) % 4 else 0
obs = ob[o0:o0 + B * N * G * G].reshape(B, N, G, G)
h = dict(obs=obs, mask=np.empty((B, N, 5), np.uint8), sc=np.empty(B, np.int32), reward=np.empty((B, N), np.float32), discount=np.empty((B, N), np.float32),
         step_type=np.empty(B, np.int8), nc=np.empty(B, np.int32), rc=np.empty(B, np.float32), tpl=np.empty(B, np.int32))
a = st.agents
s = L.rbg_state(st.grid.data_ptr(), st.step_count.data_ptr(), a.id.data_ptr(), a.start.data_ptr(), a.target.data_ptr(), a.position.data_ptr(), st.key.data_ptr())
t = L.rbg_timestep(*(h[k].ctypes.data for k in ("obs", "mask", "sc", "reward", "discount", "step_type", "nc", "rc", "tpl")))
params = L.rbg_env_params(TL, -0.03, 0.1, 0)
L.host_transfer_stats(reset=True)
for step in range(6):
    act = orc.random_actions_batch(rst)
    L.check(lib.rbg_connector_step_host_io(C.byref(s), act.ctypes.data, B, G, N, C.byref(params), C.byref(t), -1))
    rst, rts = orc.connector_step_batch(rst, act, time_limit=TL, autoreset_kind="parallel_random_walk")
    assert np.array_equal(obs, rts["obs"]) and np.array_equal(h["mask"], rts["action_mask"]), step
    assert np.array_equal(h["reward"].view(np.uint32), rts["reward"].view(np.uint32)) and np.array_equal(h["step_type"], rts["step_type"]), step
    assert np.array_equal(h["tpl"], rts["total_path_length"]) and np.array_equal(h["sc"], rts["obs_step_count"]) and np.array_equal(h["nc"], rts["num_connections"]), step
assert (ob[:o0] == -1).all() and (ob[o0 + B * N * G * G:] == -1).all()  # nothing written around the buffer
h2d, d2h, threads = L.host_transfer_stats()
small = B * (N * 5 + 4 + N * 8 + 1 + 12)
obs_moved = B * N * G * G
if 3 * N <= 15 and (N * G * G) % 2 == 0:
    obs_moved //= 2  # codes <= 15: two cells per byte over the bus
assert h2d == 6 * B * N * 4 and d2h == 6 * (obs_moved + small), (h2d, d2h)
assert threads > 0
print("ok", threads)
"""


@pytest.mark.gpu
@pytest.mark.parametrize("env_vars,G,N,B", [({}, 5, 3, 4101), ({}, 7, 2, 70), ({"RBG_HOST_THREADS": "3"}, 10, 5, 9000),
                                            ({"RBG_HOST_THREADS": "3"}, 10, 5, 33001), ({}, 10, 5, 4500),
                                            ({}, 5, 3, 33001), ({}, 10, 5, 4133), ({}, 8, 4, 300), ({}, 9, 6, 700), ({}, 6, 5, 131),
                                            ({}, 20, 1, 300), ({}, 28, 2, 150), ({}, 40, 4, 70)])
def test_step_host_io_transports(env_vars, G, N, B):
    """rbg_connector_step_host_io moves the observation as bytes (as nibbles when the codes are <= 15: at most 5 agents and
    an even number of cells per env) and widens it on the host threads of the call: same TimeSteps as the oracle with 1, 8
    and 16 slices (B >= 32768) of either code width, ragged last slices, shapes without the vector path, unpinned and
    odd-aligned destination, few agents on boards whose step needs more than 48 KB of shared memory, and the byte
    counters say what crossed."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = _HOST_IO_CODE.format(root=root, G=G, N=N, B=B, TL=3)
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env_vars), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip().startswith("ok"), (r.stdout[-800:], r.stderr[-2000:])


def test_step_host_io_survives_other_host_calls(rbg, orc):
    """The host-variant step keeps its auto-reset workspaces in the library's device scratch.  Another
    host-variant call in between overwrites that scratch, and a new env batch of the same shape comes
    next: the step must notice and start from a clean workspace (every env resets every step here)."""
    L, lib = rbg._lib, rbg._lib.load()
    G, N, B = 10, 5, 4500
    params = L.rbg_env_params(1, -0.03, 0.1, 0)
    h = dict(obs=np.empty((B, N, G, G), np.int32), mask=np.empty((B, N, 5), np.uint8), sc=np.empty(B, np.int32), reward=np.empty((B, N), np.float32), discount=np.empty((B, N), np.float32),
             step_type=np.empty(B, np.int8), nc=np.empty(B, np.int32), rc=np.empty(B, np.float32), tpl=np.empty(B, np.int32))
    t = L.rbg_timestep(*(h[k].ctypes.data for k in ("obs", "mask", "sc", "reward", "discount", "step_type", "nc", "rc", "tpl")))
    for batch in range(3):
        keys, kref = _keys(rbg, orc, 60 + batch, B)
        env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.ParallelRandomWalkGenerator(G, N), time_limit=1))
        st, _ = env.reset(keys)
        rst, _ = orc.connector_reset_batch("parallel_random_walk", kref, G, N)
        a = st.agents
        s = L.rbg_state(st.grid.data_ptr(), st.step_count.data_ptr(), a.id.data_ptr(), a.start.data_ptr(), a.target.data_ptr(), a.position.data_ptr(), st.key.data_ptr())
        for step in range(3):
            act = orc.random_actions_batch(rst)
            L.check(lib.rbg_connector_step_host_io(C.byref(s), act.ctypes.data, B, G, N, C.byref(params), C.byref(t), -1))
            rst, rts = orc.connector_step_batch(rst, act, time_limit=1, autoreset_kind="parallel_random_walk")
            assert np.array_equal(h["obs"], rts["obs"]) and np.array_equal(h["step_type"], rts["step_type"]), (batch, step)
            _assert_state(st, rst, f"batch {batch} step {step}")
        # something else uses (and overwrites) the scratch
        n2 = 6000 + 500 * batch
        k2 = orc.split(orc.PRNGKey(9), n2)
        heads, targets, solved = np.empty((n2, 2, N), np.int32), np.empty((n2, 2, N), np.int32), np.empty((n2, G, G), np.int32)
        assert lib.rbg_prw_generate_host(k2.ctypes.data, n2, G, N, heads.ctypes.data, targets.ctypes.data, solved.ctypes.data, -1) == 0
        assert np.array_equal(solved, orc.prw_generate_batch(k2, G, N)[2])


def test_mixed_api_stress(rbg):
    """tools/stress_mixed.py: env batches of all generator kinds created, stepped in random order through
    step / step_random / rollout_random and dropped at random (workspaces change hands), every result
    against the oracle."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "stress_mixed.py"), "160", "7"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and r.stdout.strip().startswith("ok"), (r.stdout[-800:], r.stderr[-2000:])


def test_cabi_argument_errors(rbg):
    """Bad arguments come back as negative codes with a message, never as a crash or a silent fallback."""
    import torch

    lib = rbg._lib.load()
    keys = rbg.split(rbg.PRNGKey(0), 8)
    out = torch.empty(8 * 100 + 1, dtype=torch.int32, device="cuda")
    h = torch.empty((8, 2, 5), dtype=torch.int32, device="cuda")
    # solved not 16-byte aligned
    assert lib.rbg_prw_generate(keys.data_ptr(), 8, 10, 5, h.data_ptr(), h.data_ptr(), out.data_ptr() + 4, None, None) == -2
    assert b"aligned" in lib.rbg_last_error()
    assert lib.rbg_prw_generate(keys.data_ptr(), -1, 10, 5, h.data_ptr(), h.data_ptr(), out.data_ptr(), None, None) == -1
    assert lib.rbg_prw_generate(keys.data_ptr(), 8, 10, 33, h.data_ptr(), h.data_ptr(), out.data_ptr(), None, None) == -1
    assert lib.rbg_seedext_solved(keys.data_ptr(), 8, 6, 10, 0.0, 1, 1, -1, out.data_ptr(), None) == -1  # lattice too small
    st = rbg.ParallelRandomWalkGenerator(10, 5)(keys)
    ts = rbg.engine.alloc_timestep(8, 10, 5)
    s, t = rbg.engine._state_struct(st), rbg.engine._timestep_struct(ts)
    params = rbg._lib.rbg_env_params(50, -0.03, 0.1, 0)
    act = torch.zeros((8, 5), dtype=torch.int32, device="cuda")
    # auto-reset without a workspace
    assert lib.rbg_connector_step(C.byref(s), C.byref(s), act.data_ptr(), 8, 10, 5, C.byref(params), C.byref(t), None, None) == -1
    assert b"workspace" in lib.rbg_last_error()
    params = rbg._lib.rbg_env_params(50, -0.03, 0.1, 7)  # unknown generator kind
    ws = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    assert lib.rbg_connector_step(C.byref(s), C.byref(s), act.data_ptr(), 8, 10, 5, C.byref(params), C.byref(t), ws.data_ptr(), None) == -1
    assert lib.rbg_kernel_time(99, None, None) == -1


def test_errors_are_reported_not_swallowed(rbg):
    import torch

    keys = rbg.split(rbg.PRNGKey(0), 4)
    with pytest.raises(rbg.RbgError):
        rbg.ParallelRandomWalkBoard(41, 41, 3).generate_board(keys)
    with pytest.raises(rbg.RbgError):
        rbg.ParallelRandomWalkBoard(3, 3, 10).generate_board(keys)  # N > G*G: choice(replace=False) would raise
    with pytest.raises(ValueError):
        rbg.ParallelRandomWalkBoard(4, 5, 2)
    with pytest.raises(ValueError):
        rbg.ParallelRandomWalkBoard(5, 5, 2).generate_board(torch.zeros(3, dtype=torch.int32, device="cuda"))


# ------------------------------------------------------ SequentialRandomWalk
def _seqrw_fixtures():
    import json
    import os

    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "seqrw_reference.json")) as f:
        return json.load(f)


def test_seqrw_reference_fixtures_on_gpu(rbg):
    """The CUDA path against the reference's own SequentialRandomWalkBoard / SequentialRandomWalkGenerator run on the
    jax shim (tests/golden/seqrw_reference.json, made by tests/tools/make_seqrw_fixtures.py): boards that succeed at once,
    boards that need several attempts, boards on which every attempt fails."""
    import torch

    fx = _seqrw_fixtures()
    assert fx["numpy_log_strictly_monotone_on_all_uniforms"] and fx["gumbel_draws_checked"] > 5000
    seen = set()
    for cfg in fx["generate"]:
        board = rbg.SequentialRandomWalkBoard(cfg["G"], cfg["G"], cfg["N"])
        key = torch.tensor(cfg["key"], dtype=torch.int64)
        out = board.generate(key)
        assert out.dtype == torch.float32 and out.shape == (cfg["G"], cfg["G"])  # the reference's dtype (jnp.zeros default)
        assert _np(out).astype(np.int64).tolist() == cfg["board"], cfg["key"]
        b2, stats = board.generate_with_stats(key)
        assert b2.dtype == torch.int32 and _np(b2).tolist() == cfg["board"] and int(stats[0]) == cfg["attempt"]
        seen.add(0 if cfg["attempt"] == 0 else 1 if cfg["attempt"] == 1 else 2)
    assert seen == {0, 1, 2}
    for cfg in fx["starts_ends"]:
        (sr, sc), (er, ec) = rbg.SequentialRandomWalkBoard(cfg["G"], cfg["G"], cfg["N"]).generate_starts_ends(torch.tensor(cfg["key"], dtype=torch.int64))
        assert [_np(sr).tolist(), _np(sc).tolist()] == cfg["starts"] and [_np(er).tolist(), _np(ec).tolist()] == cfg["ends"], cfg["key"]
    for cfg in fx["generator_states"]:
        st = rbg.SequentialRandomWalkGenerator(cfg["G"], cfg["N"])(torch.tensor(cfg["key_in"], dtype=torch.int64))
        assert _np(st.key).tolist() == cfg["key"] and _np(st.grid).tolist() == cfg["grid"] and int(st.step_count) == cfg["step_count"]
        assert _np(st.agents.id).tolist() == cfg["agent_id"] and _np(st.agents.start).tolist() == cfg["start"]
        assert _np(st.agents.target).tolist() == cfg["target"] and _np(st.agents.position).tolist() == cfg["position"]


@pytest.mark.parametrize("G,N,B", [(3, 1, 257), (3, 4, 2048), (4, 6, 2048), (5, 3, 2048), (6, 12, 1024), (7, 4, 2048), (10, 5, 4096), (10, 20, 512), (14, 7, 2048), (17, 9, 512),
                                   (20, 10, 1024), (32, 16, 256), (40, 32, 64)])
def test_seqrw_generate_matches_oracle(rbg, orc, G, N, B):
    keys, kref = _keys(rbg, orc, 11, B)
    board = rbg.SequentialRandomWalkBoard(G, G, N)
    got, stats = board.generate_with_stats(keys)
    ref, rstats = orc.seqrw_generate_batch(kref, G, N)
    assert np.array_equal(_np(stats), rstats), "attempt / step counts differ"
    assert np.array_equal(_np(got), ref)
    assert np.array_equal(_np(board.generate(keys)), ref.astype(np.float32))
    (sr, sc), (er, ec) = board.generate_starts_ends(keys)
    for b in range(0, B, max(1, B // 64)):
        rs, re_ = orc.seqrw_starts_ends(kref[b], G, N)
        assert np.array_equal(np.stack([_np(sr)[b], _np(sc)[b]]), rs) and np.array_equal(np.stack([_np(er)[b], _np(ec)[b]]), re_)
    # a generated board is sound by the reference's validity rules; a failed one is all zeros
    ok = rstats[:, 0] > 0
    flags = _np(rbg.engine.validate(got, N))
    assert ((flags[ok] & (1 | 8 | 32 | 64 | 128)) == 0).all()
    assert (ref[~ok] == 0).all()


@pytest.mark.parametrize("G,N", [(3, 4), (5, 3), (10, 5), (14, 7)])
def test_seqrw_generator_state_matches_oracle(rbg, orc, G, N):
    keys, kref = _keys(rbg, orc, 5, 777)
    _assert_state(rbg.SequentialRandomWalkGenerator(G, N)(keys), orc.state_batch("sequential_random_walk", kref, G, N))


def test_seqrw_single_key_ragged_and_errors(rbg, orc):
    k = rbg.PRNGKey(42)
    out = rbg.SequentialRandomWalkBoard(6, 6, 3).generate(k, as_float32=False)
    assert out.shape == (6, 6) and np.array_equal(_np(out), orc.seqrw_generate(orc.PRNGKey(42), 6, 3))
    for B in (1, 3, 15, 16, 17, 129):
        keys, kref = _keys(rbg, orc, 9, B)
        assert np.array_equal(_np(rbg.SequentialRandomWalkBoard(8, 8, 4).generate(keys, as_float32=False)), orc.seqrw_generate_batch(kref, 8, 4)[0])
    import torch

    # more agents than cells: every attempt fails (zero board, every pin at (0, 0)), as the reference's loop would end
    keys, kref = _keys(rbg, orc, 9, 40)
    assert not _np(rbg.SequentialRandomWalkBoard(3, 3, 12).generate(keys)).any() and not orc.seqrw_generate_batch(kref, 3, 12)[0].any()
    _assert_state(rbg.SequentialRandomWalkGenerator(3, 12)(keys), orc.state_batch("sequential_random_walk", kref, 3, 12))
    empty = torch.empty((0, 2), dtype=torch.uint32, device="cuda")
    assert rbg.SequentialRandomWalkBoard(8, 8, 4).generate(empty).shape == (0, 8, 8)
    assert rbg.SequentialRandomWalkGenerator(8, 4)(empty).grid.shape == (0, 8, 8)
    with pytest.raises(ValueError):
        rbg.SequentialRandomWalkBoard(2, 2, 1)
    with pytest.raises(ValueError):
        rbg.SequentialRandomWalkBoard(5, 6, 2)
    import torch

    lib = rbg._lib.load()
    keys = rbg.split(rbg.PRNGKey(0), 4)
    out = torch.empty((4, 2, 2), dtype=torch.int32, device="cuda")
    assert lib.rbg_seqrw_generate(keys.data_ptr(), 4, 2, 1, out.data_ptr(), 0, None, None) == -1  # rows < 3


def test_seqrw_connector_autoreset_matches_oracle(rbg, orc):
    """Connector(generator=SequentialRandomWalkGenerator) as `online_seq_rw` builds it (setup_train.py:137-141,158): reset, steps,
    auto-resets through the reset-list path; crowded boards include failed generations (every pin at (0, 0))."""
    n_last = _rollout(rbg, orc, "sequential_random_walk", 10, 5, B=512, steps=40, autoreset=True, time_limit=15)
    assert n_last > 512
    _rollout(rbg, orc, "sequential_random_walk", 3, 4, B=300, steps=9, autoreset=True, time_limit=2, seed=23)
    _rollout(rbg, orc, "sequential_random_walk", 6, 3, B=300, steps=12, autoreset=False, time_limit=8, seed=24)


def test_seqrw_rollout_random_matches_oracle(rbg, orc):
    G, N, B, T, TL = 8, 4, 600, 14, 5
    keys, kref = _keys(rbg, orc, 31, B)
    env = rbg.VmapAutoResetWrapper(rbg.Connector(generator=rbg.SequentialRandomWalkGenerator(G, N), time_limit=TL))
    st, _ = env.reset(keys)
    rst, _ = orc.connector_reset_batch("sequential_random_walk", kref, G, N)
    st, ts, act = env.rollout_random(st, T)
    for t in range(T):
        a = orc.random_actions_batch(rst)
        assert np.array_equal(_np(act[t]), a), t
        rst, rts = orc.connector_step_batch(rst, a, time_limit=TL, autoreset_kind="sequential_random_walk")
        assert np.array_equal(_np(ts.observation.grid[t]), rts["obs"]) and np.array_equal(_np(ts.step_type[t]), rts["step_type"]), t
        assert np.array_equal(_np(ts.reward[t]).view(np.uint32), rts["reward"].view(np.uint32)), t
    _assert_state(st, rst, "after the rollout")


@pytest.mark.parametrize("G,N,B", [(10, 5, 65536), (20, 10, 16384)])
def test_seqrw_full_size_invariants(rbg, G, N, B):
    """Size-independent properties at full batch size, on the device: a successful board holds one head and one target per
    wire, exactly steps + N filled cells (a step fills one cell, a wire starts on one), passes the reference's validity rules;
    a failed one is all zeros.  Idempotence: the same keys give the same boards."""
    import torch

    keys = rbg.split(rbg.PRNGKey(0), B)
    gen = rbg.SequentialRandomWalkBoard(G, G, N)
    board, stats = gen.generate_with_stats(keys)
    ok = stats[:, 0] > 0
    assert int(ok.sum()) > 0.99 * B
    assert int((board != 0).sum(dim=(1, 2))[~ok].sum()) == 0
    assert torch.equal((board != 0).sum(dim=(1, 2))[ok], (stats[:, 1] + N)[ok].to(torch.int64))
    for w in range(N):
        assert torch.equal(((board == 3 * w + 2).sum(dim=(1, 2)) == 1), ok) and torch.equal(((board == 3 * w + 3).sum(dim=(1, 2)) == 1), ok)
    flags = rbg.engine.validate(board, N)
    assert int((flags[ok] & (1 | 8 | 32 | 64 | 128)).abs().max()) == 0
    assert int(stats[:, 0].max()) < 2 * G and int(stats[:, 0].min()) >= 0
    again = gen.generate(keys, as_float32=False)
    assert torch.equal(again, board)


@pytest.mark.parametrize("lanes", ["6", "8"])
def test_seqrw_lanes_per_board_switch(lanes):
    """seqrw_walk_kernel comes with 6 or 8 lanes per board (6 by default up to 16x16, 8 beyond): RBG_SEQRW_W forces either one
    on every shape, incl. crowded boards (retries, failed generations) and a board larger than the default range of each."""
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import sys, numpy as np; sys.path.insert(0, %r)\n"
        "import routing_board_generation_b200 as rbg\n"
        "from oracle import oracle as orc\n"
        "for G, N, B in ((3, 4, 600), (4, 6, 600), (7, 4, 1500), (10, 5, 3000), (10, 20, 300), (17, 9, 300), (20, 10, 400), (33, 8, 60)):\n"
        "    k = rbg.split(rbg.PRNGKey(13), B); kr = orc.split(orc.PRNGKey(13), B)\n"
        "    b, s = rbg.SequentialRandomWalkBoard(G, G, N).generate_with_stats(k)\n"
        "    rb, rs = orc.seqrw_generate_batch(kr, G, N)\n"
        "    assert np.array_equal(b.cpu().numpy(), rb) and np.array_equal(s.cpu().numpy(), rs), (G, N)\n"
        "    st = rbg.SequentialRandomWalkGenerator(G, N)(k)\n"
        "    assert np.array_equal(st.grid.cpu().numpy(), orc.state_batch('sequential_random_walk', kr, G, N)['grid']), (G, N)\n"
        "print('ok')\n"
    ) % root
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, RBG_SEQRW_W=lanes), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip().startswith("ok"), (r.stdout[-500:], r.stderr[-2000:])
