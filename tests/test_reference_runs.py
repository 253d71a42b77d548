"""The CPU oracle against outputs of the REFERENCE'S OWN Python source.

tests/golden/reference_runs.json was produced by tests/tools/make_reference_fixtures.py, which
imports the reference's files unmodified from a checkout of the reference and runs them on the NumPy
stand-in for jax in tests/tools/jax_shim (jax / jumanji are not installable here).  This pins what the
reference's own goldens do not cover: the ParallelRandomWalk collision branch, SeedExtension with
every option, and the three generators' States.  No GPU needed.

The last two tests run the reference's own source, which this repository does not contain: they
skip unless RBG_REFERENCE names a checkout of mwolinska/Routing-Board-Generation.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("RBG_REFERENCE", "")
needs_reference = pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, "routing_board_generation"))), reason="RBG_REFERENCE does not name a checkout of the reference")


@pytest.fixture(scope="module")
def runs():
    with open(os.path.join(ROOT, "tests", "golden", "reference_runs.json")) as f:
        return json.load(f)


def test_prw_generate_board_incl_collisions(orc, runs):
    collided = 0
    for cfg in runs["prw_generate_board"]:
        G, N = cfg["G"], cfg["N"]
        keys = orc.split(orc.PRNGKey(cfg["seed"]), cfg["n"])
        heads, targets, solved, stats = orc.prw_generate_batch(keys, G, N)
        for b, row in enumerate(cfg["boards"]):
            assert solved[b].tolist() == row["solved"], (G, N, b)
            assert heads[b].tolist() == row["heads"] and targets[b].tolist() == row["targets"]
        collided += int(stats[:, 1].sum())
    assert collided >= 20  # the fixtures exercise parallel_random_walk.py:127-145 many times


def test_generator_states(orc, runs):
    for cfg in runs["generator_states"]:
        keys = orc.split(orc.PRNGKey(cfg["seed"]), cfg["n"])
        st = orc.state_batch(cfg["kind"], keys, cfg["G"], cfg["N"])
        for b, ref in enumerate(cfg["states"]):
            where = (cfg["kind"], cfg["G"], cfg["N"], b)
            assert st["grid"][b].tolist() == ref["grid"], where
            assert st["key"][b].tolist() == ref["key"], where
            assert st["start"][b].tolist() == ref["start"] and st["target"][b].tolist() == ref["target"], where
            assert st["position"][b].tolist() == ref["position"] and st["agent_id"][b].tolist() == ref["id"], where
            assert int(st["step_count"][b]) == ref["step_count"]


def _okw(opt):
    return dict(randomness=opt.get("randomness", 0.0), two_sided=opt.get("two_sided", True), iterations=opt.get("extension_iterations", 1), ext_steps=int(opt.get("extension_steps", -1)))


def test_seedext_solved_and_starts_ends(orc, runs):
    for cfg in runs["seedext_solved"]:
        G, N, kw = cfg["G"], cfg["N"], _okw(cfg["options"])
        keys = orc.split(orc.PRNGKey(cfg["seed"]), cfg["n"])
        boards, _ = orc.seedext_solved_batch(keys, G, N, **kw)
        for b, row in enumerate(cfg["boards"]):
            assert boards[b].tolist() == row["solved"], (G, N, cfg["options"], b)
            s, e = orc.seedext_starts_ends(keys[b], G, N, **kw)
            assert s.tolist() == row["starts"] and e.tolist() == row["ends"], (G, N, cfg["options"], b)


def test_seedext_stages(orc, runs):
    for row in runs["seedext_stages"]:
        G, N, key = row["G"], row["N"], np.array(row["key"], np.uint32)
        seeded = orc.seedext_seeded_board(key, G, N)
        assert seeded.tolist() == row["seeded"]
        ext, _ = orc.extend_wires(seeded, key)
        assert ext.tolist() == row["extended"]
        opt, _, rc = orc.optimise_wire(key, ext, 0)
        assert rc == 0 and opt.tolist() == row["optimised_wire0"]


def test_dataset_generator(orc, runs):
    """BoardDatasetGeneratorJAX (dataset_generator_jax.py): stored boards and the randint pick."""
    assert runs.get("dataset_generator"), "fixtures missing: rerun tests/tools/make_reference_fixtures.py dataset"
    for cfg in runs["dataset_generator"]:
        G, N, K = cfg["G"], cfg["N"], cfg["K"]
        kref = orc.split(orc.PRNGKey(0), K)
        if cfg["board_name"] == "offline_seed_extension":
            ref = [orc.seedext_starts_ends(kref[b], G, N, randomness=1.0, two_sided=False) for b in range(K)]
            rh, rt = np.stack([r[0] for r in ref]), np.stack([r[1] for r in ref])
        else:
            rh, rt, _, _ = orc.prw_generate_batch(kref, G, N)
        assert rh.tolist() == cfg["heads"] and rt.tolist() == cfg["targets"]
        keys = orc.split(orc.PRNGKey(cfg["seed"]), cfg["n"])
        st = orc.dataset_state_batch(keys, G, N, rh, rt)
        for b, ref_st in enumerate(cfg["states"]):
            assert st["grid"][b].tolist() == ref_st["grid"] and st["key"][b].tolist() == ref_st["key"]
            assert st["start"][b].tolist() == ref_st["start"] and st["target"][b].tolist() == ref_st["target"]


@needs_reference
def test_shim_passes_the_references_own_tests(tmp_path):
    """The NumPy jax stand-in the fixtures were made with runs the reference's only test file green."""
    shim = os.path.join(ROOT, "tests", "tools", "jax_shim")
    test = os.path.join(REF, "routing_board_generation/board_generation_methods/jax_implementation/board_generation/test_parallel_random_walk_board.py")
    env = dict(os.environ, PYTHONPATH=shim + os.pathsep + REF)
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", test], cwd=tmp_path, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:]
    assert "35 passed" in r.stdout


@needs_reference
def test_sequential_random_walk_is_not_instantiable(tmp_path):
    """SURVEY 8(f).4: SequentialRandomWalkBoard subclasses the NumPy AbstractBoard without implementing
    its abstract methods, so the reference cannot construct it (nor the generator built on it) as shipped.
    The engine's mirror IS instantiable and reproduces the method bodies, which tests/tools/make_seqrw_fixtures.py
    runs with the abstract-method check lifted (DESIGN.md section 8, f4)."""
    shim = os.path.join(ROOT, "tests", "tools", "jax_shim")
    code = (
        "from routing_board_generation.board_generation_methods.jax_implementation.board_generation.sequential_random_walk import SequentialRandomWalkBoard\n"
        "try:\n"
        "    SequentialRandomWalkBoard(6, 6, 3)\n"
        "except TypeError as e:\n"
        "    print('TypeError:', e)\n"
    )
    env = dict(os.environ, PYTHONPATH=shim + os.pathsep + REF)
    r = subprocess.run([sys.executable, "-c", code], cwd=tmp_path, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "TypeError" in r.stdout and "abstract" in r.stdout
