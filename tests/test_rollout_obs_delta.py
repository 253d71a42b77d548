"""The fused rollout kernels' delta staging of observation.grid, against the oracle.

When one warp's whole observation range fits its staging buffer (10x10/5, 8x8/4, 6x6/3, 4x4/2), the fused rollout
kernels keep step t's views in shared memory and restage at step t + 1 only the cells that changed: the two cells of
each agent that moved, and everything of an env that reset.  The first step of every group of envs a warp takes is
staged in full.  The cases below run that path where it is hardest to get right: every env resetting at every step
(time_limit 1), persistent warps taking about nine groups per launch at full size, a ragged last group, and two
20-step launches chained on the stream, the second starting under the tail of the first.  Every TimeStep leaf of
every step and the final State are compared exactly (float32 values by their bits).
"""
import pytest

from test_connector_shapes import _check_rollout, _env, _reset

pytestmark = pytest.mark.gpu

T = 40  # two 20-step launches in one call, chained on the stream


@pytest.mark.parametrize("time_limit", [1, 2, 3])
@pytest.mark.parametrize("B", [65536, 65539])
def test_rollout_delta_full_size(rbg, orc, B, time_limit):
    """The headline shape, 10x10/5 with ParallelRandomWalk resets (rollout_persist_kernel), at full size and with a
    ragged last group."""
    G, N, kind = 10, 5, "parallel_random_walk"
    env = rbg.VmapAutoResetWrapper(_env(rbg, kind, G, N, time_limit))
    st, rst, ds = _reset(rbg, orc, env, kind, G, N, B, seed=B + time_limit)
    _check_rollout(rbg, orc, env, st, rst, kind, T, time_limit, ds, where=f"(B={B}, time_limit={time_limit})")


@pytest.mark.parametrize("time_limit", [1, 3])
@pytest.mark.parametrize("kind", ["parallel_random_walk", "uniform", "dataset"])
@pytest.mark.parametrize("G,N", [(10, 5), (8, 4), (6, 3), (4, 2)])
def test_rollout_delta_shapes(rbg, orc, G, N, kind, time_limit):
    """Every shape that takes the delta path, with each generator: the persistent kernel for ParallelRandomWalk and
    Uniform, rollout_warp_kernel for the dataset.  20 011 envs: several groups per persistent warp, the last one
    ragged."""
    B = 20011
    env = rbg.VmapAutoResetWrapper(_env(rbg, kind, G, N, time_limit))
    st, rst, ds = _reset(rbg, orc, env, kind, G, N, B, seed=G * 100 + N * 10 + time_limit)
    st, rst = _check_rollout(rbg, orc, env, st, rst, kind, T, time_limit, ds, where="(first call)")
    _check_rollout(rbg, orc, env, st, rst, kind, 7, time_limit, ds, where="(second call)")
