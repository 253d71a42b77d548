"""Batched board statistics and random-agent / policy evaluation on the CUDA engine.

Mirrors `EvaluateEmptyBoard` (routing_board_generation/benchmarking/benchmarks/empty_board_evaluation.py:31-155),
the per-board consumer of solved boards in the reference's benchmark
(`evaluate_generator_outputs_averaged_on_n_boards`, :158-225): `scored_board`, `count_detours()` and the
`heatmap_score_diversity` entry of `board_statistics`.  A board [G,G] or a batch [B,G,G].

The reference's constructor first sends the board through `BoardProcessor`, which re-routes every wire along a
shortest path picked with an unseeded `random.shuffle` (board_processor.py:111-162); that preprocessing and the
wire-length / bend statistics derived from it have no deterministic result and are not reproduced: the board is
scored as given (for boards whose wires are already shortest paths the two coincide).
"""
from __future__ import annotations

from typing import Dict

import torch

from . import engine


class EvaluateEmptyBoard:
    def __init__(self, filled_training_board):
        self.filled_board = engine.as_tensor(filled_training_board)
        self.empty_slot_score = -2
        self.end_score = 3
        self.wire_score = 2
        self.scored_board, self._detours, self._diversity = engine.board_statistics(self.filled_board)
        self.board_statistics = {"count_detours": self._detours, "heatmap_score_diversity": self._diversity}

    def score_from_neighbours(self):
        return self.scored_board

    def count_detours(self, count_current_wire: bool = False):
        if not count_current_wire:
            return self._detours
        return engine.board_statistics(self.filled_board, count_current_wire=True, with_scores=False)[1]


def _unwrap_eval_env(eval_env):
    """(the Connector inside `eval_env`, the reward aggregator of its MultiToSingleWrapper or None)."""
    from .connector import Connector, MultiToSingleWrapper

    env, agg = eval_env, None
    while not isinstance(env, Connector):
        if isinstance(env, MultiToSingleWrapper):
            if agg is not None:
                raise TypeError("eval_env has two MultiToSingleWrappers: the second would aggregate a scalar reward")
            # the return of an aggregated reward is the aggregate of the per-agent returns only for a linear aggregator
            if env._ragg not in (torch.sum, torch.mean):
                raise ValueError(f"MultiToSingleWrapper's reward_aggregator {env._ragg!r}: episode returns are summed per agent in the kernel, "
                                 "so only torch.sum and torch.mean (linear) can be applied to them")
            agg = env._ragg
        env = getattr(env, "_env", None)
        if env is None:
            raise TypeError("eval_env must be a Connector or a wrapper around one")
    return env, agg


class RandomAgentEvaluator:
    """Scores a board generator by what the library's random policy achieves on its boards.

    `eval_env` is a Connector, optionally wrapped (MultiToSingleWrapper, VmapAutoResetWrapper; the latter has no
    effect: an evaluation episode ends at its LAST step).  A MultiToSingleWrapper's reward aggregator is applied to the
    per-agent returns, which equals the return of the aggregated reward for torch.sum and torch.mean; another
    (non-linear) aggregator raises ValueError.  Each episode is reduced to the five numbers the
    reference's benchmarks and evaluators log (BenchmarkData / PickleLogger): episode_return, episode_length,
    num_connections, ratio_connections, total_path_length.  The episodes run in one kernel launch from the reset
    State to each env's first LAST step (engine.connector_episodes_random); nothing is written per step.

    Episode i starts from the eval env's generator called on key i.  jumanji's Evaluator derives its reset keys in
    its own way, so the board of a given key may differ from a jumanji run; the distribution of episodes is the same.
    """

    def __init__(self, eval_env, total_batch_size: int):
        self.eval_env = eval_env
        self.total_batch_size = int(total_batch_size)
        self._env, self._reward_agg = _unwrap_eval_env(eval_env)

    def _reset_state(self, keys):
        """The reset State of each key (no observation): the generator's own kernel, table lookup or __call__."""
        from .connector import _stack_states

        e = self._env
        if e._kind == "dataset":
            return engine.dataset_state(keys, e.grid_size, e.num_agents, engine.as_tensor(e._generator.heads, torch.int32), engine.as_tensor(e._generator.targets, torch.int32))
        if e._kind != "user":
            return engine.generator_state(e._kind, keys, e.grid_size, e.num_agents)
        st = e._generator(keys)
        if st.grid.dim() == 2:  # a generator that only handles single keys
            st = _stack_states([e._generator(k) for k in keys])
        return engine._contig_state(st.map(engine.as_tensor))

    def episode_metrics(self, keys) -> Dict[str, torch.Tensor]:
        """Reset on `keys` (uint32[B,2], or one key of shape (2,) for unbatched results) and run every episode to
        its LAST step.  episode_return is [B,N] per agent, or [B] aggregated over the agents with the reward aggregator
        (torch.sum by default, or torch.mean) when the eval env has a MultiToSingleWrapper."""
        keys, batched = engine.as_keys(keys)
        st = self._reset_state(keys)
        m = engine.connector_episodes_random(st, **self._env._env_args())
        if self._reward_agg is not None:
            m["episode_return"] = self._reward_agg(m["episode_return"], dim=-1)
        return m if batched else {k: v[0] for k, v in m.items()}

    def run_evaluation(self, key) -> Dict[str, torch.Tensor]:
        """Means over `total_batch_size` episodes whose reset keys are split(key, total_batch_size)."""
        m = self.episode_metrics(engine.split(key, self.total_batch_size))
        return {k: v.to(torch.float32).mean(dim=0) for k, v in m.items()}


class PolicyEvaluator:
    """Scores a policy: every episode from its reset to its first LAST step, reduced on the device to the five numbers
    of `RandomAgentEvaluator` (episode_return, episode_length, num_connections, ratio_connections, total_path_length).

    `policy(observation, key)` takes the batched Observation and uint32[B,2] action keys, one per env, and returns
    int32[B,N] actions; whether it samples or acts greedily is its own business (as with jumanji's `Evaluator(...,
    stochastic=...)`).  Rows of envs whose episode has ended carry a stale observation, and the actions returned for
    them are ignored.  Each step is one policy call and one library step (engine.connector_eval_step) that advances
    only the envs still in their first episode and accumulates their metrics in place; the loop ends when none is
    left, at most `time_limit` steps after the reset.  `eval_env` is unwrapped, and a MultiToSingleWrapper's reward
    aggregator applied, as in RandomAgentEvaluator.

    Episode i resets with the unwrapped Connector.reset on key i, so for the same keys it scores the same boards as
    RandomAgentEvaluator.  The action keys are this library's convention, modelled on jumanji's Evaluator but not its
    derivation: chain = split_each(keys)[:, 1], then at every step chain, action_key = split_each(chain).
    """

    def __init__(self, eval_env, policy, total_batch_size: int):
        self.eval_env = eval_env
        self.policy = policy
        self.total_batch_size = int(total_batch_size)
        self._env, self._reward_agg = _unwrap_eval_env(eval_env)

    def episode_metrics(self, keys) -> Dict[str, torch.Tensor]:
        """Reset on `keys` (uint32[B,2], or one key of shape (2,) for unbatched results) and run the policy until
        every episode has had its LAST step.  episode_return is [B,N] per agent, or [B] aggregated as in
        RandomAgentEvaluator.episode_metrics."""
        keys, batched = engine.as_keys(keys)
        B, N = keys.shape[0], self._env.num_agents
        st, ts = self._env.reset(keys)
        dev = st.grid.device
        m = {k: torch.zeros((B, N) if k == "episode_return" else (B,), dtype=torch.float32 if k in ("episode_return", "ratio_connections") else torch.int32, device=dev)
             for k in engine.EPISODE_METRICS}
        live = torch.ones(B, dtype=torch.uint8, device=dev)
        live_count = torch.full((1,), B, dtype=torch.int32, device=dev)
        # the count is read one step late (a step over an all-dead batch changes nothing): at most one host wait per step
        seen = torch.empty(2, dtype=torch.int32, pin_memory=True)
        done = [torch.cuda.Event(), torch.cuda.Event()]
        chain = engine.split_each(keys)[:, 1]
        t = 0
        while True:
            s = engine.split_each(chain)
            chain, action_key = s[:, 0], s[:, 1].contiguous()
            engine.connector_eval_step(st, self.policy(ts.observation, action_key), live, live_count, m, ts, **self._env._env_args())
            seen[t % 2].copy_(live_count[0], non_blocking=True)
            done[t % 2].record()
            if t > 0:
                done[(t - 1) % 2].synchronize()
                if int(seen[(t - 1) % 2]) == 0:
                    break
            t += 1
        if self._reward_agg is not None:
            m["episode_return"] = self._reward_agg(m["episode_return"], dim=-1)
        return m if batched else {k: v[0] for k, v in m.items()}

    def run_evaluation(self, key) -> Dict[str, torch.Tensor]:
        """Means over `total_batch_size` episodes whose reset keys are split(key, total_batch_size)."""
        m = self.episode_metrics(engine.split(key, self.total_batch_size))
        return {k: v.to(torch.float32).mean(dim=0) for k, v in m.items()}
