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
from .types import Observation


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

    live_only=True runs the policy on the live envs only (engine.connector_eval_step_live): each call receives the
    Observation rows of the envs still in their first episode, in ascending env order, and their action keys, so the
    batch dimension L shrinks from call to call, and the policy must return int32[L,N].  The step compacts the live
    envs' observation as it steps them.  For a policy that computes each row from that row alone the metrics are those
    of the default mode, bit for bit.  Reading L costs one host wait per step; the default mode keeps a static batch
    shape (what torch.compile or a CUDA graph of the policy needs) and waits on a count read one step late.  The gain
    is the policy work on finished envs; with a cheap policy, or episodes that nearly all run to time_limit, the wait
    and the list step cost more than that: on a B200 live_only measured 0.67x to 0.96x the default mode's speed for a
    cheap policy and a small MLP (DESIGN.md K7, tools/bench_policy_eval.py --live-only).

    cuda_graph=True runs every evaluation as one CUDA graph launch: the policy call, the key split and the evaluation
    step are captured once per batch size B (torch.cuda.CUDAGraph) and repeated on the device by a WHILE node until no
    env is live (engine.EvalLoop), with no host wait per step and no step past the last episode.  The reset stays
    eager (any generator, user Generators included) and is copied into the graph's static buffers.  The policy must be
    capturable: static shapes, no host sync, no allocation outside torch's caching allocator.  The loop does not advance
    torch's RNG from one iteration to the next: a stochastic policy must draw from the action keys it is given.  For a
    policy that computes each row from that row alone the metrics are the default mode's, bit for bit.  A capture costs
    a policy warm-up and a device synchronisation; the graph is kept until B changes or `close()`.  Not with live_only.
    """

    def __init__(self, eval_env, policy, total_batch_size: int, live_only: bool = False, cuda_graph: bool = False):
        self.eval_env = eval_env
        self.policy = policy
        self.total_batch_size = int(total_batch_size)
        self.live_only = bool(live_only)
        self.cuda_graph = bool(cuda_graph)
        if self.live_only and self.cuda_graph:
            raise ValueError("cuda_graph=True needs a static batch shape, and live_only=True changes it from step to step")
        self._env, self._reward_agg = _unwrap_eval_env(eval_env)
        self._captured = None  # _CapturedEvaluation of the last batch size (cuda_graph=True)

    def episode_metrics(self, keys) -> Dict[str, torch.Tensor]:
        """Reset on `keys` (uint32[B,2], or one key of shape (2,) for unbatched results) and run the policy until
        every episode has had its LAST step.  episode_return is [B,N] per agent, or [B] aggregated as in
        RandomAgentEvaluator.episode_metrics."""
        keys, batched = engine.as_keys(keys)
        B, N = keys.shape[0], self._env.num_agents
        st, ts = self._env.reset(keys)
        dev = st.grid.device
        if self.cuda_graph:
            m = self._run_graph(st, ts, keys)
        else:
            m = {k: torch.zeros((B, N) if k == "episode_return" else (B,), dtype=torch.float32 if k in ("episode_return", "ratio_connections") else torch.int32, device=dev)
                 for k in engine.EPISODE_METRICS}
            chain = engine.split_each(keys)[:, 1]
            if self.live_only:
                self._run_live(st, ts.observation, m, chain)
            else:
                self._run_masked(st, ts, m, chain)
        if self._reward_agg is not None:
            m["episode_return"] = self._reward_agg(m["episode_return"], dim=-1)
        return m if batched else {k: v[0] for k, v in m.items()}

    def _run_masked(self, st, ts, m, chain) -> None:
        """The whole batch to every policy call; a live byte per env selects the envs the step advances."""
        B, dev = st.grid.shape[0], st.grid.device
        live = torch.ones(B, dtype=torch.uint8, device=dev)
        live_count = torch.full((1,), B, dtype=torch.int32, device=dev)
        # the count is read one step late (a step over an all-dead batch changes nothing): at most one host wait per step
        seen = torch.empty(2, dtype=torch.int32, pin_memory=True)
        done = [torch.cuda.Event(), torch.cuda.Event()]
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

    def _run_live(self, st, obs, m, chain) -> None:
        """The live envs only: rows [0, L) of `obs` are the envs order[0][:L]; the step compacts both for the next call."""
        B, dev = st.grid.shape[0], st.grid.device
        order = [torch.arange(B, dtype=torch.int32, device=dev), torch.empty(B, dtype=torch.int32, device=dev)]
        count = torch.empty(1, dtype=torch.int32, device=dev)
        seen = torch.empty(1, dtype=torch.int32, pin_memory=True)
        done = torch.cuda.Event()
        L = B
        while L > 0:
            s = engine.split_each(chain)
            chain, action_key = s[:, 0], s[:, 1]
            idx = order[0][:L]
            view = Observation(grid=obs.grid[:L], action_mask=obs.action_mask[:L], step_count=obs.step_count[:L])
            action = self.policy(view, action_key.contiguous() if L == B else action_key.view(torch.int32)[idx.long()].view(torch.uint32))
            engine.connector_eval_step_live(st, action, order[0], L, order[1], count, m, obs, **self._env._env_args())
            seen.copy_(count, non_blocking=True)
            done.record()
            done.synchronize()  # the next call's batch size
            L = int(seen[0])
            order.reverse()

    def _run_graph(self, st, ts, keys) -> Dict[str, torch.Tensor]:
        """One launch of the captured loop (captured first when the batch size is new); the metrics cloned out."""
        B = keys.shape[0]
        if self._captured is not None and self._captured.B != B:
            self.close()
        first = self._captured is None
        if first:
            self._captured = _CapturedEvaluation(self._env, self.policy, B)
        c = self._captured
        c.load(st, ts, keys)
        if first:
            try:
                c.capture()
            except BaseException:
                self.close()
                raise
        c.loop.launch()
        return {k: v.clone() for k, v in c.m.items()}

    @property
    def loop_steps(self) -> int:
        """Iterations of the device-side loop in the last cuda_graph=True evaluation: the longest episode's length
        (reads the device)."""
        if self._captured is None:
            raise RuntimeError("no cuda_graph=True evaluation has run")
        return int(self._captured.steps.item())

    def close(self) -> None:
        """Frees the captured graph and its static buffers (cuda_graph=True); the next evaluation captures again."""
        if self._captured is not None:
            if self._captured.loop is not None:
                self._captured.loop.close()
            self._captured = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def run_evaluation(self, key) -> Dict[str, torch.Tensor]:
        """Means over `total_batch_size` episodes whose reset keys are split(key, total_batch_size)."""
        m = self.episode_metrics(engine.split(key, self.total_batch_size))
        return {k: v.to(torch.float32).mean(dim=0) for k, v in m.items()}


def _i32(t: torch.Tensor) -> torch.Tensor:
    return t.view(torch.int32) if t.dtype == torch.uint32 else t


class _CapturedEvaluation:
    """PolicyEvaluator(cuda_graph=True) at one batch size: the static buffers and the device-side loop over them.

    Loop body (captured once): chain, action_key = split_each(chain); action = policy(observation, action_key); the
    evaluation step of the live envs; the loop condition (steps += 1, go on while an env is live and steps <= time_limit).
    `graph` owns the memory of the body's intermediate tensors, so it lives as long as the loop."""

    def __init__(self, env, policy, B: int):
        G, N = env.grid_size, env.num_agents
        dev = engine._device()
        self.B, self._env, self._policy = B, env, policy
        self.st, self.ts = engine.alloc_state(B, G, N), engine.alloc_timestep(B, G, N)
        self.live = torch.empty(B, dtype=torch.uint8, device=dev)
        self.live_count = torch.empty(1, dtype=torch.int32, device=dev)
        self.steps = torch.empty(1, dtype=torch.int32, device=dev)
        self.m = {k: torch.empty((B, N) if k == "episode_return" else (B,), dtype=torch.float32 if k in ("episode_return", "ratio_connections") else torch.int32, device=dev)
                  for k in engine.EPISODE_METRICS}
        self.chain = torch.empty((B, 2), dtype=torch.uint32, device=dev)
        self.action_key = torch.empty((B, 2), dtype=torch.uint32, device=dev)
        self.action = torch.empty((B, N), dtype=torch.int32, device=dev)
        self.graph = self.loop = None

    def load(self, st, ts, keys) -> None:
        """The per-evaluation start: the reset State and observation, every env live, the counters and metrics zeroed,
        chain = split_each(keys)[:, 1]."""
        for dst, src in zip((self.st.grid, self.st.step_count, self.st.key, self.st.agents.id, self.st.agents.start, self.st.agents.target, self.st.agents.position),
                            (st.grid, st.step_count, st.key, st.agents.id, st.agents.start, st.agents.target, st.agents.position)):
            _i32(dst).copy_(_i32(src))
        o, so = self.ts.observation, ts.observation
        o.grid.copy_(so.grid)
        o.action_mask.copy_(so.action_mask)
        o.step_count.copy_(so.step_count)
        self.live.fill_(1)
        self.live_count.fill_(self.B)
        self.steps.zero_()
        for v in self.m.values():
            v.zero_()
        _i32(self.chain).copy_(_i32(engine.split_each(keys)[:, 1]))

    def capture(self) -> None:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):  # torch's warm-up before a capture: the policy once, eagerly, on a side stream
            self._policy(self.ts.observation, engine.split_each(self.chain)[:, 1].contiguous())
        torch.cuda.current_stream().wait_stream(side)
        args = self._env._env_args()
        self.loop = engine.EvalLoop()
        self.graph = torch.cuda.CUDAGraph(keep_graph=True)
        with torch.cuda.graph(self.graph):
            s = engine.split_each(self.chain)
            _i32(self.chain).copy_(_i32(s[:, 0]))
            _i32(self.action_key).copy_(_i32(s[:, 1]))
            self.action.copy_(self._policy(self.ts.observation, self.action_key))
            engine.connector_eval_step(self.st, self.action, self.live, self.live_count, self.m, self.ts, **args)
            self.loop.condition(self.live_count, self.steps, args["time_limit"] + 1)
        self.loop.finalize(self.graph)
