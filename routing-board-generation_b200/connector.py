"""Connector environment + wrappers on the CUDA engine.

Mirrors jumanji==0.2.2 (UPSTREAM, requirements.txt:5) as the reference uses it:
  Connector(generator, reward_fn, time_limit)       rl_training/setup_train.py:158
  reset(key) -> (State, TimeStep), step(state, action) -> (State, TimeStep)
  _get_action_mask / _obs_from_grid / _get_extras   demos/board_generator_demo.py:83-96
  MultiToSingleWrapper, VmapAutoResetWrapper        rl_training/setup_train.py:160,166
Batching: the leading axis of keys / state leaves is the vmap axis; a single
key of shape (2,) gives single-env (unbatched) pytrees like the reference.

`Connector(generator=...)` takes what the reference's Connector takes (setup_train.py:107-158):
the kernel-backed generators of this package (Uniform / ParallelRandomWalk / SeedExtension), the
dataset generator `BoardDatasetGeneratorJAX` (a table lookup inside the step kernels), and ANY other
`Generator` subclass / callable `key -> State` with `grid_size` and `num_agents` (reset and auto-reset
then call it on the keys of the finished envs and scatter the result; see `_generic_autoreset`).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from . import engine
from .online_generators import Generator, UniformRandomGenerator
from .types import LAST, Agent, Observation, State, TimeStep

_KERNEL_KINDS = ("uniform", "parallel_random_walk", "seed_extension", "sequential_random_walk")


@dataclass
class DenseRewardFn:
    """jumanji DenseRewardFn: connected_reward when an agent connects, timestep_reward per unconnected step."""

    timestep_reward: float = -0.03
    connected_reward: float = 0.1


def _batch(tree, batched: bool):
    return tree if batched else tree.map(lambda t: t[None])


def _unbatch(tree, batched: bool):
    return tree if batched else tree[0]


class Connector:
    def __init__(self, generator: Optional[Generator] = None, reward_fn: Optional[DenseRewardFn] = None, time_limit: int = 50, viewer=None) -> None:
        self._generator = generator or UniformRandomGenerator(grid_size=10, num_agents=5)
        if not callable(self._generator) or not hasattr(self._generator, "grid_size") or not hasattr(self._generator, "num_agents"):
            raise TypeError("generator must be a Generator: callable `key -> State` with `grid_size` and `num_agents` (uniform_generator.py:26-53)")
        kind = getattr(self._generator, "kind", "") or "user"
        if kind == "dataset" and not (hasattr(self._generator, "heads") and hasattr(self._generator, "targets")):
            kind = "user"
        self._kind = kind if kind in _KERNEL_KINDS or kind == "dataset" else "user"
        self._reward_fn = reward_fn or DenseRewardFn()
        self.time_limit = time_limit
        self.num_agents = self._generator.num_agents
        self.grid_size = self._generator.grid_size
        self._agent_ids = None
        self._viewer = viewer

    def __repr__(self) -> str:
        return f"Connector(grid_size={self.grid_size}, num_agents={self.num_agents}, time_limit={self.time_limit})"

    @property
    def unwrapped(self) -> "Connector":
        return self

    def _transform_timestep(self, ts: TimeStep) -> TimeStep:
        """What the wrappers between this env and an outer VmapAutoResetWrapper do to a TimeStep (nothing here)."""
        return ts

    def _env_args(self) -> dict:
        return dict(time_limit=self.time_limit, timestep_reward=self._reward_fn.timestep_reward, connected_reward=self._reward_fn.connected_reward)

    def _autoreset_args(self) -> dict:
        """engine keyword arguments that select this env's generator for in-kernel auto-reset."""
        if self._kind == "dataset":
            return dict(autoreset_kind="dataset", dataset=(self._generator.heads, self._generator.targets))
        return dict(autoreset_kind=self._kind)

    # -- public API ---------------------------------------------------------
    def reset(self, key) -> Tuple[State, TimeStep]:
        keys, batched = engine.as_keys(key)
        if self._kind == "user":  # any Generator: State from the plugin, the observation half from the kernel
            st = self._generator(keys)
            if st.grid.dim() == 2:  # a generator that only handles single keys
                st = _stack_states([self._generator(k) for k in keys])
            st = engine._contig_state(st.map(engine.as_tensor))
            ts = engine.connector_observe(st)
        elif self._kind == "dataset":
            st, ts = engine.connector_reset("dataset", keys, self.grid_size, self.num_agents, dataset=(self._generator.heads, self._generator.targets))
        else:
            st, ts = engine.connector_reset(self._kind, keys, self.grid_size, self.num_agents)
        return _unbatch(st, batched), _unbatch(ts, batched)

    def step(self, state: State, action) -> Tuple[State, TimeStep]:
        batched = state.grid.dim() == 3
        st = _batch(state, batched)
        new, ts = engine.connector_step(st, action, **self._env_args())
        return _unbatch(new, batched), _unbatch(ts, batched)

    # -- the private trio the reference's own scripts call ------------------
    def _observe(self, state: State) -> TimeStep:
        batched = state.grid.dim() == 3
        return _unbatch(engine.connector_observe(_batch(state, batched)), batched)

    def _get_action_mask_all(self, agents: Agent, grid: torch.Tensor) -> torch.Tensor:
        """vmap(_get_action_mask, (0, None))(agents, grid) -> bool[N,5] (or [B,N,5])."""
        batched = grid.dim() == 3
        st = self._state_from(agents, grid, batched)
        return _unbatch(engine.connector_observe(st), batched).observation.action_mask

    def _get_action_mask(self, agent: Agent, grid: torch.Tensor) -> torch.Tensor:
        """One agent's mask bool[5] on `grid` (jumanji env.py _get_action_mask)."""
        aid = int(agent.id)
        n = self.num_agents
        dev = grid.device
        pad = lambda v, fill: torch.full((n, 2), fill, dtype=torch.int32, device=dev).index_put((torch.tensor(aid, device=dev),), v.to(torch.int32))
        agents = Agent(id=torch.arange(n, dtype=torch.int32, device=dev), start=pad(agent.start, -1), target=pad(agent.target, -2), position=pad(agent.position, 0))
        return self._get_action_mask_all(agents, grid)[aid]

    def _obs_from_grid(self, grid: torch.Tensor) -> torch.Tensor:
        batched = grid.dim() == 3
        n = self.num_agents
        g = grid if batched else grid[None]
        z = torch.zeros((g.shape[0], n, 2), dtype=torch.int32, device=g.device)
        agents = Agent(id=torch.arange(n, dtype=torch.int32, device=g.device).expand(g.shape[0], n).contiguous(), start=z, target=z - 1, position=z)
        ts = engine.connector_observe(self._state_from(agents, g, True))
        return ts.observation.grid if batched else ts.observation.grid[0]

    def _get_extras(self, state: State) -> dict:
        return self._observe(state).extras

    def _state_from(self, agents: Agent, grid: torch.Tensor, batched: bool) -> State:
        g = grid if batched else grid[None]
        ag = agents if batched else agents.map(lambda t: t[None])
        B = g.shape[0]
        return State(key=torch.zeros((B, 2), dtype=torch.uint32, device=g.device), grid=g.to(torch.int32).contiguous(), step_count=torch.zeros((B,), dtype=torch.int32, device=g.device), agents=ag.map(lambda t: t.to(torch.int32).contiguous()))


def _stack_states(states) -> State:
    return State(
        key=torch.stack([s.key for s in states]), grid=torch.stack([s.grid for s in states]), step_count=torch.stack([s.step_count for s in states]),
        agents=Agent(id=torch.stack([s.agents.id for s in states]), start=torch.stack([s.agents.start for s in states]),
                     target=torch.stack([s.agents.target for s in states]), position=torch.stack([s.agents.position for s in states])))


class VmapAutoResetWrapper:
    """jumanji.wrappers.VmapAutoResetWrapper: on LAST, `key, _ = split(state.key)`, reset(key), keep the
    terminal reward / discount / step_type / extras and swap in the reset observation.
    The stepping, the compaction of finished envs and their regeneration run inside the library; the
    wrappers between this one and the Connector (MultiToSingleWrapper, setup_train.py:160-166) are applied to
    the resulting TimeStep through their `_transform_timestep` hooks."""

    def __init__(self, env):
        self._env = env

    @property
    def unwrapped(self) -> Connector:
        return self._env.unwrapped

    def __getattr__(self, name):
        return getattr(self._env, name)

    def _transform_timestep(self, ts: TimeStep) -> TimeStep:
        return self._env._transform_timestep(ts)

    def reset(self, key):
        keys, _ = engine.as_keys(key)
        return self._env.reset(keys)

    def step(self, state: State, action, inplace: bool = False):
        e = self._env.unwrapped
        if e._kind == "user":
            st, ts = _generic_autoreset_step(e, state, action, inplace)
        else:
            st, ts = engine.connector_step(state, action, **e._env_args(), **e._autoreset_args(), inplace=inplace, owner=e)
        return st, self._transform_timestep(ts)

    def step_random(self, state: State, inplace: bool = False):
        """Random-policy step in the same launch (the agent=random benchmark loop)."""
        e = self._env.unwrapped
        if e._kind == "user":
            act = engine.random_actions(engine._contig_state(state))
            st, ts = _generic_autoreset_step(e, state, act, inplace)
        else:
            st, ts, act = engine.connector_step(state, None, **e._env_args(), **e._autoreset_args(), inplace=inplace, random_policy=True, owner=e)
        return st, self._transform_timestep(ts), act

    def rollout_random(self, state: State, n_steps: int, out: Optional[TimeStep] = None):
        """`n_steps` random-policy steps with auto-reset in one library call: generation, reset and
        stepping fused into one launch sequence.  Updates `state` in place; returns
        (state, TimeStep stacked [n_steps, B, ...], actions[n_steps, B, N])."""
        e = self._env.unwrapped
        if e._kind == "user":
            raise NotImplementedError("rollout_random fuses generation into the kernel: it needs one of this package's generators (use step_random with a user Generator)")
        st, ts, act = engine.connector_rollout_random(state, n_steps, **e._env_args(), **e._autoreset_args(), out=out, owner=e)
        return st, self._transform_timestep(ts), act


def _generic_autoreset_step(env: Connector, state: State, action, inplace: bool):
    """VmapAutoResetWrapper.step for ANY Generator: plain Connector.step in the kernel, then for the envs whose
    step_type is LAST: `key, _ = split(state.key)`, `generator(key)`, the observation half of reset from the
    kernel, scattered over the batch (jumanji wrappers.py `_auto_reset` / `_maybe_reset`)."""
    if torch.cuda.is_current_stream_capturing():
        raise RuntimeError("auto-reset with a user Generator selects the finished envs on the host (a data-dependent index), "
                           "which a CUDA graph cannot capture: step it eagerly, or use one of this package's generators")
    st, ts = engine.connector_step(state, action, **env._env_args(), inplace=inplace)
    idx = torch.nonzero(ts.step_type == LAST).flatten()
    if idx.numel() == 0:
        return st, ts
    i32 = lambda t: t.view(torch.int32) if t.dtype == torch.uint32 else t  # torch's uint32 indexing support is thin
    keys = engine.split_each(i32(st.key)[idx].contiguous(), 2)[:, 0].contiguous()
    fresh = env._generator(keys)
    if fresh.grid.dim() == 2:
        fresh = _stack_states([env._generator(k) for k in keys])
    fresh = engine._contig_state(fresh.map(engine.as_tensor))
    fts = engine.connector_observe(fresh)
    a, fa = st.agents, fresh.agents
    i32(st.key)[idx] = i32(fresh.key)
    st.grid[idx] = fresh.grid
    st.step_count[idx] = fresh.step_count
    a.id[idx], a.start[idx], a.target[idx], a.position[idx] = fa.id, fa.start, fa.target, fa.position
    o, fo = ts.observation, fts.observation
    o.grid[idx], o.action_mask[idx], o.step_count[idx] = fo.grid, fo.action_mask, fo.step_count
    return st, ts


class MultiToSingleWrapper:
    """jumanji.wrappers.MultiToSingleWrapper: reward -> sum over agents, discount -> max over agents."""

    def __init__(self, env, reward_aggregator=torch.sum, discount_aggregator=torch.amax):
        self._env = env
        self._ragg = reward_aggregator
        self._dagg = discount_aggregator

    @property
    def unwrapped(self):
        return self._env.unwrapped

    def __getattr__(self, name):
        return getattr(self._env, name)

    def _aggregate(self, ts: TimeStep) -> TimeStep:
        return ts.replace(reward=self._ragg(ts.reward, dim=-1), discount=self._dagg(ts.discount, dim=-1))

    def _transform_timestep(self, ts: TimeStep) -> TimeStep:
        return self._aggregate(self._env._transform_timestep(ts))

    def reset(self, key):
        st, ts = self._env.reset(key)
        return st, self._aggregate(ts)

    def step(self, state, action, **kw):
        st, ts = self._env.step(state, action, **kw)
        return st, self._aggregate(ts)


def make_random_policy_connector():
    """Uniform over the legal actions (NOOP included), as jumanji's make_random_policy_connector
    (rl_training/setup_train.py:246) in distribution; see include/rbg_b200.h rbg_random_actions."""

    def policy(state: State) -> torch.Tensor:
        batched = state.grid.dim() == 3
        act = engine.random_actions(_batch(state, batched))
        return act if batched else act[0]

    return policy
