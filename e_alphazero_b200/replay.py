"""Compact replay ring (SURVEY.md 8f-3): the device-side stand-in for the reference's flashbax prioritised flat buffer
(main.py:217-225 `make_prioritised_flat_buffer(..., add_sequences=True, add_batch_size=selfplay_batch_size)`,
main.py:383-385 `buffer_fn.add`, main.py:413 `buffer_fn.sample`).

The reference stores a full `pgx.State` per env per step -- for DeepSea-30 that is 900 observation bytes + bookkeeping,
for DeepSea-100 10 KB.  Here a step is the COMPACT state (`eaz_env_compact`: 4 bytes DeepSea, 40 + ws bytes Subleq) plus
the rewards leaf; `sample()` draws (t, env) pairs and decodes `ExperiencePair(first=state_t, second=state_t+1)` on the
device with `eaz_env_uncompact` (observations are materialised only on request: the fused search and the network kernels
read compact states directly).  `CompactReplayRing.sample()` draws uniformly over the stored consecutive pairs.  The
reference's buffer is prioritised: it is built with `priority_exponent` (main.py:217-225, config.py:54), the training loop
reads `batch.indices` (main.py:414) and writes the learner's scores back with `set_priorities` (main.py:454).
`PrioritisedReplayRing` reproduces that data distribution with a device sum tree (csrc/replay.cu).  Multi-GPU: every rank
owns the ring of its env shard, priorities included."""
from __future__ import annotations

from dataclasses import dataclass

from . import ops
from ._lib import EazError, require_cuda
from .reanalyze import ExperiencePair


class CompactReplayRing:
    def __init__(self, env_spec: ops.EnvSpec, max_length_time_axis: int, add_batch_size: int, device="cuda", seed: int = 0):
        torch = require_cuda()
        self.env, self.T, self.B, self.device = env_spec, int(max_length_time_axis), int(add_batch_size), device
        if self.T < 2:
            raise EazError("the ring needs at least two time steps to form (state, next state) pairs")
        self.S = env_spec.compact_bytes
        self.states = torch.zeros((self.T, self.B, self.S), dtype=torch.uint8, device=device)
        self.rewards = torch.zeros((self.T, self.B), dtype=torch.float32, device=device)
        self.cursor = 0   # next time slot to write
        self.length = 0   # number of valid time slots
        self.gen = torch.Generator(device=device).manual_seed(seed)

    @property
    def bytes_per_step(self) -> int:
        return self.B * (self.S + 4)

    def add(self, state: dict) -> None:
        """Append one time step for all `add_batch_size` envs (call once per self-play step, in order)."""
        self.states[self.cursor].copy_(ops.env_compact(self.env, state))
        self.rewards[self.cursor].copy_(state["rewards"].reshape(self.B))
        self.cursor = (self.cursor + 1) % self.T
        self.length = min(self.length + 1, self.T)

    def add_sequence(self, x) -> None:
        """Append T' time steps at once, in time order: the cursor and length advance by T' (only the last T rows survive when
        T' > T), exactly as T' add() calls would.  `x` is a scan's SelfplayOutput.state, dict(compact=[T',B,S] uint8, rewards=[T',B])
        (SelfplayRunner.scan), or state leaves with a leading time axis [T',B,...], as a dict or the pgx State of selfplay(); those
        are compacted in one eaz_env_compact call over the T' * B rows."""
        compact, rewards = self._sequence(x)
        n = compact.shape[0]
        keep = min(n, self.T)
        s0 = (self.cursor + n - keep) % self.T
        k1 = min(keep, self.T - s0)  # rows before the ring wraps
        self.states[s0:s0 + k1].copy_(compact[n - keep:n - keep + k1])
        self.rewards[s0:s0 + k1].copy_(rewards[n - keep:n - keep + k1])
        self.states[:keep - k1].copy_(compact[n - keep + k1:])
        self.rewards[:keep - k1].copy_(rewards[n - keep + k1:])
        self._advance(n)

    def _advance(self, n: int) -> None:
        self.cursor = (self.cursor + n) % self.T
        self.length = min(self.length + n, self.T)

    def _sequence(self, x):
        """-> (compact [T',B,S] uint8, rewards [T',B] float32), contiguous device tensors"""
        torch = require_cuda()
        if isinstance(x, dict) and "compact" in x:
            compact, rewards = x["compact"], x["rewards"]
        else:
            leaves = x.leaves if hasattr(x, "leaves") else x  # pgx State of e_alphazero_b200.pgx, or a dict of its leaves
            n, B = leaves["step_count"].shape[:2]
            flat = {k: leaves[k].reshape((n * B,) + tuple(leaves[k].shape[2:])).contiguous() for k in ops.state_fields(self.env)}
            compact = ops.env_compact(self.env, flat).reshape(n, B, self.S) if n > 0 else torch.empty((0, B, self.S), dtype=torch.uint8,
                                                                                                       device=self.device)
            rewards = leaves["rewards"].reshape(n, B)
        if compact.dim() != 3 or tuple(compact.shape[1:]) != (self.B, self.S) or tuple(rewards.shape[:2]) != tuple(compact.shape[:2]):
            raise EazError(f"add_sequence: expected [T', {self.B}, ...] time steps of the ring's {self.B} envs (compact records "
                           f"[T', {self.B}, {self.S}], rewards [T', {self.B}])")
        return compact.contiguous(), rewards.reshape(compact.shape[:2]).to(torch.float32).contiguous()

    def can_sample(self, min_length: int = 2) -> bool:
        return self.length >= max(2, min_length)

    def sample(self, batch_size: int, with_obs: bool = False) -> ExperiencePair:
        """Uniformly sampled consecutive pairs (state_t, state_t+1) of the same env; t+1 never crosses the write cursor."""
        torch = require_cuda()
        if not self.can_sample():
            raise EazError("not enough steps in the ring to sample a pair")
        oldest = (self.cursor - self.length) % self.T
        k = torch.randint(0, self.length - 1, (batch_size,), device=self.device, generator=self.gen)  # pair index in logical time
        b = torch.randint(0, self.B, (batch_size,), device=self.device, generator=self.gen)
        t0, t1 = (oldest + k) % self.T, (oldest + k + 1) % self.T
        first = ops.env_uncompact(self.env, self.states[t0, b], self.rewards[t0, b], with_obs=with_obs)
        second = ops.env_uncompact(self.env, self.states[t1, b], self.rewards[t1, b], with_obs=with_obs)
        return ExperiencePair(first=first, second=second)


@dataclass
class PrioritisedSample:
    """flashbax's PrioritisedTrajectoryBufferSample: `experience` (ExperiencePair of decoded states), `indices` int32 [K] (opaque
    handles for set_priorities) and `probabilities` float32 [K] (weight / total weight).  `compact` holds the gathered compact
    records and rewards of both slots the decode read."""

    experience: ExperiencePair
    indices: object
    probabilities: object
    compact: dict


class PrioritisedReplayRing(CompactReplayRing):
    """flashbax `make_prioritised_flat_buffer(..., priority_exponent)` (main.py:217-225) on the compact ring: the same storage and
    add(), plus a device sum tree over the pairs (item t * B + b = slots (t, t+1) of env b).  New pairs enter with the largest
    priority seen so far (flashbax's rule); sample() draws in proportion to priority ** priority_exponent by stratified sampling;
    set_priorities() writes the learner's scores back (main.py:454).

    sample(out=...) and set_priorities() with int32 / float32 device tensors neither allocate nor synchronise, so a reanalyze
    step (sample, decode, ReanalyzeRunner, set_priorities) can be captured in one CUDA graph.  add() writes the slot its host
    cursor names: a captured add() rewrites that same slot (and refreshes the priority of the pairs ending there) on every replay."""

    def __init__(self, env_spec: ops.EnvSpec, max_length_time_axis: int, add_batch_size: int, priority_exponent: float = 0.6, device="cuda",
                 seed: int = 0):
        super().__init__(env_spec, max_length_time_axis, add_batch_size, device=device, seed=seed)
        torch = require_cuda()
        self.priority_exponent = float(priority_exponent)
        self.tree = torch.zeros(ops.priority_tree_bytes(self.T, self.B), dtype=torch.uint8, device=device)
        ops.priority_init(self.tree, self.T, self.B, self.priority_exponent, int(seed) & 0xFFFFFFFF)

    def add(self, state: dict) -> None:
        slot = self.cursor
        super().add(state)
        ops.priority_add_step(self.tree, self.T, self.B, slot)

    def add_sequence(self, x) -> None:
        """CompactReplayRing.add_sequence with the tree: one eaz_replay_add_sequence call (the rows, the leaves they touch and the
        header), bit for bit what T' add() calls leave."""
        compact, rewards = self._sequence(x)
        ops.replay_add_sequence(self.env, compact, rewards, self.states, self.rewards, self.tree)
        self._advance(compact.shape[0])

    def alloc_sample(self, batch_size: int, with_obs: bool = False) -> PrioritisedSample:
        """Output buffers for sample(batch_size, with_obs, out=...)."""
        torch = require_cuda()
        K, dev = int(batch_size), self.device
        compact = dict(first=torch.empty((K, self.S), dtype=torch.uint8, device=dev), second=torch.empty((K, self.S), dtype=torch.uint8, device=dev),
                       first_rewards=torch.empty(K, dtype=torch.float32, device=dev), second_rewards=torch.empty(K, dtype=torch.float32, device=dev))
        exp = ExperiencePair(first=ops.alloc_state(self.env, K, with_obs, dev), second=ops.alloc_state(self.env, K, with_obs, dev))
        return PrioritisedSample(exp, torch.empty(K, dtype=torch.int32, device=dev), torch.empty(K, dtype=torch.float32, device=dev), compact)

    def sample(self, batch_size: int, with_obs: bool = False, out: PrioritisedSample | None = None) -> PrioritisedSample:
        """K = batch_size pairs drawn in proportion to their weights; `out` (alloc_sample) is overwritten in place."""
        if not self.can_sample():
            raise EazError("not enough steps in the ring to sample a pair")
        if out is None:
            out = self.alloc_sample(batch_size, with_obs)
        elif out.indices.numel() != batch_size or ("observation" in out.experience.first) != with_obs:
            raise EazError("sample(out=...): buffers were allocated for another batch size / with_obs")
        c = out.compact
        ops.priority_sample(self.tree, self.T, self.B, out.indices, out.probabilities, self.states, self.rewards, c["first"], c["first_rewards"],
                            c["second"], c["second_rewards"])
        ops.env_uncompact(self.env, c["first"], c["first_rewards"], with_obs, out=out.experience.first)
        ops.env_uncompact(self.env, c["second"], c["second_rewards"], with_obs, out=out.experience.second)
        return out

    def set_priorities(self, indices, priorities) -> None:
        """flashbax set_priorities: item indices[k] gets priorities[k] (the last of duplicated indices wins; a stale index, whose
        pair has since been overwritten, keeps weight 0).  Host arrays are range-checked here; device tensors are checked on
        the device (an out-of-range index is skipped and reported by numeric_status())."""
        torch = require_cuda()
        if not (torch.is_tensor(indices) and indices.is_cuda):
            import numpy as np

            idx = np.asarray(indices.cpu() if torch.is_tensor(indices) else indices).reshape(-1)
            if idx.size and (idx.min() < 0 or idx.max() >= self.T * self.B):
                raise EazError(f"set_priorities: index outside [0, {self.T * self.B})")
        indices = torch.as_tensor(indices, device=self.device).to(torch.int32).reshape(-1).contiguous()
        priorities = torch.as_tensor(priorities, device=self.device).to(torch.float32).reshape(-1).contiguous()
        ops.priority_set(self.tree, self.T, self.B, indices, priorities)

    def numeric_status(self) -> int:
        """Synchronises; raises EazError if a priority was negative / non-finite (stored as 0), an index was out of range, a sample
        met an empty tree or add() ran out of order since the ring was built.  Returns 0."""
        return ops.priority_status(self.tree)
