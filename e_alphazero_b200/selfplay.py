"""Host-side mirror of the reference's selfplay step (selfplay.py:86-143) and reanalyze search
(reanalyze.py:52-131) on top of the fused CUDA path.  One `SelfplayRunner.step()` is the unit the
benchmark times: root forward -> E-MCTS search -> auto-reset env step."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Any

from . import _abi, ops
from ._lib import require_cuda


@dataclass
class SelfplayOutput:  # selfplay.py:17-23
    state: Any
    root_value: Any
    root_epistemic_std: Any
    value_prediction: Any
    ube_prediction: Any
    q_values_epistemic_variance: Any
    action: Any = None


class SelfplayRunner:
    """Pre-allocates the search plan; `step(states, gumbel=None)` advances a batch of envs by one move.

    ALIASING: the returned SelfplayOutput fields (and `states`) are views of buffers this runner reuses on every step -- the
    plan's output tensors, the CUDA graph's static buffers, the in-place state dict.  The reference's lax.scan stacks per-step
    outputs (selfplay.py:148); a caller collecting outputs over several steps must clone what it keeps, or pass
    `clone_outputs=True`, or use `trajectory()` (one packed int32 [B,4] record per step, written into a caller-owned [T,B,4] buffer).

    device_noise=True draws the root Gumbel noise inside the search (counter-based stream keyed by `seed`, the number of searches run
    and the tree index) instead of five elementwise torch kernels per step; parity tests pass `gumbel=` explicitly.

    The optional parts of the reference's step: uniform_prior=True searches from a uniform root prior instead of the network's root
    logits (selfplay.py:92-98); action_sampling="visit_counts" / "improved_policy" plays an action drawn from the search's visit
    counts / action_weights at `temperature` instead of its own action (selfplay.py:125-134).  Both run inside the search kernels.
    The noise of that draw follows the rules of the root noise: `sample_gumbel=` if given, else drawn from the runner's generator
    (inside the CUDA graph when captured), or by the search itself with device_noise=True.  `SelfplayOutput.action` and
    `trajectory()` carry the played action."""

    ACTION_SAMPLING = {"search": _abi.ACTION_SEARCH, "visit_counts": _abi.ACTION_VISITS, "improved_policy": _abi.ACTION_IMPROVED}

    def __init__(self, env_spec: ops.EnvSpec, net: ops.FcParams, batch: int, num_simulations: int, discount: float,
                 exploration_beta: float = 0.0, directed_exploration: bool = False, rescale_values: bool = True,
                 mlp_mode: int = _abi.MLP_EXACT, tasks=(1,), device="cuda", seed: int = 0, use_graph: bool = False, fused_root: bool = False,
                 streams: int = 1, device_noise: bool = False, clone_outputs: bool = False, uniform_prior: bool = False,
                 action_sampling: str = "search", temperature: float = 1.0):
        torch = require_cuda()
        if action_sampling not in self.ACTION_SAMPLING:
            raise ValueError(f"action_sampling must be one of {sorted(self.ACTION_SAMPLING)}, got {action_sampling!r}")
        self.env, self.net, self.B, self.device = env_spec, net, batch, device
        self.directed = directed_exploration
        self.cfg = _abi.default_search_config(batch=batch, num_simulations=num_simulations, discount=discount,
                                              exploration=int(directed_exploration), rescale_values=int(rescale_values), mlp_mode=mlp_mode)
        self.cfg.noise_seed = int(seed) & 0xFFFFFFFF
        self.cfg.root_prior = _abi.ROOT_PRIOR_UNIFORM if uniform_prior else _abi.ROOT_PRIOR_GIVEN
        self.cfg.action_sampling = self.ACTION_SAMPLING[action_sampling]
        self.cfg.temperature = float(temperature)
        self.sampling = self.cfg.action_sampling != _abi.ACTION_SEARCH
        self.device_noise, self.clone_outputs = bool(device_noise), bool(clone_outputs)
        if streams > 1:  # EAZ_FLAG_STREAMS: sub-batches searched concurrently (tree kernel of one overlaps the network kernel of another)
            self.cfg.flags |= _abi.flag_streams(streams)
        self.plan = ops.SearchPlan(self.cfg, env_spec, net, want_tree=False, device=device)
        beta = exploration_beta if directed_exploration else 0.0  # selfplay.py:92, config.py:172
        self.beta = (beta * torch.linspace(0, 1, batch, device=device)).contiguous()  # selfplay.py:105
        self.gen = torch.Generator(device=device).manual_seed(seed)
        self.tasks = torch.tensor(list(tasks), dtype=torch.int32, device=device)
        self.A = env_spec.num_actions
        # launches per step: compact+mlp (root forward), search, env step
        self.launches_per_step = 2 + self.plan.num_launches + 1  # (fused root: pack+mlp are replaced by one network launch inside the search)
        self.launches_per_step_reuse = 2 + self.plan.num_launches_reuse + 1  # steps that reuse the parameter-derived tables
        # CUDA graph of one whole step (noise draw -> root forward -> search -> env step): the launch sequence is fixed and
        # nothing synchronises or allocates, so it is captured once and replayed.  Two variants exist: the first step
        # after a parameter update rebuilds the parameter-derived tables (weight images, novelty table, seq-halving
        # table), the others reuse them (EAZ_FLAG_REUSE_PREPARED) -- the model is constant within one selfplay() scan.
        self.use_graph = use_graph
        self.fused_root = fused_root  # let the search evaluate the root network itself (same kernels, one launch less path)
        self._graphs = {}
        self._static = None
        self._stale = True

    def params_updated(self):
        """Call after the network parameters / hash set changed (learner update, broadcast)."""
        self._stale = True

    def draw_gumbel(self):
        torch = require_cuda()
        u = torch.rand((self.B, self.A), device=self.device, generator=self.gen).clamp_(1e-20, 1.0 - 1e-7)
        return (-(-u.log()).log()).contiguous()

    def _draw_tasks(self):
        torch = require_cuda()
        idx = torch.randint(0, self.tasks.numel(), (self.B,), device=self.device, generator=self.gen)
        return self.tasks[idx].contiguous()

    def step(self, states: dict, gumbel=None, task_ids=None, sample_gumbel=None):
        """states: device state dict (updated in place); sample_gumbel: the noise of the action draw (action_sampling only).
        Returns (states, SelfplayOutput)."""
        if self.use_graph:
            return self._step_graph(states, gumbel, task_ids, sample_gumbel)
        reuse = not self._stale
        self._stale = False
        return self._step_eager(states, gumbel, task_ids, reuse_prepared=reuse, sample_gumbel=sample_gumbel)

    def _step_graph(self, states, gumbel, task_ids, sample_gumbel=None):
        torch = require_cuda()
        subleq = self.env.kind == _abi.ENV_SUBLEQ
        if self._static is None:
            # the graph's state buffers live in ONE arena (ops.alloc_arena): a host caller uploads / downloads all fields with one copy
            self.state_specs = [(k, tuple(v.shape), v.dtype) for k, v in states.items()]
            self.static_flat, st = ops.alloc_arena(self.state_specs, self.device)
            for k, v in states.items():
                st[k].copy_(v)
            sg = torch.zeros((self.B, self.A), dtype=torch.float32, device=self.device)
            ss = torch.zeros((self.B, self.A), dtype=torch.float32, device=self.device)
            stt = torch.ones(self.B, dtype=torch.int32, device=self.device) if subleq else None
            self._step_eager({k: v.clone() for k, v in st.items()}, self.draw_gumbel(), self._draw_tasks() if subleq else None,
                             reuse_prepared=False, sample_gumbel=ss)  # warm-up: one-time attribute setup / allocations
            torch.cuda.synchronize()
            self._static = (st, sg, stt, ss)
        st, sg, stt, ss = self._static
        draw = gumbel is None and sample_gumbel is None and (task_ids is None or not subleq)  # noise drawn inside the graph unless
        in_search = draw and self.device_noise                                                # supplied ... by the search itself
        host_sample = self.sampling and (sample_gumbel is not None or not self.device_noise)  # the action draw's noise in `ss`
        key = (not self._stale, draw, in_search, host_sample)
        if key not in self._graphs:
            g = torch.cuda.CUDAGraph()
            g.register_generator_state(self.gen)
            with torch.cuda.graph(g):
                if draw:
                    if not in_search:
                        sg.copy_(self.draw_gumbel())
                    if host_sample:
                        ss.copy_(self.draw_gumbel())
                    if subleq:
                        stt.copy_(self._draw_tasks())
                _, out = self._step_eager(st, None if in_search else sg, stt, reuse_prepared=key[0], sample_gumbel=ss if host_sample else None)
            self._graphs[key] = (g, out)
        g, out = self._graphs[key]
        for k in st:
            if states[k].data_ptr() != st[k].data_ptr():
                st[k].copy_(states[k])
        if not draw:
            sg.copy_(gumbel if gumbel is not None else self.draw_gumbel())
            if host_sample:
                ss.copy_(sample_gumbel if sample_gumbel is not None else self.draw_gumbel())
            if subleq:
                stt.copy_(task_ids if task_ids is not None else self._draw_tasks())
        g.replay()
        self._stale = False
        for k in st:
            if states[k].data_ptr() != st[k].data_ptr():
                states[k].copy_(st[k])
        return states, out

    def static_states(self):
        """The graph's own state buffers (step them in place to avoid the copies in/out)."""
        return self._static[0] if self._static else None

    def host_arenas(self):
        """Pinned host mirrors of the two device arenas of a graph runner -- (states_flat, states_views, out_flat, out_views) with the
        device layouts, so that a host caller moves a whole step's inputs / results with ONE copy each way per arena:
        `runner.static_flat.copy_(states_flat, non_blocking=True)` ... step ... `out_flat.copy_(runner.plan.out_flat, non_blocking=True)`."""
        if self._static is None:
            raise ops.EazError("host_arenas(): run one graph step first (the state arena is created by it)")
        sf, sv = ops.alloc_arena(self.state_specs, "cpu", pinned=True)
        of, ov = ops.alloc_arena(self.plan.out_specs, "cpu", pinned=True)
        return sf, sv, of, ov

    def _step_eager(self, states: dict, gumbel=None, task_ids=None, reuse_prepared=None, sample_gumbel=None):
        torch = require_cuda()
        if gumbel is None and not self.device_noise:
            gumbel = self.draw_gumbel()
        if sample_gumbel is None and self.sampling and not self.device_noise:
            sample_gumbel = self.draw_gumbel()
        if self.fused_root:  # selfplay.py:89 inside the search call (policy head = the recurrent_fn's: main.py:262)
            root = dict(beta=self.beta, embedding=states, gumbel=gumbel)
        else:
            ev = ops.mlp_forward_states(self.net, self.env, states)  # selfplay.py:89
            logits = ev["explore_logits"] if self.directed else ev["exploit_logits"]  # :93-95
            root = dict(prior_logits=logits, value=ev["value"], value_epistemic_variance=ev["ube"], beta=self.beta, embedding=states,
                        gumbel=gumbel)
        if self.sampling:
            root["sample_gumbel"] = sample_gumbel
        out = self.plan.run(root, reuse_prepared=reuse_prepared)  # :107-117 (invalid_actions = ~legal_action_mask = none)
        if self.fused_root:
            ev = dict(value=out["root_value"], ube=out["root_ube"])
        if task_ids is None and self.env.kind == _abi.ENV_SUBLEQ:
            task_ids = self._draw_tasks()
        ops.env_step_(self.env, states, out["action"], auto_reset=True, task_ids=task_ids)  # :135
        res = SelfplayOutput(state=states, root_value=out["value"], root_epistemic_std=out["value_epistemic_std"],
                             value_prediction=ev["value"], ube_prediction=ev["ube"],
                             q_values_epistemic_variance=out["qvalues_epistemic_variance"], action=out["action"])
        if self.clone_outputs and not torch.cuda.is_current_stream_capturing():
            res = SelfplayOutput(**{k: (v.clone() if torch.is_tensor(v) else v) for k, v in vars(res).items() if k != "state"}, state=states)
        return states, res

    def trajectory(self, states: dict, out: SelfplayOutput, dst):
        """Pack this step's replay record (ops.trajectory_pack: action, reward bits, flags, compact-state word) into `dst`
        (int32 [B,4], e.g. one row of a [T,B,4] scan buffer): one small kernel, nothing aliased."""
        return ops.trajectory_pack(self.env, states, out.action, dst)
