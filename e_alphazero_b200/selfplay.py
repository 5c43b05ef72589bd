"""Host-side mirror of the reference's selfplay step (selfplay.py:86-143) and reanalyze search
(reanalyze.py:52-131) on top of the fused CUDA path.  One `SelfplayRunner.step()` is the unit the
benchmark times: root forward -> E-MCTS search -> auto-reset env step.  `SelfplayRunner.scan()` and the
drop-in `selfplay()` run the reference's whole scan of such steps (selfplay.py:78-149) as one device
program (csrc/selfplay.cu: eaz_selfplay)."""
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
    trajectory: Any = None  # scan(): the eaz_trajectory_pack records [T,B,4] of the states after every step


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
        self._scan_plan = None   # eaz_selfplay's workspace (its own parameter-derived tables: staleness tracked apart from step()'s)
        self._scan_stale = True
        self._scan_out = None    # (T, stacked output buffers)

    def params_updated(self):
        """Call after the network parameters / hash set changed (learner update, broadcast)."""
        self._stale = True
        self._scan_stale = True

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

    def scan(self, states: dict, T: int, gumbel=None, sample_gumbel=None, task_ids=None):
        """The reference's selfplay() scan (selfplay.py:78-149): T steps of step() as one device program (a CUDA graph whose loop the
        device stops after T steps; the host launches it once).  states: device state dict, stepped in place to the final carry.
        gumbel / sample_gumbel [T,B,A] and task_ids [T,B] hold row t for step t; without them the noise follows the runner's rules
        (drawn from its generator, [T,B,A] in one call, or inside the search with device_noise=True) and the Subleq reset tasks are
        drawn from the generator in one [T,B] call.
        Returns (states, SelfplayOutput) whose fields are [T,B] stacks in buffers this runner owns (the next scan of the same T
        overwrites them): row t equals step t's output of T step() calls.  `state` is the states after every step in the replay ring's
        wire format, dict(compact=[T,B,S] uint8, rewards=[T,B]) (ops.env_uncompact decodes a row); `trajectory` holds the
        trajectory() records [T,B,4]."""
        torch = require_cuda()
        T = int(T)
        if T < 0:
            raise ValueError(f"scan: T must be >= 0, got {T}")
        if self._scan_plan is None:
            self._scan_plan = ops.SelfplayPlan(self.cfg, self.env, self.net, device=self.device)
        if self._scan_out is None or self._scan_out[0] != T:
            self._scan_out = (T, ops.alloc_selfplay_outputs(self.env, T, self.B, device=self.device))
        out = self._scan_out[1]
        noise = lambda: (-(-torch.rand((T, self.B, self.A), device=self.device, generator=self.gen).clamp_(1e-20, 1.0 - 1e-7).log()).log())
        if gumbel is None and not self.device_noise:
            gumbel = noise()
        if sample_gumbel is None and self.sampling and not self.device_noise:
            sample_gumbel = noise()
        if task_ids is None and self.env.kind == _abi.ENV_SUBLEQ:
            task_ids = self.tasks[torch.randint(0, self.tasks.numel(), (T, self.B), device=self.device, generator=self.gen)]
        as_f32 = lambda t: None if t is None else t.to(dtype=torch.float32).contiguous()
        task_ids = None if task_ids is None else task_ids.to(dtype=torch.int32).contiguous()
        self._scan_plan.run(self.beta, states, T, out, gumbel=as_f32(gumbel), sample_gumbel=as_f32(sample_gumbel) if self.sampling else None,
                            task_ids=task_ids, reuse_prepared=not self._scan_stale)
        if T > 0:
            self._scan_stale = False
        res = SelfplayOutput(state=dict(compact=out["states"], rewards=out["rewards"]), root_value=out["root_value"],
                             root_epistemic_std=out["root_epistemic_std"], value_prediction=out["value_prediction"],
                             ube_prediction=out["ube_prediction"], q_values_epistemic_variance=out["q_values_epistemic_variance"],
                             action=out["action"], trajectory=out["trajectory"])
        return states, res

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


_runners: dict = {}


def _leaves(state):
    return state.leaves if hasattr(state, "leaves") else state


def selfplay(model, config, context, last_states, rng_key=None):
    """Drop-in for selfplay.selfplay (selfplay.py:78-149): config.selfplay_steps steps of the self-play step from `last_states` (a
    pgx State of e_alphazero_b200.pgx, not modified) as one device program.  `config` needs the attributes the reference reads:
    selfplay_steps, selfplay_simulations_per_step, discount, exploration_beta, directed_exploration, rescale_q_values_in_search
    (+ optional mlp_mode); `context.env` is an e_alphazero_b200.pgx env.  rng_key: an emctx.PreDrawnGumbel carrying the root noise
    [T,B,A], an int seed of the runner's generator, or None (the generator continues).

    The reference's return statement is not in the sources this mirrors; the order here follows lax.scan's (carry, ys):
    (final states, SelfplayOutput) with every field stacked over the T steps and `state` decoded to pgx State leaves [T,B,...] (the
    states after each step), plus `trajectory` [T,B,4]."""
    from .context import as_fc_params
    from .emctx import PreDrawnGumbel
    from .pgx import State, Subleq

    require_cuda()
    env = context.env
    net = as_fc_params(model, env=env)
    states = {k: v.clone() for k, v in _leaves(last_states).items() if k != "observation"}
    B, T = states["terminated"].shape[0], int(config.selfplay_steps)
    key = (id(env), id(net), B, int(config.selfplay_simulations_per_step), float(config.discount), float(config.exploration_beta),
           bool(config.directed_exploration), bool(config.rescale_q_values_in_search), int(getattr(config, "mlp_mode", _abi.MLP_EXACT)))
    hit = _runners.get(key)  # (env, net, runner): the strong references keep the id()s in the key unique
    if hit is None or hit[0] is not env or hit[1] is not net:
        while len(_runners) >= 8:
            _runners.pop(next(iter(_runners)))
        hit = _runners[key] = (env, net, SelfplayRunner(env.spec, net, B, int(config.selfplay_simulations_per_step), float(config.discount),
                                                        exploration_beta=float(config.exploration_beta),
                                                        directed_exploration=bool(config.directed_exploration),
                                                        rescale_values=bool(config.rescale_q_values_in_search),  # selfplay.py:114-116
                                                        mlp_mode=int(getattr(config, "mlp_mode", _abi.MLP_EXACT)),
                                                        tasks=env.tasks if isinstance(env, Subleq) else (1,), device=str(states["terminated"].device),
                                                        fused_root=True))
    r = hit[2]
    tok = net.content_token()
    if getattr(r, "_net_token", None) != tok:  # rebuild the parameter-derived tables only when the parameters moved
        r.params_updated()
        r._net_token = tok
    gumbel = None
    if isinstance(rng_key, PreDrawnGumbel):
        gumbel = rng_key.gumbel
    elif isinstance(rng_key, int):
        r.gen.manual_seed(rng_key)
    states, out = r.scan(states, T, gumbel=gumbel)
    S = env.spec.compact_bytes
    dec = ops.env_uncompact(env.spec, out.state["compact"].reshape(T * B, S), out.state["rewards"].reshape(T * B))
    stacked = State(env, {k: v.reshape((T, B) + tuple(v.shape[1:])) for k, v in dec.items()})
    keep = lambda t: t.clone()
    return State(env, states), SelfplayOutput(state=stacked, root_value=keep(out.root_value), root_epistemic_std=keep(out.root_epistemic_std),
                                              value_prediction=keep(out.value_prediction), ube_prediction=keep(out.ube_prediction),
                                              q_values_epistemic_variance=keep(out.q_values_epistemic_variance), action=keep(out.action),
                                              trajectory=keep(out.trajectory))
