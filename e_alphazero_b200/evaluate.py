"""Mirror of the reference's evaluate.py:13-57 on the fused CUDA path: greedy (gumbel_scale = 0) episodes from `env.init`
until every env has terminated or `max_episode_length` steps have passed; plain `env.step` (no auto-reset: terminated envs are
absorbing and contribute zero reward), exploitation logits at the root, the recurrent_fn's exploitation head inside the tree,
beta = config.exploitation_beta.  Returns the mean sum of rewards (evaluate.py:57).

The whole loop is one eaz_evaluate call: a CUDA graph whose WHILE node repeats the search and the env step and whose condition the
device decides (csrc/evaluate.cu), so the host neither waits nor launches per move.  `EvaluateRunner` owns the buffers, so that the
evaluations of a training run (every evaluation_interval) reuse the graph built by the first one."""
from __future__ import annotations

from . import _abi, ops
from ._lib import require_cuda


class EvaluateRunner:
    """evaluate() for a fixed (env, net, batch, search) configuration: workspace, env states, returns and the task pool."""

    def __init__(self, net: ops.FcParams, env_spec: ops.EnvSpec, num_eval_episodes: int, num_simulations: int, discount: float,
                 max_episode_length: int, exploitation_beta: float = 0.0, rescale_values: bool = True, mlp_mode: int = _abi.MLP_EXACT,
                 tasks=(1,), device="cuda"):
        torch = require_cuda()
        B = int(num_eval_episodes)
        self.env, self.net, self.B, self.device = env_spec, net, B, device
        self.max_episode_length = int(max_episode_length)
        self.cfg = _abi.default_search_config(batch=B, num_simulations=int(num_simulations), discount=float(discount), exploration=0, gumbel_scale=0.0,
                                              rescale_values=int(rescale_values), mlp_mode=int(mlp_mode))
        self.plan = ops.EvaluatePlan(self.cfg, env_spec, net, device=device)
        self.beta = torch.full((B,), float(exploitation_beta), device=device)  # :34
        self.returns = torch.zeros(B, device=device)
        self.states = ops.alloc_state(env_spec, B, device=device)
        self.task_pool = torch.tensor(list(tasks), dtype=torch.int32, device=device) if env_spec.kind == _abi.ENV_SUBLEQ else None
        self.task_ids = torch.empty(B, dtype=torch.int32, device=device)
        self.gen = torch.Generator(device=device)

    def __call__(self, seed: int = 0):
        """One evaluation: env.init (evaluate.py:52-54), then the episode loop.  Returns (mean, returns) as device tensors; `returns`
        and `states` are this runner's buffers (the next call overwrites them)."""
        import torch

        task_ids = None
        if self.task_pool is not None:  # Subleq._init draws the task (subleq.py:624): once per evaluation, from `seed`
            self.gen.manual_seed(seed)
            torch.index_select(self.task_pool, 0, torch.randint(0, self.task_pool.numel(), (self.B,), device=self.device, generator=self.gen),
                               out=self.task_ids)
            task_ids = self.task_ids
        ops.env_init_(self.env, self.states, task_ids)
        self.plan.run(self.beta, self.states, self.returns, self.max_episode_length)
        return self.returns.mean(), self.returns


_runners: dict = {}


def evaluate(net: ops.FcParams, env_spec: ops.EnvSpec, num_eval_episodes: int, num_simulations: int, discount: float, max_episode_length: int,
             exploitation_beta: float = 0.0, rescale_values: bool = True, mlp_mode: int = _abi.MLP_EXACT, tasks=(1,), device="cuda", seed: int = 0):
    key = (id(env_spec), id(net), int(num_eval_episodes), int(num_simulations), float(discount), int(max_episode_length), float(exploitation_beta),
           bool(rescale_values), int(mlp_mode), tuple(int(t) for t in tasks), str(device))
    hit = _runners.get(key)  # (env, net, runner): the strong references keep the id()s in the key unique
    if hit is None or hit[0] is not env_spec or hit[1] is not net:
        while len(_runners) >= 8:
            _runners.pop(next(iter(_runners)))
        hit = _runners[key] = (env_spec, net, EvaluateRunner(net, env_spec, num_eval_episodes, num_simulations, discount, max_episode_length,
                                                             exploitation_beta, rescale_values, mlp_mode, tasks, device))
    mean, total = hit[2](seed)
    return mean, total.clone()
