"""The evaluation loop as one device program (csrc/evaluate.cu: eaz_evaluate, eval_step_kernel) against the per-move host loop it
replaces -- the loop body of the former evaluate.py, run here as the reference: returns, final states leaf by leaf and the number of
moves must agree bit for bit."""
import ctypes as C

import numpy as np
import pytest

from e_alphazero_b200 import _abi
from tests import helpers as H

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch

    assert torch.cuda.is_available()
    return torch


def host_loop(torch, denv, dnet, cfg, max_len, beta, tasks=(1,), seed=0):
    """evaluate() as it was: one search, one env step and one `+=` per move, with the host checking termination in between."""
    from e_alphazero_b200 import ops

    B = cfg.batch
    gen = torch.Generator(device="cuda").manual_seed(seed)
    task_ids = None
    if denv.kind == _abi.ENV_SUBLEQ:
        tt = torch.tensor(list(tasks), dtype=torch.int32, device="cuda")
        task_ids = tt[torch.randint(0, tt.numel(), (B,), device="cuda", generator=gen)].contiguous()
    states = ops.env_init(denv, B, task_ids=task_ids)
    plan = ops.SearchPlan(cfg, denv, dnet, want_tree=False)
    beta_t = torch.full((B,), float(beta), device="cuda")
    gumbel = torch.zeros((B, denv.num_actions), device="cuda")
    total = torch.zeros(B, device="cuda")
    counter = 0
    while not bool(states["terminated"].all().item()) and counter <= max_len:
        out = plan.run(dict(beta=beta_t, embedding=states, gumbel=gumbel), reuse_prepared=counter > 0)
        states = ops.env_step(denv, states, out["action"])
        total += states["rewards"][:, 0]
        counter += 1
    return total, states, counter


def eval_cfg(B, n, gamma, mode, streams=1):
    cfg = _abi.default_search_config(batch=B, num_simulations=n, discount=gamma, exploration=0, gumbel_scale=0.0, rescale_values=1, mlp_mode=mode)
    if streams > 1:
        cfg.flags |= _abi.flag_streams(streams)
    return cfg


def assert_same_episode(torch, got_returns, got_states, got_moves, exp, what):
    total, states, counter = exp
    torch.cuda.synchronize()
    assert got_moves == counter, (what, got_moves, counter)
    H.assert_same_bits(got_returns.cpu().numpy(), total.cpu().numpy(), f"{what} returns")
    for k in states:
        H.assert_same_bits(got_states[k].cpu().numpy(), states[k].cpu().numpy(), f"{what} state {k}")


def run_device(torch, denv, dnet, cfg, max_len, beta, tasks=(1,), seed=0):
    from e_alphazero_b200 import ops
    from e_alphazero_b200.evaluate import EvaluateRunner

    r = EvaluateRunner(dnet, denv, cfg.batch, cfg.num_simulations, cfg.discount, max_len, beta, True, cfg.mlp_mode, tasks)
    if cfg.flags != r.cfg.flags:  # (EAZ_FLAG_STREAMS: the runner's plan with the caller's flags)
        r.cfg.flags = cfg.flags
        r.plan = ops.EvaluatePlan(r.cfg, denv, dnet)
    _, ret = r(seed)
    return r, ret


CASES = [  # (kind, env kwargs, B, simulations, mlp_mode, streams)
    ("deepsea", dict(size=10), 64, 16, _abi.MLP_EXACT, 1),
    ("deepsea", dict(size=10), 300, 16, _abi.MLP_EXACT, 2),   # EAZ_FLAG_STREAMS: fork / join inside the loop body
    ("deepsea", dict(size=10), 200, 16, _abi.MLP_TENSOR, 1),  # persistent ds_search_kernel
    ("deepsea", dict(size=6), 40000, 4, _abi.MLP_TENSOR, 1),  # tensor-mode launch chain (more trees than two waves of the persistent kernel)
    ("subleq", dict(word_size=16), 96, 16, _abi.MLP_EXACT, 1),
    ("subleq", dict(word_size=16), 70, 12, _abi.MLP_TENSOR, 1),
]


@pytest.mark.parametrize("max_len", [3, 60, 0])
@pytest.mark.parametrize("kind,kw,B,n,mode,streams", CASES)
def test_evaluate_equals_host_loop(torch, kind, kw, B, n, mode, streams, max_len):
    """max_len 3: stopped by the move counter; 60: above both horizons, stopped by termination; 0: exactly one move (counter <= 0)."""
    env = H.make_env(kind, seed=201, **kw)
    net = H.make_net(env, seed=202, fill=0.5)
    denv, dnet = H.device_env(env), H.device_net(net)
    cfg = eval_cfg(B, n, 0.97, mode, streams)
    tasks = (1, 2, 3)
    r, ret = run_device(torch, denv, dnet, cfg, max_len, 0.3, tasks, seed=5)
    exp = host_loop(torch, denv, dnet, cfg, max_len, 0.3, tasks, seed=5)
    assert_same_episode(torch, ret, r.states, r.plan.moves(), exp, f"{kind} B={B} mode={mode} max_len={max_len}")
    if max_len == 60:
        assert bool(r.states["terminated"].all())
    # the counters are re-armed and the condition is off once the loop has stopped
    moves, live, ticket, cont = r.plan.counters.cpu().tolist()
    assert (live, ticket, cont) == (0, 0, 0)


def test_evaluate_stops_when_every_env_solved(torch):
    """Subleq-16, task 1: a network whose policy plays 14 then 13 (the two-word program that solves task 1) -- every env is solved after
    move 2 and terminates in move 3, so the device counter stops at 3 moves, far below the horizon (ws - 3 = 13 steps)."""
    env = H.make_env("subleq", word_size=16)
    net = H.make_net(env, seed=211)
    w, b = net.w[_abi.HEAD_EXPLOIT], net.b[_abi.HEAD_EXPLOIT]
    for layer in (w, b):
        for x in layer:
            x[...] = 0
    w[0][1, 0] = 1.0  # hidden 0 = bit 1 of memory word 0 (observation row 0, column 1): set once 14 = 0b1110 is written there
    b[0][1] = 1.0     # hidden 1 = 1
    w[1][0, 0] = w[1][1, 1] = 1.0
    w[2][0, 13], w[2][1, 14], w[2][0, 14] = 50.0, 50.0, -50.0  # logits: 14 before the first move, 13 after it
    denv, dnet = H.device_env(env), H.device_net(net)
    cfg = eval_cfg(64, 16, 0.97, _abi.MLP_EXACT)
    r, ret = run_device(torch, denv, dnet, cfg, 100, 0.0, (1,))
    exp = host_loop(torch, denv, dnet, cfg, 100, 0.0, (1,))
    assert_same_episode(torch, ret, r.states, r.plan.moves(), exp, "solved early")
    assert r.plan.moves() == 3
    assert bool(r.states["solved"].all()) and bool(r.states["terminated"].all())
    assert float(ret.min()) > 0.0


def test_runner_after_parameter_update(torch):
    """Two evaluations on one runner (one graph) with an in-place parameter update in between: the second rebuilds the tables (here the
    tensor-core weight images) before its loop and equals a fresh host loop with the new parameters."""
    env = H.make_env("subleq", word_size=16)
    net = H.make_net(env, seed=222, fill=0.5)
    denv, dnet = H.device_env(env), H.device_net(net)
    cfg = eval_cfg(70, 12, 0.97, _abi.MLP_TENSOR)
    tasks = (1, 2, 3)
    r, ret = run_device(torch, denv, dnet, cfg, 60, 0.3, tasks)
    assert_same_episode(torch, ret, r.states, r.plan.moves(), host_loop(torch, denv, dnet, cfg, 60, 0.3, tasks), "first call")
    before = r.states["memory"].clone()
    g = torch.Generator(device="cuda").manual_seed(7)
    for h in range(4):
        for l in range(3):
            dnet.w[h][l].add_(torch.randn(dnet.w[h][l].shape, device="cuda", generator=g))
    _, ret = r(0)
    assert_same_episode(torch, ret, r.states, r.plan.moves(), host_loop(torch, denv, dnet, cfg, 60, 0.3, tasks), "after update")
    assert not torch.equal(before, r.states["memory"]), "the update must change the episodes (else this test shows nothing)"


def test_warm_evaluate_has_no_host_sync(torch):
    from e_alphazero_b200.evaluate import evaluate

    env = H.make_env("subleq", word_size=16)
    net = H.make_net(env, seed=231, fill=0.5)
    denv, dnet = H.device_env(env), H.device_net(net)
    args = (dnet, denv, 40, 8, 0.97, 20)
    m1, t1 = evaluate(*args, exploitation_beta=0.2, tasks=(1, 2, 3), seed=3)  # builds the graph
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        m2, t2 = evaluate(*args, exploitation_beta=0.2, tasks=(1, 2, 3), seed=3)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert torch.equal(t1, t2) and torch.equal(m1, m2)


@pytest.mark.parametrize("kind,kw,B", [("deepsea", dict(size=8), 700), ("subleq", dict(word_size=16), 90), ("subleq", dict(word_size=40), 33)])
def test_eval_step_kernel_outside_graph(torch, kind, kw, B):
    """eval_step_kernel launched on its own, move by move, equals eaz_env_step + `returns += rewards[:, 0]`; its counters count the
    moves and its decision is cond_fn (evaluate.py:18-20) on the stepped states."""
    from e_alphazero_b200 import _lib, ops

    lib = _lib.load()
    env = H.make_env(kind, seed=241, **kw)
    denv = H.device_env(env)
    rng = np.random.default_rng(242)
    tasks = torch.as_tensor(rng.integers(1, 4, B).astype(np.int32), device="cuda") if kind == "subleq" else None
    ref = ops.env_init(denv, B, task_ids=tasks)
    got = {k: v.clone() for k, v in ref.items()}
    ref_total = torch.zeros(B, device="cuda")
    got_total = torch.zeros(B, device="cuda")
    ctr = torch.zeros(4, dtype=torch.int32, device="cuda")
    max_len = 6
    for move in range(1, 12):
        act = rng.integers(0, denv.num_actions, B).astype(np.int32)
        if kind == "subleq":
            act = np.where(rng.random(B) < 0.5, rng.integers(denv.word_size - 4, denv.word_size, B), act).astype(np.int32)
        a = torch.as_tensor(act, device="cuda")
        ref = ops.env_step(denv, ref, a)
        ref_total += ref["rewards"][:, 0]
        e, s = denv.struct(), ops.state_struct(denv, got)
        rc = lib.eaz_debug_eval_step(C.byref(e), C.byref(s), ops._ptr(a), ops._ptr(got_total), ops._ptr(ctr), max_len, B, ops._stream())
        assert rc == 0, lib.eaz_last_error()
        torch.cuda.synchronize()
        for k in ref:
            H.assert_same_bits(got[k].cpu().numpy(), ref[k].cpu().numpy(), f"move {move} {k}")
        H.assert_same_bits(got_total.cpu().numpy(), ref_total.cpu().numpy(), f"move {move} returns")
        moves, live, ticket, cont = ctr.cpu().tolist()
        assert (moves, live, ticket) == (move, 0, 0)
        assert cont == int(bool((ref["terminated"] == 0).any()) and move <= max_len), move
