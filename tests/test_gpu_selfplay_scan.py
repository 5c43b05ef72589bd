"""The self-play scan as one device program (csrc/selfplay.cu: eaz_selfplay, selfplay_step_kernel) against the steps it replaces: T
eager SelfplayRunner(fused_root=True).step() calls given the same per-step noise and reset tasks.  Every stacked output, the trajectory
records, the compact states and rewards of every step and the final state leaves must agree bit for bit.

With EAZ_NO_PERSISTENT set (read once per process by the library) the DeepSea tensor-core cases run the launch chain instead of the
persistent kernel; test_launch_chain_subprocess re-runs them that way."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from e_alphazero_b200 import _abi
from tests import helpers as H

pytestmark = pytest.mark.gpu

NO_PERSISTENT = os.environ.get("EAZ_NO_PERSISTENT") is not None
FIELDS = ["action", "root_value", "root_epistemic_std", "value_prediction", "ube_prediction", "q_values_epistemic_variance", "trajectory"]


@pytest.fixture(scope="module")
def torch():
    import torch

    assert torch.cuda.is_available()
    return torch


def setup(kind, kw, seed=401):
    env = H.make_env(kind, seed=seed, **kw)
    net = H.make_net(env, seed=seed + 1, fill=0.5)
    return env, H.device_env(env), net


def runner(denv, dnet, B, n, mode, streams=1, **kw):
    from e_alphazero_b200.selfplay import SelfplayRunner

    r = SelfplayRunner(denv, dnet, B, n, 0.97, exploration_beta=0.4, directed_exploration=True, mlp_mode=mode, fused_root=True, streams=streams,
                       seed=77, **kw)
    r.plan.workspace.zero_()  # the draw counter of step()'s workspace starts at 0, as in a fresh scan workspace
    return r


def inputs(torch, denv, B, T, seed, sample=False, tasks=(1, 2, 3)):
    g = torch.Generator(device="cuda").manual_seed(seed)
    noise = lambda: -(-torch.rand((T, B, denv.num_actions), device="cuda", generator=g).clamp_(1e-20, 1 - 1e-7).log()).log()
    gumbel = noise()
    samp = noise() if sample else None
    tt = None
    if denv.kind == _abi.ENV_SUBLEQ:
        pool = torch.tensor(list(tasks), dtype=torch.int32, device="cuda")
        tt = pool[torch.randint(0, pool.numel(), (T, B), device="cuda", generator=g)].contiguous()
    return gumbel, samp, tt


def init_states(torch, denv, B, seed=3):
    from e_alphazero_b200 import ops

    tasks = torch.tensor(np.random.default_rng(seed).integers(1, 4, B).astype(np.int32), device="cuda") if denv.kind == _abi.ENV_SUBLEQ else None
    return ops.env_init(denv, B, task_ids=tasks)


def eager(torch, r, denv, states, T, gumbel, sample, tasks):
    """T step() calls; returns the per-step rows stacked like a scan's outputs."""
    from e_alphazero_b200 import ops

    rows = {k: [] for k in FIELDS + ["states", "rewards"]}
    for t in range(T):
        _, out = r.step(states, gumbel=None if gumbel is None else gumbel[t], task_ids=None if tasks is None else tasks[t],
                        sample_gumbel=None if sample is None else sample[t])
        rec = r.trajectory(states, out, torch.empty((r.B, 4), dtype=torch.int32, device="cuda"))
        for k in FIELDS[:-1]:
            rows[k].append(getattr(out, k).clone())
        rows["trajectory"].append(rec.clone())
        rows["states"].append(ops.env_compact(denv, states))
        rows["rewards"].append(states["rewards"][:, 0].clone())
    return {k: torch.stack(v) for k, v in rows.items()}


def assert_scan_equals(torch, got_states, out, exp_states, exp, what):
    torch.cuda.synchronize()
    for k in FIELDS:
        H.assert_same_bits(getattr(out, k).cpu().numpy(), exp[k].cpu().numpy(), f"{what} {k}")
    H.assert_same_bits(out.state["compact"].cpu().numpy(), exp["states"].cpu().numpy(), f"{what} compact states")
    H.assert_same_bits(out.state["rewards"].cpu().numpy(), exp["rewards"].cpu().numpy(), f"{what} rewards")
    for k in exp_states:
        H.assert_same_bits(got_states[k].cpu().numpy(), exp_states[k].cpu().numpy(), f"{what} final state {k}")


def check_case(torch, kind, kw, B, n, mode, T, streams=1, sample=False, device_noise=False, **rkw):
    env, denv, net = setup(kind, kw)
    init = init_states(torch, denv, B)
    gumbel, samp, tasks = inputs(torch, denv, B, T, seed=9, sample=sample)
    if device_noise:
        gumbel = samp = None
    ref = runner(denv, H.device_net(net), B, n, mode, streams, device_noise=device_noise, **rkw)
    exp_states = {k: v.clone() for k, v in init.items()}
    exp = eager(torch, ref, denv, exp_states, T, gumbel, samp, tasks)
    r = runner(denv, H.device_net(net), B, n, mode, streams, device_noise=device_noise, **rkw)
    states = {k: v.clone() for k, v in init.items()}
    _, out = r.scan(states, T, gumbel=gumbel, sample_gumbel=samp, task_ids=tasks)
    assert_scan_equals(torch, states, out, exp_states, exp, f"{kind} B={B} mode={mode} T={T}")
    return states, out, exp


def test_deepsea_exact_resets_mid_scan(torch):
    """DeepSea-10 episodes end after 9 steps: with T = 12 every env terminates and is reset inside the scan."""
    states, out, _ = check_case(torch, "deepsea", dict(size=10), 64, 16, _abi.MLP_EXACT, 12)
    flags = out.trajectory[:, :, 2].cpu().numpy()
    assert (flags[8] & 1).all() and not (flags[9] & 1).any(), "step 9 ends every episode, step 10 resets it"


TENSOR_CASES = [  # (B, simulations, streams)
    (200, 16, 1),  # persistent ds_search_kernel (launch chain under EAZ_NO_PERSISTENT)
    (300, 16, 2),  # EAZ_FLAG_STREAMS(2): fork / join inside the loop body on the launch chain
]


@pytest.mark.parametrize("B,n,streams", TENSOR_CASES)
def test_deepsea_tensor(torch, B, n, streams):
    check_case(torch, "deepsea", dict(size=30), B, n, _abi.MLP_TENSOR, 8, streams=streams)


def test_launch_chain_subprocess():
    """test_deepsea_tensor once more with EAZ_NO_PERSISTENT=1 (read once per process, hence the subprocess): the launch chain
    (mlp_gather_kernel + tree_step*_kernel) inside the loop body."""
    if NO_PERSISTENT:
        pytest.skip("this process already runs the launch chain")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, EAZ_NO_PERSISTENT="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k", "deepsea_tensor", "-p", "no:cacheprovider"],
                       cwd=root, env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and "failed" not in r.stdout


@pytest.mark.parametrize("mode", [_abi.MLP_EXACT, _abi.MLP_TENSOR])
def test_subleq_every_env_resets(torch, mode):
    """Subleq-16 binary, tasks 1-3: episodes end after at most ws - 3 = 13 steps, so T = 16 resets every env at least once, with the
    task of row t of task_ids."""
    states, out, _ = check_case(torch, "subleq", dict(word_size=16), 70, 12, mode, 16)
    term = out.trajectory[:, :, 2].cpu().numpy() & 1
    assert term.any(axis=0).all(), "every env must terminate (and so reset) inside the scan"


@pytest.mark.parametrize("opts", [dict(uniform_prior=True), dict(action_sampling="visit_counts", temperature=0.7),
                                  dict(action_sampling="improved_policy")])
@pytest.mark.parametrize("kind,kw,B", [("deepsea", dict(size=10), 64), ("subleq", dict(word_size=16), 40)])
def test_step_options(torch, kind, kw, B, opts):
    check_case(torch, kind, kw, B, 12, _abi.MLP_EXACT, 5, sample="action_sampling" in opts, **opts)


@pytest.mark.parametrize("opts", [dict(), dict(action_sampling="improved_policy")])
def test_in_search_noise(torch, opts):
    """device_noise=True: both noises are drawn in the search from the workspace's draw counter.  A scan on a fresh runner equals T eager
    steps from the same seed only if the table preparation before the loop leaves the counter alone and every step advances it once."""
    check_case(torch, "deepsea", dict(size=10), 64, 16, _abi.MLP_EXACT, 6, device_noise=True, **opts)


def test_one_step(torch):
    check_case(torch, "subleq", dict(word_size=16), 33, 8, _abi.MLP_EXACT, 1)


def test_zero_steps_write_nothing(torch):
    from e_alphazero_b200 import _lib, ops

    env, denv, net = setup("deepsea", dict(size=10))
    B = 32
    r = runner(denv, H.device_net(net), B, 8, _abi.MLP_EXACT)
    init = init_states(torch, denv, B)
    states = {k: v.clone() for k, v in init.items()}
    _, out = r.scan(states, 0)
    assert out.action.shape == (0, B)
    plan = r._scan_plan
    bufs = ops.alloc_selfplay_outputs(denv, 1, B)
    for t in bufs.values():
        t.fill_(7)
    o = _abi.EazSelfplayOutputs(*[ops._ptr(bufs[k]) for k in ops.SELFPLAY_OUTPUTS])
    e, n, s = denv.struct(), r.net.struct(), ops.state_struct(denv, states)
    inp = _abi.EazSearchInputs(None, None, None, ops._ptr(r.beta), None, None, None, C.pointer(e), None, None)
    rc = _lib.load().eaz_selfplay(C.byref(r.cfg), C.byref(inp), C.byref(n), C.byref(s), 0, None, C.byref(o), plan._ws_ptr, plan._ws_bytes,
                                  ops._stream())
    assert rc == 0
    torch.cuda.synchronize()
    for k, t in bufs.items():
        assert (t == 7).all(), k
    for k in init:
        H.assert_same_bits(states[k].cpu().numpy(), init[k].cpu().numpy(), f"state {k}")


def test_two_scans_with_parameter_update(torch):
    """Two scans on one runner with an in-place parameter update and params_updated() in between: the second scan rebuilds the tables
    (here the tensor-core weight images) before its loop, and equals eager steps that saw the same update."""
    env, denv, net = setup("subleq", dict(word_size=16))
    B, n, T = 70, 12, 6
    init = init_states(torch, denv, B)
    g1, _, t1 = inputs(torch, denv, B, T, seed=21)
    g2, _, t2 = inputs(torch, denv, B, T, seed=22)
    nets = [H.device_net(net), H.device_net(net)]
    ref, r = runner(denv, nets[0], B, n, _abi.MLP_TENSOR), runner(denv, nets[1], B, n, _abi.MLP_TENSOR)
    exp_states = {k: v.clone() for k, v in init.items()}
    states = {k: v.clone() for k, v in init.items()}
    eager(torch, ref, denv, exp_states, T, g1, None, t1)
    r.scan(states, T, gumbel=g1, task_ids=t1)
    for dn in nets:
        g = torch.Generator(device="cuda").manual_seed(7)
        for h in range(4):
            for l in range(3):
                dn.w[h][l].add_(torch.randn(dn.w[h][l].shape, device="cuda", generator=g))
    ref.params_updated()
    r.params_updated()
    exp = eager(torch, ref, denv, exp_states, T, g2, None, t2)
    _, out = r.scan(states, T, gumbel=g2, task_ids=t2)
    assert_scan_equals(torch, states, out, exp_states, exp, "after update")


def test_new_output_buffers_rebuild_the_graph(torch):
    """A second call on the same workspace with other output buffers rebuilds the graph: the new buffers get the rows, the old ones are
    left alone."""
    from e_alphazero_b200 import ops

    env, denv, net = setup("deepsea", dict(size=10))
    B, n, T = 64, 16, 7
    init = init_states(torch, denv, B)
    gumbel, _, _ = inputs(torch, denv, B, T, seed=31)
    ref = runner(denv, H.device_net(net), B, n, _abi.MLP_EXACT)
    exp_states = {k: v.clone() for k, v in init.items()}
    exp = eager(torch, ref, denv, exp_states, T, gumbel, None, None)
    r = runner(denv, H.device_net(net), B, n, _abi.MLP_EXACT)
    plan = ops.SelfplayPlan(r.cfg, denv, r.net)
    first = ops.alloc_selfplay_outputs(denv, T, B)
    states = {k: v.clone() for k, v in init.items()}
    plan.run(r.beta, states, T, first, gumbel=gumbel)
    for t in first.values():
        t.zero_()
    second = ops.alloc_selfplay_outputs(denv, T, B)
    states = {k: v.clone() for k, v in init.items()}
    plan.run(r.beta, states, T, second, gumbel=gumbel, reuse_prepared=True)
    torch.cuda.synchronize()
    for k, t in first.items():
        assert not t.view(torch.uint8).any(), f"old buffer {k} was written"
    for k in FIELDS:
        H.assert_same_bits(second[k].cpu().numpy(), exp[k].cpu().numpy(), f"new buffers {k}")
    H.assert_same_bits(second["states"].cpu().numpy(), exp["states"].cpu().numpy(), "new buffers states")
    H.assert_same_bits(second["rewards"].cpu().numpy(), exp["rewards"].cpu().numpy(), "new buffers rewards")
    for k in exp_states:
        H.assert_same_bits(states[k].cpu().numpy(), exp_states[k].cpu().numpy(), f"final state {k}")


def test_warm_scan_has_no_host_sync(torch):
    env, denv, net = setup("subleq", dict(word_size=16))
    B, T = 40, 5
    r = runner(denv, H.device_net(net), B, 8, _abi.MLP_EXACT, tasks=(1, 2, 3))
    init = init_states(torch, denv, B)
    states = {k: v.clone() for k, v in init.items()}
    r.scan(states, T)  # builds the graph (noise and tasks from the runner's generator)
    torch.cuda.synchronize()
    first = r.scan(states, T)[1].trajectory.clone()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        _, out = r.scan(states, T)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert out.trajectory.shape == (T, B, 4) and not torch.equal(first, out.trajectory)


def test_selfplay_drop_in(torch):
    """selfplay(model, config, context, last_states, rng_key): the decoded `state` equals ops.env_uncompact of the compact rows of the
    same scan, the other outputs equal a runner's scan, and last_states is left alone."""
    from types import SimpleNamespace

    from e_alphazero_b200 import ops, pgx
    from e_alphazero_b200.emctx import PreDrawnGumbel
    from e_alphazero_b200.selfplay import SelfplayRunner, selfplay

    env, denv, net = setup("deepsea", dict(size=10))
    B, T, n = 48, 8, 16
    penv = pgx.DeepSea(10, env.action_map)
    dnet = H.device_net(net)
    config = SimpleNamespace(selfplay_steps=T, selfplay_simulations_per_step=n, discount=0.97, exploration_beta=0.3, directed_exploration=True,
                             rescale_q_values_in_search=True)
    last = penv.init(batch_size=B)
    before = {k: v.clone() for k, v in last.leaves.items()}
    gumbel, _, _ = inputs(torch, denv, B, T, seed=41)
    final, out = selfplay(dnet, config, SimpleNamespace(env=penv), last, PreDrawnGumbel(gumbel))
    r = SelfplayRunner(penv.spec, dnet, B, n, 0.97, exploration_beta=0.3, directed_exploration=True, fused_root=True)
    states = {k: v.clone() for k, v in before.items()}
    _, ref = r.scan(states, T, gumbel=gumbel)
    torch.cuda.synchronize()
    dec = ops.env_uncompact(penv.spec, ref.state["compact"].reshape(T * B, -1), ref.state["rewards"].reshape(T * B))
    for k, v in dec.items():
        H.assert_same_bits(out.state.leaves[k].cpu().numpy(), v.reshape(out.state.leaves[k].shape).cpu().numpy(), f"decoded {k}")
        assert out.state.leaves[k].shape[:2] == (T, B)
    for k in FIELDS:
        H.assert_same_bits(getattr(out, k).cpu().numpy(), getattr(ref, k).cpu().numpy(), f"drop-in {k}")
    for k in states:
        H.assert_same_bits(final.leaves[k].cpu().numpy(), states[k].cpu().numpy(), f"final {k}")
        H.assert_same_bits(last.leaves[k].cpu().numpy(), before[k].cpu().numpy(), f"last_states {k} untouched")
