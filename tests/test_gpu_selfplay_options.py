"""The optional parts of the self-play step inside the search (eaz_search_config.root_prior / action_sampling, selfplay.py:92-98,
125-134): bit-exact parity with the CPU oracle (tests/selfplay_oracle.c) in EXACT mode, the draw on the GPU's own search results in
TENSOR mode (persistent DeepSea kernel, launch chain, two trees per warp, EAZ_FLAG_STREAMS), the in-kernel noise stream and its draw
counter, the sampled distribution, the uniform root, SelfplayRunner graph == eager, and the argument checks."""
import ctypes as C

import numpy as np
import pytest

from e_alphazero_b200 import _abi
from tests import helpers as H
from tests import selfplay_oracle as SO

pytestmark = pytest.mark.gpu

F32_MIN = np.float32(-3.4028234663852886e38)
ENVS = {"deepsea10": ("deepsea", dict(size=10)), "deepsea30": ("deepsea", dict(size=30)), "subleq16": ("subleq", dict(word_size=16)),
        "subleq20_onehot": ("subleq", dict(word_size=20, binary=False))}
PRIORS = {"given": _abi.ROOT_PRIOR_GIVEN, "uniform": _abi.ROOT_PRIOR_UNIFORM}
SAMPLING = {"search": _abi.ACTION_SEARCH, "visits": _abi.ACTION_VISITS, "improved": _abi.ACTION_IMPROVED}


@pytest.fixture(scope="module")
def ops():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from e_alphazero_b200 import ops as _ops

    return _ops


def host(t):
    return t.detach().cpu().numpy()


_CASES = {}


def case(name, B=64):
    """(env, net, root) of one environment: rows with invalid actions, row 0 all invalid, pre-drawn gumbel and sample_gumbel."""
    if (name, B) not in _CASES:
        kind, kw = ENVS[name]
        env = H.make_env(kind, seed=11, **kw)
        net = H.make_net(env, seed=12, fill=0.5)
        root = H.make_root(env, net, B, seed=13, invalid_frac=0.25)
        root["sample_gumbel"] = np.random.default_rng(14).gumbel(size=(B, env.num_actions)).astype(np.float32)
        _CASES[(name, B)] = (env, net, root)
    return _CASES[(name, B)]


def gpu_search(ops, env, net, root, cfg, fused=False, want_tree=True, drop=()):
    denv, dnet = H.device_env(env), H.device_net(net)
    droot = H.device_root(env, denv, root)
    for k in (("prior_logits", "value", "value_epistemic_variance") if fused else ()) + tuple(drop):
        droot.pop(k, None)
    plan = ops.SearchPlan(_abi.EazSearchConfig.from_buffer_copy(cfg), denv, dnet, want_tree=want_tree)
    return {k: host(v).copy() for k, v in plan.run(droot).items()}, plan


def launches(ops, plan, n):
    cfg = _abi.EazSearchConfig.from_buffer_copy(plan.cfg)
    cfg.num_simulations = n
    return ops.load().eaz_search_num_launches(C.byref(cfg), C.byref(plan.env.struct()))


def ran_persistent(ops, plan):
    """As test_gpu_tensor_search.ran_persistent: ds_search_kernel's launch count does not grow with num_simulations."""
    return plan.num_launches == launches(ops, plan, plan.cfg.num_simulations - 1)


def weights_of(got, sampling):
    return got["visit_probs"] if sampling == _abi.ACTION_VISITS else got["action_weights"]


# ----------------------------------------------------------------------------- 1. exact parity with the oracle
@pytest.mark.parametrize("fused", [False, True], ids=["caller_root", "fused_root"])
@pytest.mark.parametrize("sampling", list(SAMPLING))
@pytest.mark.parametrize("prior", list(PRIORS))
@pytest.mark.parametrize("name", list(ENVS))
def test_exact_parity(ops, name, prior, sampling, fused):
    env, net, root = case(name)
    cfg = _abi.default_search_config(batch=64, num_simulations=20, discount=0.97, root_prior=PRIORS[prior], action_sampling=SAMPLING[sampling],
                                     temperature=0.8)
    exp = SO.search(_abi.EazSearchConfig.from_buffer_copy(cfg), env, net, root, want_tree=True, fused_root=fused)
    got, _ = gpu_search(ops, env, net, root, cfg, fused)
    for name_, _, _ in _abi.SUMMARY_FIELDS + _abi.TREE_FIELDS:
        H.assert_same_bits(got[name_], exp[name_], name_)
    if fused:
        H.assert_same_bits(got["root_value"], exp["root_value"], "root_value")
        H.assert_same_bits(got["root_ube"], exp["root_ube"], "root_ube")
    inv = root["invalid_actions"].astype(bool)
    dead = inv.all(1)  # rows whose actions are all invalid (row 0, and some DeepSea rows) play 0; no other row plays an invalid one
    assert dead[0] and (got["action"][dead] == 0).all()
    assert not inv[~dead, got["action"][~dead]].any()
    if sampling != "search":  # the draw is not the search's action everywhere
        assert (exp["search_action"] != got["action"]).any()


# ----------------------------------------------------------------------------- 2. TENSOR mode: every search path through the two kernels
def check_tensor_draws(ops, env, net, root, B, n, persistent, streams=0):
    ref = None
    for prior in PRIORS.values():
        for sampling in SAMPLING.values():
            cfg = _abi.default_search_config(batch=B, num_simulations=n, discount=0.97, mlp_mode=_abi.MLP_TENSOR, root_prior=prior,
                                             action_sampling=sampling, temperature=0.7)
            got, plan = gpu_search(ops, env, net, root, cfg, want_tree=False)
            if persistent is not None:
                assert ran_persistent(ops, plan) == persistent, f"num_launches {plan.num_launches}"
            if sampling == _abi.ACTION_SEARCH:
                ref = got
                continue
            exp = SO.sample_actions(weights_of(got, sampling), root["sample_gumbel"], 0.7, root["invalid_actions"])
            H.assert_same_bits(got["action"], exp, "action")
            for k in got:  # only the action changes
                if k != "action":
                    H.assert_same_bits(got[k], ref[k], k)
            assert (got["action"] != ref["action"]).any()
            if streams:  # EAZ_FLAG_STREAMS(k): sub-batches searched concurrently, identical results
                cfg.flags |= _abi.flag_streams(streams)
                got_k, _ = gpu_search(ops, env, net, root, cfg, want_tree=False)
                for k in got:
                    H.assert_same_bits(got_k[k], got[k], f"streams {k}")


def test_tensor_persistent_deepsea(ops):
    env = H.make_env("deepsea", seed=21, size=10)
    net = H.make_net(env, seed=22, fill=0.5)
    B = 512
    root = H.make_root(env, net, B, seed=23, invalid_frac=0.2)
    root["sample_gumbel"] = np.random.default_rng(24).gumbel(size=(B, 2)).astype(np.float32)
    check_tensor_draws(ops, env, net, root, B, 24, persistent=True, streams=4)


def test_tensor_launch_chain_two_trees_per_warp(ops):
    """16384 DeepSea trees: more than two waves of ds_search_kernel's CTAs, so the launch chain with two trees per warp
    (tree_step2_kernel, batches >= 6144) runs.  (Not with EAZ_FLAG_STREAMS: its 4096-tree sub-batches would take the persistent kernel,
    whose network outputs come from the per-cell table instead of mlp_gather_kernel.)"""
    env = H.make_env("deepsea", seed=31, size=10)
    net = H.make_net(env, seed=32, fill=0.5)
    B = 16384
    root = H.make_root(env, net, B, seed=33, invalid_frac=0.2)
    root["sample_gumbel"] = np.random.default_rng(34).gumbel(size=(B, 2)).astype(np.float32)
    check_tensor_draws(ops, env, net, root, B, 8, persistent=False)


def test_tensor_launch_chain_subleq(ops):
    env, net, root = case("subleq16", B=384)
    check_tensor_draws(ops, env, net, root, 384, 16, persistent=False, streams=4)


# ----------------------------------------------------------------------------- 3. in-kernel noise and the draw counter
@pytest.mark.parametrize("streams", [0, 4])
def test_in_kernel_noise_and_draw_counter(ops, streams):
    env, net, root = case("deepsea10", B=300)  # 300 trees: sub-batches of 128, 128, 44 with EAZ_FLAG_STREAMS
    B, A, seed = 300, env.num_actions, 0xC0FFEE
    cfg = _abi.default_search_config(batch=B, num_simulations=16, discount=0.97, noise_seed=seed, flags=_abi.SEARCH_DEFAULT_FLAGS | _abi.flag_streams(streams))
    denv, dnet = H.device_env(env), H.device_net(net)
    plan = ops.SearchPlan(cfg, denv, dnet, want_tree=False)
    plan.workspace.zero_()  # a fresh workspace's draw counter is whatever the allocation held: start the counters at 0
    full = H.device_root(env, denv, root)

    def run(sampling, root_noise, sample_noise):
        plan.cfg.action_sampling = sampling
        d = dict(full)
        if not root_noise:
            d.pop("gumbel")
        if not sample_noise:
            d.pop("sample_gumbel")
        return {k: host(v).copy() for k, v in plan.run(d).items()}

    def oracle(sampling, root_ctr, sample_ctr):
        r = dict(root)
        if root_ctr is not None:
            r["gumbel"] = SO.stream_gumbel(seed, root_ctr, B, A, sample=False)
        if sample_ctr is not None:
            r["sample_gumbel"] = SO.stream_gumbel(seed, sample_ctr, B, A)
        c = _abi.EazSearchConfig.from_buffer_copy(cfg)
        c.action_sampling = sampling
        return SO.search(c, env, net, r, want_tree=False)

    V = _abi.ACTION_VISITS
    steps = [  # (sampling, caller root noise, caller sample noise) -> oracle counters (root, sample); the counter after each step
        ((_abi.ACTION_SEARCH, False, False), (0, None)),  # root noise only: counter 0 -> 1, as before the options
        ((V, True, True), (None, None)),                  # everything supplied: no advance
        ((V, True, False), (None, 1)),                    # sample noise only: 1 -> 2
        ((V, False, False), (2, 2)),                      # both streams share one counter value: 2 -> 3
        ((V, False, False), (3, 3)),                      # ... and the next search draws new noise
        ((_abi.ACTION_SEARCH, False, False), (4, None)),
    ]
    acts = []
    for (sampling, rn, sn), (rc, sc) in steps:
        got = run(sampling, rn, sn)
        exp = oracle(sampling, rc, sc)
        for name_, _, _ in _abi.SUMMARY_FIELDS:
            H.assert_same_bits(got[name_], exp[name_], f"{(sampling, rn, sn)} {name_}")
        acts.append(got["action"])
    assert (acts[3] != acts[4]).any()  # two consecutive searches drew different noise


# ----------------------------------------------------------------------------- 4. the sampled distribution
def test_sampled_distribution(ops):
    """4096 identical Subleq-16 roots with one fixed root noise: every tree is the same and only the noise of the draw (drawn in the
    kernel, new on every search) varies; ~10^6 draws per setting against visit_probs^(1/T) (normalised) and action_weights."""
    import torch
    from scipy import stats

    env = H.make_env("subleq", seed=41, word_size=16)
    net = H.make_net(env, seed=42, fill=0.5)
    one = H.make_root(env, net, 8, seed=43)
    B, A, reps = 4096, env.num_actions, 245
    root = {k: (np.repeat(v[3:4], B, axis=0) if k != "embedding" else {f: np.repeat(x[3:4], B, axis=0) for f, x in v.items()})
            for k, v in one.items()}
    denv, dnet = H.device_env(env), H.device_net(net)
    droot = H.device_root(env, denv, root)
    for sampling, T in ((_abi.ACTION_VISITS, 1.0), (_abi.ACTION_VISITS, 0.5), (_abi.ACTION_IMPROVED, 1.0)):
        cfg = _abi.default_search_config(batch=B, num_simulations=32, discount=0.97, action_sampling=sampling, temperature=T, noise_seed=7)
        plan = ops.SearchPlan(cfg, denv, dnet, want_tree=False)
        counts = torch.zeros(A, dtype=torch.int64, device="cuda")
        for r in range(reps):
            out = plan.run(droot, reuse_prepared=r > 0)
            counts += torch.bincount(out["action"].long(), minlength=A)
        w = host(weights_of(out, sampling)).astype(np.float64)
        assert (w == w[0]).all(), "the trees differ"
        p = w[0] ** (1.0 / T)
        p /= p.sum()
        obs = host(counts)
        live = p > 1e-12
        assert obs[~live].sum() == 0 and live.sum() >= 2
        pval = stats.chisquare(obs[live], obs.sum() * p[live] / p[live].sum()).pvalue
        assert pval > 1e-3, (sampling, T, obs, p, pval)


# ----------------------------------------------------------------------------- 5. the uniform root prior
@pytest.mark.parametrize("mlp_mode", [_abi.MLP_EXACT, _abi.MLP_TENSOR])
@pytest.mark.parametrize("name", ["deepsea10", "subleq16"])
def test_uniform_prior(ops, name, mlp_mode):
    env, net, root = case(name)
    kw = dict(batch=64, num_simulations=20, discount=0.97, mlp_mode=mlp_mode)
    uni = _abi.default_search_config(root_prior=_abi.ROOT_PRIOR_UNIFORM, **kw)
    fused, _ = gpu_search(ops, env, net, root, uni, fused=True)
    inv = root["invalid_actions"].astype(bool)
    pl = fused["children_prior_logits"][:, 0]
    assert (pl[~inv] == 0).all() and (pl[inv] == F32_MIN).all()
    # the fused root == the caller's root with zero logits and the network's value / UBE
    caller = dict(root, prior_logits=np.zeros_like(root["prior_logits"]), value=fused["root_value"], value_epistemic_variance=fused["root_ube"])
    got, _ = gpu_search(ops, env, net, caller, _abi.default_search_config(**kw))
    for name_, _, _ in _abi.SUMMARY_FIELDS + _abi.TREE_FIELDS:
        H.assert_same_bits(fused[name_], got[name_], name_)
    # root_value / root_ube are those of the search without the option
    given, _ = gpu_search(ops, env, net, root, _abi.default_search_config(**kw), fused=True)
    H.assert_same_bits(fused["root_value"], given["root_value"], "root_value")
    H.assert_same_bits(fused["root_ube"], given["root_ube"], "root_ube")
    assert not np.array_equal(fused["action_weights"], given["action_weights"])
    # with a caller root the given logits are ignored: only value / UBE come from the caller
    got2, _ = gpu_search(ops, env, net, dict(root, value=fused["root_value"], value_epistemic_variance=fused["root_ube"]), uni)
    for name_, _, _ in _abi.SUMMARY_FIELDS + _abi.TREE_FIELDS:
        H.assert_same_bits(got2[name_], got[name_], name_)


# ----------------------------------------------------------------------------- 6. SelfplayRunner
RUNNER_OPTIONS = [(True, "search"), (False, "visit_counts"), (False, "improved_policy"), (True, "visit_counts")]


@pytest.mark.parametrize("device_noise", [False, True])
@pytest.mark.parametrize("uniform,sampling", RUNNER_OPTIONS)
def test_selfplay_runner_graph_equals_eager(ops, uniform, sampling, device_noise):
    import torch

    from e_alphazero_b200.selfplay import SelfplayRunner

    env = H.make_env("deepsea", seed=51, size=10)
    net = H.make_net(env, seed=52, fill=0.5)
    denv, dnet = H.device_env(env), H.device_net(net)
    B, T, seed = 256, 0.6, 5
    runs = {}
    for mode in ("eager", "graph"):
        r = SelfplayRunner(denv, dnet, B, 16, 0.97, exploration_beta=1.0, directed_exploration=True, mlp_mode=_abi.MLP_TENSOR,
                           use_graph=(mode == "graph"), fused_root=uniform, seed=seed, device_noise=device_noise,
                           uniform_prior=uniform, action_sampling=sampling, temperature=T)
        r.plan.workspace.zero_()  # both runners' draw counters start at 0
        if mode == "eager":
            r.draw_gumbel()  # the graph runner's warm-up step draws one root noise from the generator
        st = ops.env_init(denv, B)
        traj = torch.zeros((10, B, 4), dtype=torch.int32, device="cuda")
        acts = []
        for step in range(10):
            st, out = r.step(st)
            r.trajectory(st, out, traj[step])
            acts.append(host(out.action).copy())
            if mode == "eager" and device_noise and sampling != "search":  # the draw from the search's own output with the kernel's noise
                w = host(weights_of(r.plan.out, SelfplayRunner.ACTION_SAMPLING[sampling]))
                H.assert_same_bits(acts[-1], SO.sample_actions(w, SO.stream_gumbel(seed, step, B, 2), T), f"step {step} action")
        runs[mode] = (np.stack(acts), host(traj), {k: host(v).copy() for k, v in st.items()})
    (ae, te, se), (ag, tg, sg) = runs["eager"], runs["graph"]
    H.assert_same_bits(ae, ag, "actions")
    H.assert_same_bits(te, tg, "trajectory")
    assert (te[:, :, 0] == ae).all()  # the records hold the played actions
    for k in se:
        H.assert_same_bits(se[k], sg[k], k)


def test_selfplay_runner_sample_noise_given(ops):
    """sample_gumbel= passed to step() is the noise of the draw, in the graph as in eager mode."""
    import torch

    from e_alphazero_b200.selfplay import SelfplayRunner

    env = H.make_env("subleq", seed=61, word_size=16)
    net = H.make_net(env, seed=62, fill=0.5)
    denv, dnet = H.device_env(env), H.device_net(net)
    B = 64
    tasks = torch.ones(B, dtype=torch.int32, device="cuda")
    gen = np.random.default_rng(63)
    noise = [(H.to_device(gen.gumbel(size=(B, 16)).astype(np.float32)), H.to_device(gen.gumbel(size=(B, 16)).astype(np.float32))) for _ in range(4)]
    runs = {}
    for mode in ("eager", "graph"):
        r = SelfplayRunner(denv, dnet, B, 12, 0.97, mlp_mode=_abi.MLP_TENSOR, use_graph=(mode == "graph"), action_sampling="improved_policy", temperature=1.5)
        st = ops.env_init(denv, B, task_ids=tasks)
        acts = []
        for g, s in noise:
            st, out = r.step(st, gumbel=g, task_ids=tasks, sample_gumbel=s)
            acts.append(host(out.action).copy())
            w = host(r.plan.out["action_weights"])
            H.assert_same_bits(acts[-1], SO.sample_actions(w, host(s), 1.5), f"{mode} action")
        runs[mode] = np.stack(acts)
    H.assert_same_bits(runs["eager"], runs["graph"], "actions")


# ----------------------------------------------------------------------------- 7. argument errors
def test_argument_errors(ops):
    from e_alphazero_b200.selfplay import SelfplayRunner

    env, net, root = case("deepsea10")
    bad = [dict(flags=_abi.SEARCH_DEFAULT_FLAGS | _abi.FLAG_PUCT, root_prior=_abi.ROOT_PRIOR_UNIFORM),
           dict(flags=_abi.SEARCH_DEFAULT_FLAGS | _abi.FLAG_PUCT, action_sampling=_abi.ACTION_VISITS),
           dict(root_prior=2), dict(root_prior=-1), dict(action_sampling=3), dict(action_sampling=-1),
           dict(action_sampling=_abi.ACTION_VISITS, temperature=0.0), dict(action_sampling=_abi.ACTION_IMPROVED, temperature=-1.0),
           dict(action_sampling=_abi.ACTION_VISITS, temperature=float("nan")), dict(action_sampling=_abi.ACTION_VISITS, temperature=float("inf"))]
    for kw in bad:
        with pytest.raises(ops.EazError):
            gpu_search(ops, env, net, root, _abi.default_search_config(batch=64, num_simulations=8, **kw))
    # the temperature is read only while sampling
    gpu_search(ops, env, net, root, _abi.default_search_config(batch=64, num_simulations=8, temperature=0.0))
    with pytest.raises(ValueError):
        SelfplayRunner(H.device_env(env), H.device_net(net), 64, 8, 0.97, action_sampling="visits")
