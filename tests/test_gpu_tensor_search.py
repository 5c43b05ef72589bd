"""mlp_mode=TENSOR search across its configuration: the persistent DeepSea kernel (psearch.cuh: ds_search_kernel) under every
search flag and at its cold paths, the fused root, PUCT, and the layer-1 producers of mlp_tensor_kernel over word size x encoding.

Every case applies the two checks of test_gpu_parity.test_search_tensor_mode:
  (a) every expanded node's network outputs against the fp32 oracle network (rtol 1e-5, atol 2e-6);
  (b) the oracle search replayed with the GPU's own per-node network outputs reproduces every tree array bit for bit;
and asserts that it took the code path it is meant to test, so that an eligibility change cannot turn it into a silent no-op.

With EAZ_NO_PERSISTENT set (read once per process by the library) the DeepSea cases run the launch chain
(mlp_gather_kernel + tree_step*_kernel) instead; test_launch_chain_subprocess re-runs them that way."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from e_alphazero_b200 import _abi
from oracle import oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu

NO_PERSISTENT = os.environ.get("EAZ_NO_PERSISTENT") is not None
RTOL, ATOL = 1e-5, 2e-6


@pytest.fixture(scope="module")
def ops():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from e_alphazero_b200 import ops as _ops

    return _ops


def host(t):
    return t.detach().cpu().numpy()


# ----------------------------------------------------------------------------- shared checks
def tensor_search(ops, env, net, root, cfg_kw, fused_root=False):
    """One TENSOR-mode search with the tree exported; returns (host outputs, plan)."""
    B = root["gumbel"].shape[0]
    denv, dnet = H.device_env(env), H.device_net(net)
    plan = ops.SearchPlan(_abi.default_search_config(batch=B, mlp_mode=_abi.MLP_TENSOR, **cfg_kw), denv, dnet, want_tree=True)
    droot = H.device_root(env, denv, root)
    if fused_root:
        for k in ("prior_logits", "value", "value_epistemic_variance"):
            del droot[k]
    got = {k: host(v).copy() for k, v in plan.run(droot).items()}
    return got, plan


def launches(ops, plan, n):
    cfg = _abi.EazSearchConfig.from_buffer_copy(plan.cfg)
    cfg.num_simulations = n
    return ops.load().eaz_search_num_launches(C.byref(cfg), C.byref(plan.env.struct()))


def ran_persistent(ops, plan):
    """ds_search_kernel runs all simulations in one launch: the launch count does not grow with num_simulations.  (Eligibility only
    shrinks as n grows, so n and n - 1 agree exactly when n is persistent.)"""
    n = plan.cfg.num_simulations
    assert n >= 2
    return plan.num_launches == launches(ops, plan, n - 1)


def assert_path(ops, plan, persistent):
    expect = persistent and not NO_PERSISTENT
    assert ran_persistent(ops, plan) == expect, f"expected {'ds_search_kernel' if expect else 'the launch chain'} (num_launches {plan.num_launches})"


def node_depths(parents):
    """Depth of every node from the exported parent indices (-1 for the root and for slots never expanded)."""
    B, N = parents.shape
    d = np.full((B, N), -1, np.int64)
    d[:, 0] = 0
    rows = np.arange(B)
    for i in range(1, N):
        p = parents[:, i]
        d[:, i] = np.where(p >= 0, d[rows, np.maximum(p, 0)] + 1, -1)
    return d


def reference_outputs(env, net, st, exploration):
    """The compared quantities of check (a) from the fp32 oracle network: max-subtracted logits, value and UBE (0 at terminal states)."""
    ev = O.mlp_forward_states(net, env, st)
    return outputs_of(ev, st, exploration)


def outputs_of(ev, st, exploration):
    lg = ev["explore_logits"] if exploration else ev["exploit_logits"]
    term = st["terminated"].astype(bool)
    return lg - lg.max(1, keepdims=True), np.where(term, 0, ev["value"]), np.where(term, 0, ev["ube"])


def check_network(env, net, got, exploration):
    """(a) every expanded node's outputs against the fp32 oracle network; returns the nodes' states.  (Under a max_depth cut-off a
    simulation may re-expand an existing leaf instead of adding node i + 1: such slots stay empty, with no visits, and are skipped.)"""
    B, N, A = got["children_prior_logits"].shape
    used = got["node_visits"][:, 1:].reshape(-1) > 0
    st = H.uncompact(env, got["embeddings"][:, 1:].reshape(B * (N - 1), -1)[used])
    lg, v, u = reference_outputs(env, net, st, exploration)
    np.testing.assert_allclose(got["children_prior_logits"][:, 1:].reshape(-1, A)[used], lg, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(got["raw_values"][:, 1:].reshape(-1)[used], v, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(got["raw_values_epistemic_variance"][:, 1:].reshape(-1)[used], u, rtol=RTOL, atol=ATOL)
    return st


def check_replay(env, root, got, cfg_kw):
    """(b) the oracle search on the GPU's own per-node network outputs: the same tree, bit for bit."""
    replay = dict(states=got["embeddings"], logits=got["children_prior_logits"], value=got["raw_values"], var=got["raw_values_epistemic_variance"])
    exp = O.search(_abi.default_search_config(**cfg_kw), env, None, root, want_tree=True, replay=replay)
    assert exp["replay_misses"] == 0
    for name, _, _ in _abi.SUMMARY_FIELDS + _abi.TREE_FIELDS:
        H.assert_same_bits(got[name], exp[name], name)
    n = cfg_kw["num_simulations"]
    assert (got["node_visits"][:, 0] == n + 1).all()
    if not cfg_kw.get("max_depth"):  # every simulation adds a node: check (a) saw all of them
        assert (got["node_visits"][:, 1:] > 0).all()


def check_both(env, net, root, got, cfg_kw):
    check_network(env, net, got, cfg_kw.get("exploration", 0))
    check_replay(env, root, got, cfg_kw)


# ----------------------------------------------------------------------------- the persistent DeepSea kernel across the configuration
def test_persistent_switch_combinations(ops):
    """All 16 BETA_INTERIOR / BETA_RAW / BETA_FINAL / BACKUP_STD combinations x mixed value on / off (rescale_values varied) inside
    ds_search_kernel: its own copies of the backward recurrences (std backup) and the refresh.  The switches must not be dead."""
    env = H.make_env("deepsea", seed=31, size=8)
    net = H.make_net(env, seed=32, fill=0.5)
    B, n = 96, 24
    root = H.make_root(env, net, B, seed=33, beta_max=2.0, invalid_frac=0.15)
    seen = set()
    for combo in range(16):
        flags = ((_abi.FLAG_BETA_INTERIOR if combo & 1 else 0) | (_abi.FLAG_BETA_RAW if combo & 2 else 0) |
                 (_abi.FLAG_BETA_FINAL if combo & 4 else 0) | (_abi.FLAG_BACKUP_STD if combo & 8 else 0))
        for mixed in (1, 0):
            cfg_kw = dict(num_simulations=n, discount=0.97, flags=flags, use_mixed_value=mixed, rescale_values=combo & 1)
            got, plan = tensor_search(ops, env, net, root, cfg_kw)
            assert_path(ops, plan, persistent=True)
            check_both(env, net, root, got, cfg_kw)
            if mixed:
                seen.add((got["node_visits"].tobytes(), got["node_values_epistemic_variance"].tobytes(), got["action_weights"].tobytes()))
    assert len(seen) >= 12, f"only {len(seen)} distinct results over 16 switch combinations"


PERSISTENT_CONFIGS = {
    "two_players": (10, dict(num_simulations=24, discount=0.997, two_players_game=1), dict(beta_max=1.0)),
    "gumbel_scale_0": (10, dict(num_simulations=24, discount=0.997, gumbel_scale=0.0), dict(beta_max=1.0)),
    "one_considered_action": (10, dict(num_simulations=24, discount=0.997, max_num_considered_actions=1), dict(beta_max=1.0)),
    "discount_0.9": (10, dict(num_simulations=24, discount=0.9), dict(beta_max=1.0)),
    "discount_1": (10, dict(num_simulations=24, discount=1.0), dict(beta_max=1.0)),
    "explore_head": (10, dict(num_simulations=24, discount=0.997, exploration=1), dict(beta_max=1.0)),
    "beta_0": (10, dict(num_simulations=24, discount=0.997), dict(beta_max=0.0)),
    "beta_2_std_two_players": (8, dict(num_simulations=24, discount=0.9, two_players_game=1, flags=_abi.FLAG_BACKUP_STD | _abi.FLAG_BETA_FINAL),
                               dict(beta_max=2.0)),
    "invalid_root_actions": (10, dict(num_simulations=24, discount=0.997), dict(beta_max=1.0, invalid_frac=0.3)),  # row 0: all invalid
    # a descent cut off at depth 3 re-expands an existing node: that simulation takes the DIRECT step and re-synchronises the caches
    "max_depth_3": (6, dict(num_simulations=40, discount=0.997, max_depth=3), dict(beta_max=0.5)),
}


@pytest.mark.parametrize("name", list(PERSISTENT_CONFIGS))
def test_persistent_search_config(ops, name):
    size, cfg_kw, root_kw = PERSISTENT_CONFIGS[name]
    env = H.make_env("deepsea", seed=41, size=size)
    net = H.make_net(env, seed=42, fill=0.5)
    root = H.make_root(env, net, 96, seed=43, **root_kw)
    got, plan = tensor_search(ops, env, net, root, cfg_kw)
    assert_path(ops, plan, persistent=True)
    check_both(env, net, root, got, cfg_kw)
    if "max_depth" in cfg_kw:
        d = node_depths(got["parents"])
        assert d.max() == cfg_kw["max_depth"]
        assert (got["node_visits"][:, 1:] == 0).any(), "no simulation re-expanded a leaf at the depth cut-off"
    if root_kw.get("invalid_frac"):
        assert root["invalid_actions"][0].all() and got["action"][0] == 0  # masked_argmax of an all-invalid row


# ----------------------------------------------------------------------------- cold paths of the persistent kernel
def test_persistent_deep_paths(ops):
    """A policy head that strongly prefers action 0 grows chains: paths longer than the staging area (kNodes - 1 = 23 edges) take
    the DIRECT step, and levels past the 32 that s_back mirrors are read from the workspace only."""
    env = H.make_env("deepsea", seed=51, size=48)
    net = H.make_net(env, seed=52, fill=0.5)
    for h in (_abi.HEAD_EXPLOIT, _abi.HEAD_EXPLORE):
        net.b[h][2][:] = np.array([6.0, -6.0], np.float32)
    cfg_kw = dict(num_simulations=128, discount=0.997)
    root = H.make_root(env, net, 64, seed=53, beta_max=1.0)
    got, plan = tensor_search(ops, env, net, root, cfg_kw)
    assert_path(ops, plan, persistent=True)
    check_both(env, net, root, got, cfg_kw)
    d = node_depths(got["parents"])
    assert (d > 24).any() and (d > 33).any(), f"deepest node at depth {d.max()}"


@pytest.mark.parametrize("size", [128, 130])
def test_persistent_action_map_boundary(ops, size):
    """The action map is mirrored in shared memory up to N * N = 16384 bytes (N = 128) and read from global memory above.  (129 is
    not a valid network input: the observation is hashed in groups of 4 elements, so N * N must be a multiple of 4.)"""
    assert (size * size <= AMAP_MAX_BYTES) == (size == 128)
    env = H.make_env("deepsea", seed=61, size=size)
    net = H.make_net(env, seed=62, fill=0.5)
    cfg_kw = dict(num_simulations=24, discount=0.997)
    root = H.make_root(env, net, 48, seed=63, beta_max=1.0)
    got, plan = tensor_search(ops, env, net, root, cfg_kw)
    assert_path(ops, plan, persistent=True)
    check_both(env, net, root, got, cfg_kw)


def probe_persistent_limit(ops, plan):
    """Largest num_simulations that still runs in ds_search_kernel for this plan's shape (its shared-memory caches grow with n)."""
    def persistent(n):
        return launches(ops, plan, n) == launches(ops, plan, n - 1)

    lo, hi = 2, 4094
    if not persistent(lo):
        return None
    while lo < hi:  # invariant: persistent(lo)
        mid = (lo + hi + 1) // 2
        if persistent(mid):
            lo = mid
        else:
            hi = mid - 1
    return lo


def test_persistent_shared_memory_boundary(ops):
    """DeepSea-30: the largest n whose trees fit the kernel's shared-memory caches runs persistent, n + 1 falls back to the launch
    chain; both replay bit for bit."""
    env = H.make_env("deepsea", seed=71, size=30)
    net = H.make_net(env, seed=72, fill=0.5)
    B = 16
    root = H.make_root(env, net, B, seed=73, beta_max=1.0)
    denv, dnet = H.device_env(env), H.device_net(net)
    probe = ops.SearchPlan(_abi.default_search_config(batch=B, num_simulations=8, mlp_mode=_abi.MLP_TENSOR), denv, dnet)
    limit = probe_persistent_limit(ops, probe)
    if NO_PERSISTENT:
        assert limit is None
        limit = 300  # (no boundary on the chain: run the same shapes)
    else:
        assert limit is not None and 64 < limit < 4094, limit
    for n, persistent in ((limit, True), (limit + 1, False)):
        cfg_kw = dict(num_simulations=n, discount=0.997)
        got, plan = tensor_search(ops, env, net, root, cfg_kw)
        assert_path(ops, plan, persistent=persistent)
        check_both(env, net, root, got, cfg_kw)


def test_launch_chain_subprocess():
    """The test_persistent_* cases once more with EAZ_NO_PERSISTENT=1 (read once per process, hence the subprocess): they then hold
    mlp_gather_kernel + tree_step*_kernel in TENSOR mode, and their path assertions expect the chain."""
    if NO_PERSISTENT:
        pytest.skip("this process already runs the launch chain")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, EAZ_NO_PERSISTENT="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k", "persistent", "-p", "no:cacheprovider"],
                       cwd=root, env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and "failed" not in r.stdout


# ----------------------------------------------------------------------------- fused root and PUCT
@pytest.mark.parametrize("kind,kw,B,cfg_kw,persistent", [
    ("deepsea", dict(size=30), 300, dict(num_simulations=32, discount=0.997, exploration=1), True),
    ("subleq", dict(word_size=16), 200, dict(num_simulations=16, discount=0.97), False),
])
def test_fused_root_tensor(ops, kind, kw, B, cfg_kw, persistent):
    """Root inputs NULL: the library evaluates the root network itself (mlp_gather_kernel / mlp_tensor_kernel) before root_init."""
    env = H.make_env(kind, seed=81, **kw)
    net = H.make_net(env, seed=82, fill=0.5)
    st = H.random_states(env, B, seed=83)
    rng = np.random.default_rng(84)
    root = dict(beta=np.linspace(0, 1, B).astype(np.float32), embedding=st, gumbel=rng.gumbel(size=(B, env.num_actions)).astype(np.float32),
                prior_logits=np.zeros((B, env.num_actions), np.float32), value=np.zeros(B, np.float32), value_epistemic_variance=np.zeros(B, np.float32))
    got, plan = tensor_search(ops, env, net, root, cfg_kw, fused_root=True)
    assert_path(ops, plan, persistent=persistent)
    # the root's network outputs against the fp32 oracle network
    lg, v, u = reference_outputs(env, net, st, cfg_kw.get("exploration", 0))
    ev = O.mlp_forward_states(net, env, st)  # (root_value / root_ube are the raw outputs: not zeroed at terminal roots)
    np.testing.assert_allclose(got["children_prior_logits"][:, 0], lg, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(got["root_value"], ev["value"], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(got["root_ube"], ev["ube"], rtol=RTOL, atol=ATOL)
    check_network(env, net, got, cfg_kw.get("exploration", 0))
    # The replay's root is the GPU's own root outputs.  Its logits are the exported max-subtracted ones: root_init subtracts the
    # maximum again, which is exactly 0, so x - 0 == x reproduces the GPU's root_init bit for bit.
    rroot = dict(root, prior_logits=got["children_prior_logits"][:, 0].copy(), value=got["root_value"], value_epistemic_variance=got["root_ube"])
    assert (rroot["prior_logits"].max(1) == 0).all()
    H.assert_same_bits(got["raw_values"][:, 0], got["root_value"], "root raw value")
    check_replay(env, rroot, got, cfg_kw)


@pytest.mark.parametrize("kind,kw,B,cfg_kw,root_kw", [
    ("deepsea", dict(size=10), 64, dict(num_simulations=32, discount=0.997), dict(beta_max=1.0, invalid_frac=0.2)),  # staged PUCT (A <= 4)
    ("subleq", dict(word_size=16), 40, dict(num_simulations=24, discount=0.97, pb_c_init=2.0), dict(beta_max=1.0)),
])
def test_puct_tensor(ops, kind, kw, B, cfg_kw, root_kw):
    """EAZ_FLAG_PUCT is not eligible for the persistent kernel: the launch chain with mlp_gather_kernel (DeepSea) / mlp_tensor_kernel."""
    env = H.make_env(kind, seed=91, **kw)
    net = H.make_net(env, seed=92, fill=0.5)
    root = H.make_root(env, net, B, seed=93, **root_kw)
    cfg_kw = dict(cfg_kw, flags=_abi.SEARCH_DEFAULT_FLAGS | _abi.FLAG_PUCT)
    got, plan = tensor_search(ops, env, net, root, cfg_kw)
    assert_path(ops, plan, persistent=False)
    check_both(env, net, root, got, cfg_kw)
    np.testing.assert_array_equal(got["action_weights"], got["visit_probs"])


# ----------------------------------------------------------------------------- mlp_tensor_kernel layer-1 producers
# constants of mlp_tensor.cu (kCK, kBitsWordsMax) and of its state staging (compact records of at most 64 bytes)
KCK, BITS_WORDS_MAX, STAGE_BYTES_MAX = 32, 40, 64
AMAP_MAX_BYTES = 16384  # psearch.cuh kAmapMax


def producer_path(env):
    """Which of mlp_tensor_kernel's layer-1 producers builds a Subleq row (mlp_tensor.cu, worker warps)."""
    k1pad = -(-env.obs_dim // KCK) * KCK
    cached = k1pad // 32 <= BITS_WORDS_MAX             # the row's bit-string lives in shared memory
    staged = cached and env.compact_bytes <= STAGE_BYTES_MAX  # the compact state is copied to shared memory first
    if not env.binary_encoding:
        return "one_hot_cached" if cached else "one_hot_uncached"
    if not cached:
        return "binary_uncached"
    if staged and env.word_size == 16 and env.obs_cols == 5:
        return "binary_ws16_pack"
    return "binary_staged_pack" if staged else "binary_cached_global"


PRODUCER_PATHS = {"binary_ws16_pack", "binary_staged_pack", "binary_cached_global", "binary_uncached", "one_hot_cached", "one_hot_uncached"}

# (word size, binary, B, n, expected D, expected k1pad, path)
PRODUCER_CASES = [
    (16, True, 64, 8, 240, 256, "binary_ws16_pack"),
    (17, True, 48, 8, 294, 320, "binary_staged_pack"),     # D not a multiple of 32
    (17, True, 128, 6, 294, 320, "binary_staged_pack"),    # exactly one row tile
    (17, True, 257, 4, 294, 320, "binary_staged_pack"),    # one row past two tiles
    (24, True, 40, 8, 336, 352, "binary_staged_pack"),     # compact_bytes == 64: still staged
    (25, True, 40, 8, 342, 352, "binary_cached_global"),   # first unstaged word size: state read from global memory
    (64, True, 24, 8, 672, 672, "binary_cached_global"),   # k1pad == D
    (128, True, 16, 8, 1280, 1280, "binary_cached_global"),  # bit cache exactly full
    (129, True, 16, 8, 1449, 1472, "binary_uncached"),     # first uncached binary, w = 9
    (16, False, 40, 8, 816, 832, "one_hot_cached"),        # the reference's experiment size
    (22, False, 24, 8, 1242, 1248, "one_hot_cached"),      # largest cached one-hot (39 words)
    (23, False, 24, 8, 1320, 1344, "one_hot_uncached"),    # first uncached one-hot
    (256, False, 4, 6, 74016, 74016, "one_hot_uncached"),  # 2313 layer-1 chunks
]


def test_producer_cases_cover_every_path():
    """The case list is derived from the kernel's constants: every producer class is covered, and each row is the class it claims."""
    seen = set()
    for ws, binary, _, _, D, k1pad, path in PRODUCER_CASES:
        env = O.Env.subleq(ws, binary)
        assert env.obs_dim == D and -(-D // KCK) * KCK == k1pad, (ws, binary)
        assert producer_path(env) == path, (ws, binary, producer_path(env))
        seen.add(path)
    assert seen == PRODUCER_PATHS
    assert O.Env.subleq(24, True).compact_bytes == STAGE_BYTES_MAX and O.Env.subleq(25, True).compact_bytes > STAGE_BYTES_MAX
    assert -(-O.Env.subleq(128, True).obs_dim // 32) == BITS_WORDS_MAX


def assert_comparison_sensitive(env, net, st, exploration, seed):
    """Flip one observation bit per row in the oracle's input: for most rows the reference moves by more than 100x the tolerance
    of check (a), so a dropped or misplaced input bit in a producer cannot pass it.  Logits and value only: the UBE output jumps
    whenever the flip lands in the hashed rows and changes the novelty bit, which would make the guard pass on its own."""
    rng = np.random.default_rng(seed)
    obs = O.env_observe(env, st).reshape(len(st["step_count"]), -1)
    M, D = obs.shape
    hd = env.hash_dim(net.hash_io)
    base = outputs_of(O.mlp_forward(net, obs, hd), st, exploration)
    flipped = obs.copy()
    flipped[np.arange(M), rng.integers(0, D, M)] ^= 1
    moved = outputs_of(O.mlp_forward(net, flipped, hd), st, exploration)
    score = np.zeros(M)
    for a, b in zip(base[:2], moved[:2]):
        r = np.abs(b - a) / (ATOL + RTOL * np.abs(a))
        score = np.maximum(score, r.reshape(M, -1).max(1))
    frac = float((score > 100).mean())
    assert frac > 0.5, f"only {frac:.2f} of the rows move by more than 100x the tolerance"


@pytest.mark.parametrize("ws,binary,B,n,D,k1pad,path", PRODUCER_CASES)
def test_subleq_layer1_producer(ops, ws, binary, B, n, D, k1pad, path):
    env = H.make_env("subleq", seed=101, word_size=ws, binary=binary)
    assert producer_path(env) == path
    net = H.make_net(env, seed=102, fill=0.5)
    root = H.make_root(env, net, B, seed=103, beta_max=1.0)
    cfg_kw = dict(num_simulations=n, discount=0.97, exploration=ws % 2)
    got, plan = tensor_search(ops, env, net, root, cfg_kw)
    assert_path(ops, plan, persistent=False)
    st = check_network(env, net, got, cfg_kw["exploration"])
    check_replay(env, root, got, cfg_kw)
    assert_comparison_sensitive(env, net, st, cfg_kw["exploration"], seed=ws)
