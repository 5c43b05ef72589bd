"""A whole scan into the prioritised replay ring in one call (csrc/replay.cu: eaz_replay_add_sequence) against what it replaces: T'
add() calls of the same rows on a twin ring, and T' add_step calls at the header's cursor in the CPU oracle of the sum tree
(tests/priority_oracle.c).  The ring states, the rewards, every byte of the tree buffer and the host cursor and length must agree bit for
bit, from every ring state and for sequences shorter and longer than the ring.  Also: a SelfplayRunner scan and the selfplay() drop-in
into the ring, ops.replay_add_sequence under CUDA-graph replay, and the XLA handler EazReplayAddSequence through tests/xla_ffi_stub/."""
import numpy as np
import pytest

from e_alphazero_b200 import _abi
from tests import helpers as H
from tests import priority_oracle as P

pytestmark = pytest.mark.gpu

ENVS = {"deepsea30": ("deepsea", dict(size=30)), "subleq16": ("subleq", dict(word_size=16)),
        "subleq256_onehot": ("subleq", dict(word_size=256, binary=False))}


@pytest.fixture(scope="module")
def torch():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def host(t):
    return t.detach().cpu().numpy()


def step_rows(torch, env, denv, B, n, seed):
    """n consecutive auto-reset steps of random play from random states: a list of n state dicts (fresh tensors)"""
    from e_alphazero_b200 import ops

    rng = np.random.default_rng(seed)
    cur = ops.state_to_device(denv, H.random_states(env, B, seed=seed))
    rows = []
    for _ in range(n):
        cur = ops.env_step(denv, cur, H.to_device(rng.integers(0, env.num_actions, B).astype(np.int32)), auto_reset=True,
                           task_ids=rng.integers(1, 4, B).astype(np.int32) if env.kind == _abi.ENV_SUBLEQ else None)
        rows.append(cur)
    return rows


def stacked(torch, rows):
    """state dicts of one step each -> leaves [T',B,...] (the selfplay() drop-in's layout)"""
    return {k: torch.stack([r[k] for r in rows]) for k in rows[0]} if rows else None


def clone_ring(ring):
    import copy

    twin = copy.copy(ring)
    twin.states, twin.rewards, twin.tree = ring.states.clone(), ring.rewards.clone(), ring.tree.clone()
    return twin


def assert_rings_equal(a, b, what):
    H.assert_same_bits(host(a.states), host(b.states), f"{what}: ring states")
    H.assert_same_bits(host(a.rewards).view(np.uint32), host(b.rewards).view(np.uint32), f"{what}: ring rewards")
    H.assert_same_bits(host(a.tree), host(b.tree), f"{what}: tree bytes")
    assert (a.cursor, a.length) == (b.cursor, b.length), (what, a.cursor, a.length, b.cursor, b.length)


def assert_same_after_sample_and_set(torch, seq, twin, buf, K, seed, what):
    """a sample and a set_priorities on both rings (and the oracle) keep them identical"""
    T, B = seq.T, seq.B
    a, b = seq.sample(K), twin.sample(K)
    torch.cuda.synchronize()
    for k in ("indices", "probabilities"):
        H.assert_same_bits(host(getattr(a, k)), host(getattr(b, k)), f"{what}: sample {k}")
    for k in a.compact:
        H.assert_same_bits(host(a.compact[k]), host(b.compact[k]), f"{what}: sample {k}")
    exp = P.sample(buf, T, B, K, host(seq.states), host(seq.rewards))
    H.assert_same_bits(host(a.indices), exp["indices"], f"{what}: sample indices vs oracle")
    rng = np.random.default_rng(seed)
    idx = np.concatenate([host(a.indices)[: K // 2], rng.integers(0, T * B, K // 2)]).astype(np.int32)
    pri = (10.0 ** rng.uniform(-2, 1, idx.size)).astype(np.float32)
    d_idx, d_pri = H.to_device(idx), H.to_device(pri)
    seq.set_priorities(d_idx, d_pri)
    twin.set_priorities(d_idx, d_pri)
    P.set_priorities(buf, T, B, idx, pri)
    torch.cuda.synchronize()
    assert_rings_equal(seq, twin, f"{what}: after sample + set_priorities")
    H.assert_same_bits(host(seq.tree), buf, f"{what}: tree vs oracle after sample + set_priorities")


CASES = [(e, 8, B) for e in ENVS for B in (40, 300)] + [("deepsea30", 64, 4096)]


@pytest.mark.parametrize("env_name,T,B", CASES, ids=[f"{e}-T{T}-B{B}" for e, T, B in CASES])
def test_add_sequence_equals_adds_and_oracle(torch, env_name, T, B):
    from e_alphazero_b200 import ops
    from e_alphazero_b200.replay import PrioritisedReplayRing

    kind, kw = ENVS[env_name]
    env = H.make_env(kind, seed=501, **kw)
    denv = H.device_env(env)
    alpha, seed = 0.6, 0xA11
    lengths = sorted({0, 1, 2, T - 1, T, T + 1, 2 * T + 3})
    pool = step_rows(torch, env, denv, B, 2 * T + 3, seed=502)
    starts = {"empty": 0, "length 1": 1, "partly filled": T // 2 + 1, "full, cursor 0": T, "full, cursor T-1": 2 * T - 1}
    prelude = step_rows(torch, env, denv, B, 2 * T - 1, seed=503)
    for si, (start, n_pre) in enumerate(starts.items()):
        base = PrioritisedReplayRing(denv, T, B, priority_exponent=alpha, seed=seed)
        buf = P.init(T, B, alpha, seed)
        for r in prelude[:n_pre]:
            base.add(r)
            P.add_step(buf, T, B, int(P.header(buf)["cursor"]))
        # priorities above 1 (max_priority moves, so new pairs enter with a weight other than 1), also on the empty ring
        rng = np.random.default_rng(504 + si)
        idx = rng.integers(0, T * B, 64).astype(np.int32)
        pri = rng.uniform(0.5, 4.0, 64).astype(np.float32)
        base.set_priorities(H.to_device(idx), H.to_device(pri))
        P.set_priorities(buf, T, B, idx, pri)
        torch.cuda.synchronize()
        H.assert_same_bits(host(base.tree), buf, f"{start}: prelude vs oracle")
        hdr = P.header(buf)
        assert (int(hdr["cursor"]), int(hdr["length"])) == (base.cursor, base.length)
        for n in lengths:
            what = f"{env_name} T={T} B={B} {start}, T'={n}"
            seq, twin, obuf = clone_ring(base), clone_ring(base), buf.copy()
            rows = pool[:n]
            if n % 2:  # the scan's wire format
                x = dict(compact=torch.stack([ops.env_compact(denv, r) for r in rows]), rewards=torch.stack([r["rewards"][:, 0] for r in rows]))
            else:  # state leaves with a leading time axis (compacted inside add_sequence)
                x = stacked(torch, rows) if n else {k: v.unsqueeze(0)[:0] for k, v in pool[0].items()}
            seq.add_sequence(x)
            for r in rows:
                twin.add(r)
                P.add_step(obuf, T, B, int(P.header(obuf)["cursor"]))
            torch.cuda.synchronize()
            assert_rings_equal(seq, twin, what)
            H.assert_same_bits(host(seq.tree), obuf, f"{what}: tree vs oracle")
            hdr = P.header(obuf)
            assert (int(hdr["cursor"]), int(hdr["length"])) == (seq.cursor, seq.length), what
            assert hdr["status"] == 0, what
            if seq.can_sample():
                assert_same_after_sample_and_set(torch, seq, twin, obuf, 256, n + 17 * si, what)
            # add() after add_sequence() continues at the same cursor on the host and the device
            seq.add(pool[-1])
            twin.add(pool[-1])
            torch.cuda.synchronize()
            assert_rings_equal(seq, twin, f"{what}: add() after add_sequence()")


def test_uniform_ring_add_sequence(torch):
    """CompactReplayRing.add_sequence copies the rows with torch: it equals T' add() calls, wrap-around and T' > T included"""
    from e_alphazero_b200.replay import CompactReplayRing

    env = H.make_env("subleq", seed=511, word_size=16)
    denv = H.device_env(env)
    T, B = 8, 300
    pool = step_rows(torch, env, denv, B, 2 * T + 3, seed=512)
    for pre in (0, 5):
        for n in (0, 1, T - 1, T + 1, 2 * T + 3):
            a, b = CompactReplayRing(denv, T, B), CompactReplayRing(denv, T, B)
            for r in pool[:pre]:
                a.add(r)
                b.add(r)
            a.add_sequence(stacked(torch, pool[:n]) if n else dict(compact=a.states[:0], rewards=a.rewards[:0]))
            for r in pool[:n]:
                b.add(r)
            torch.cuda.synchronize()
            H.assert_same_bits(host(a.states), host(b.states), f"pre={pre} T'={n}: states")
            H.assert_same_bits(host(a.rewards).view(np.uint32), host(b.rewards).view(np.uint32), f"pre={pre} T'={n}: rewards")
            assert (a.cursor, a.length) == (b.cursor, b.length)


def scan_runner(denv, dnet, B, n, mode, tasks=(1,)):
    from e_alphazero_b200.selfplay import SelfplayRunner

    return SelfplayRunner(denv, dnet, B, n, 0.97, exploration_beta=0.4, directed_exploration=True, mlp_mode=mode, fused_root=True, seed=77,
                          tasks=tasks)


@pytest.mark.parametrize("kind,kw,B,mode", [("deepsea", dict(size=30), 4096, _abi.MLP_TENSOR), ("subleq", dict(word_size=16), 8192, _abi.MLP_TENSOR)],
                         ids=["deepsea30-4096-tensor", "subleq16-8192-resets"])
def test_scan_into_ring(torch, kind, kw, B, mode):
    """SelfplayRunner.scan(T=8) twice into a 12-slot ring (the second scan wraps): ring.add_sequence(out.state) equals 8 add() calls of
    the decoded rows.  Subleq draws tasks 1-3, so envs reset mid-scan."""
    from e_alphazero_b200 import ops
    from e_alphazero_b200.replay import PrioritisedReplayRing

    env = H.make_env(kind, seed=521, **kw)
    denv = H.device_env(env)
    net = H.make_net(env, seed=522, fill=0.5)
    r = scan_runner(denv, H.device_net(net), B, 16, mode, tasks=(1, 2, 3) if kind == "subleq" else (1,))
    tasks = H.to_device(np.random.default_rng(523).integers(1, 4, B).astype(np.int32)) if kind == "subleq" else None
    states = ops.env_init(denv, B, task_ids=tasks)
    T_ring, T = 12, 8
    seq = PrioritisedReplayRing(denv, T_ring, B, priority_exponent=0.6, seed=5)
    twin = PrioritisedReplayRing(denv, T_ring, B, priority_exponent=0.6, seed=5)
    zero_steps = 0
    for scan in range(2):
        _, out = r.scan(states, T)
        seq.add_sequence(out.state)
        for t in range(T):
            twin.add(ops.env_uncompact(denv, out.state["compact"][t], out.state["rewards"][t]))
        torch.cuda.synchronize()
        assert_rings_equal(seq, twin, f"{kind} scan {scan}")
        zero_steps += int((host(ops.env_uncompact(denv, out.state["compact"].reshape(T * B, -1))["step_count"]) == 0).sum())
    if kind == "subleq":  # Subleq-16 episodes end within ws - 3 = 13 steps: the 16 steps reset every env at least once
        assert zero_steps >= B, zero_steps


def test_selfplay_drop_in_state_into_ring(torch):
    """The selfplay() drop-in's stacked pgx State [T,B,...] into the ring: one add_sequence equals T add() calls of its rows."""
    from types import SimpleNamespace

    from e_alphazero_b200 import pgx
    from e_alphazero_b200.replay import PrioritisedReplayRing
    from e_alphazero_b200.selfplay import selfplay

    env = H.make_env("deepsea", seed=531, size=10)
    dnet = H.device_net(H.make_net(env, seed=532, fill=0.5))
    B, T = 48, 8
    penv = pgx.DeepSea(10, env.action_map)
    config = SimpleNamespace(selfplay_steps=T, selfplay_simulations_per_step=16, discount=0.97, exploration_beta=0.3, directed_exploration=True,
                             rescale_q_values_in_search=True)
    _, out = selfplay(dnet, config, SimpleNamespace(env=penv), penv.init(batch_size=B), 7)
    seq = PrioritisedReplayRing(penv.spec, 6, B, priority_exponent=0.6, seed=1)
    twin = PrioritisedReplayRing(penv.spec, 6, B, priority_exponent=0.6, seed=1)
    seq.add_sequence(out.state)
    for t in range(T):
        twin.add({k: v[t] for k, v in out.state.leaves.items()})
    torch.cuda.synchronize()
    assert_rings_equal(seq, twin, "selfplay() State")


def test_add_sequence_under_graph_capture(torch):
    """ops.replay_add_sequence captured ONCE and replayed T + 2 times with new contents appends at the advancing device cursor, as the
    eager calls do, and matches the oracle."""
    from e_alphazero_b200 import ops

    env = H.make_env("subleq", seed=541, word_size=16)
    denv = H.device_env(env)
    T, B, n, alpha, seed = 8, 300, 3, 0.6, 4
    S = denv.compact_bytes

    def new_ring():
        rs = torch.zeros((T, B, S), dtype=torch.uint8, device="cuda")
        rr = torch.zeros((T, B), dtype=torch.float32, device="cuda")
        tree = torch.zeros(ops.priority_tree_bytes(T, B), dtype=torch.uint8, device="cuda")
        ops.priority_init(tree, T, B, alpha, seed)
        return rs, rr, tree

    pool = step_rows(torch, env, denv, B, n * (T + 3), seed=542)
    seqs = [(torch.stack([ops.env_compact(denv, r) for r in pool[n * i:n * i + n]]),
             torch.stack([r["rewards"][:, 0] for r in pool[n * i:n * i + n]])) for i in range(T + 3)]
    static_c, static_r = seqs[0][0].clone(), seqs[0][1].clone()
    ops.replay_add_sequence(denv, static_c, static_r, *new_ring())  # loads the kernels outside the capture
    graph_ring, eager_ring = new_ring(), new_ring()
    buf = P.init(T, B, alpha, seed)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g):
            ops.replay_add_sequence(denv, static_c, static_r, *graph_ring)
    torch.cuda.current_stream().wait_stream(side)
    for rep in range(T + 2):
        c, r = seqs[rep + 1]
        static_c.copy_(c)
        static_r.copy_(r)
        g.replay()
        ops.replay_add_sequence(denv, c, r, *eager_ring)
        for _ in range(n):
            P.add_step(buf, T, B, int(P.header(buf)["cursor"]))
        torch.cuda.synchronize()
        for a, b, name in zip(graph_ring, eager_ring, ("ring_states", "ring_rewards", "tree")):
            H.assert_same_bits(host(a).view(np.uint8), host(b).view(np.uint8), f"replay {rep}: {name}")
        H.assert_same_bits(host(graph_ring[2]), buf, f"replay {rep}: tree vs oracle")
        for j in range(n):
            slot = (n * rep + j) % T
            H.assert_same_bits(host(graph_ring[0][slot]), host(c[j]), f"replay {rep}: row {slot}")
    hdr = P.header(host(graph_ring[2]))
    assert hdr["cursor"] == n * (T + 2) % T and hdr["length"] == T and hdr["status"] == 0


@pytest.mark.parametrize("env_name,B", [("deepsea30", 100), ("subleq16", 300), ("subleq256_onehot", 40)])
def test_xla_handler_against_ring_and_oracle(torch, env_name, B):
    """EazReplayAddSequence through the XLA-FFI stand-in, aliased and not aliased, against the torch ring and the oracle"""
    from e_alphazero_b200 import ops
    from e_alphazero_b200.replay import PrioritisedReplayRing
    from tests.xla_ffi_stub import harness as X

    lib = X.load()
    kind, kw = ENVS[env_name]
    env = H.make_env(kind, seed=551, **kw)
    denv = H.device_env(env)
    T, alpha, seed = 8, 0.6, 0x5EED
    S = denv.compact_bytes
    attrs = dict(env_kind=env.kind, size=env.size if env.kind == _abi.ENV_DEEPSEA else 0, word_size=env.word_size,
                 binary_encoding=int(env.binary_encoding), reward_fn=int(env.reward_fn))
    stream = torch.cuda.current_stream().cuda_stream
    amap = denv.action_map if denv.action_map is not None else torch.zeros(1, dtype=torch.uint8, device="cuda")
    rs = torch.zeros((T, B, S), dtype=torch.uint8, device="cuda")
    rr = torch.zeros((T, B), dtype=torch.float32, device="cuda")
    tree = torch.zeros(ops.priority_tree_bytes(T, B), dtype=torch.uint8, device="cuda")
    rc, msg = X.call(lib, "EazReplayInit", [], [X.tbuf(rs), X.tbuf(rr), X.tbuf(tree)], dict(T=T, B=B, priority_exponent=alpha, seed=seed), stream)
    assert rc == 0, msg
    ring = PrioritisedReplayRing(denv, T, B, priority_exponent=alpha, seed=seed)
    buf = P.init(T, B, alpha, seed)
    lengths = (3, 0, 1, T + 1, 2, T - 1, 2 * T + 3)
    pool = step_rows(torch, env, denv, B, sum(lengths), seed=552)
    at = 0
    for i, n in enumerate(lengths):
        rows = pool[at:at + n]
        assert len(rows) == n
        at += n
        compact = torch.stack([ops.env_compact(denv, r) for r in rows]) if n else torch.zeros((0, B, S), dtype=torch.uint8, device="cuda")
        rewards = torch.stack([r["rewards"][:, 0] for r in rows]) if n else torch.zeros((0, B), dtype=torch.float32, device="cuda")
        args = [X.tbuf(t) for t in (amap, rs, rr, tree, compact, rewards)]
        if i % 2:  # functional form: fresh results, the inputs stay as they were
            rs2, rr2, tree2 = torch.full_like(rs, 0x5A), torch.full_like(rr, -1.0), torch.full_like(tree, 0x77)
            ins = [host(rs).copy(), host(rr).copy(), host(tree).copy()]
            rc, msg = X.call(lib, "EazReplayAddSequence", args, [X.tbuf(rs2), X.tbuf(rr2), X.tbuf(tree2)], attrs, stream)
            assert rc == 0, msg
            torch.cuda.synchronize()
            for a, b, name in zip(ins, (rs, rr, tree), ("ring_states", "ring_rewards", "tree")):
                H.assert_same_bits(host(b).view(np.uint8), a.view(np.uint8), f"non-aliased call {i} leaves {name} alone")
            rs, rr, tree = rs2, rr2, tree2
        else:
            rc, msg = X.call(lib, "EazReplayAddSequence", args, [X.tbuf(rs), X.tbuf(rr), X.tbuf(tree)], attrs, stream)
            assert rc == 0, msg
        ring.add_sequence(dict(compact=compact, rewards=rewards))
        for _ in range(n):
            P.add_step(buf, T, B, int(P.header(buf)["cursor"]))
        torch.cuda.synchronize()
        what = f"{env_name} call {i} (T'={n})"
        H.assert_same_bits(host(rs), host(ring.states), f"{what}: ring_states")
        H.assert_same_bits(host(rr).view(np.uint32), host(ring.rewards).view(np.uint32), f"{what}: ring_rewards")
        H.assert_same_bits(host(tree), host(ring.tree), f"{what}: tree vs PrioritisedReplayRing")
        H.assert_same_bits(host(tree), buf, f"{what}: tree vs oracle")
