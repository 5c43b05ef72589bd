"""The prioritised replay ring as a JAX program drives it: the five replay handlers of csrc/xla_ffi_shim.cc, called through the
stand-in call frame of tests/xla_ffi_stub/ on device buffers, against the torch PrioritisedReplayRing fed the same inputs and the CPU
oracle of the sum tree (tests/priority_oracle.c), bit for bit.  Also: ops.replay_add (the device cursor) under CUDA-graph replay."""
import ctypes as C

import numpy as np
import pytest

from e_alphazero_b200 import _abi
from tests import helpers as H
from tests import priority_oracle as P

pytestmark = pytest.mark.gpu

LEAVES = {_abi.ENV_DEEPSEA: ["step_count", "rewards", "terminated", "truncated", "col"],
          _abi.ENV_SUBLEQ: ["step_count", "rewards", "terminated", "truncated", "memory", "task", "solved", "input_after", "output_after"]}


@pytest.fixture(scope="module")
def shim():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from tests.xla_ffi_stub import harness as X

    return X, X.load()


def host(t):
    return t.detach().cpu().numpy()


def env_attrs(env):
    return dict(env_kind=env.kind, size=env.size if env.kind == _abi.ENV_DEEPSEA else 0, word_size=env.word_size,
                binary_encoding=int(env.binary_encoding), reward_fn=int(env.reward_fn))


U32 = 8  # xla::ffi::DataType::U32 of the stand-in header (tests/xla_ffi_stub/xla/ffi/api/ffi.h)


def u32buf(X, ptr, *dims):
    return X.StubBuf(U32, len(dims), ptr, (C.c_int64 * 4)(*dims))


def oracle_add_at_cursor(buf, T, B):
    """eaz_replay_add's add_step in the oracle: add_step at the slot the header's cursor names"""
    P.add_step(buf, T, B, int(P.header(buf)["cursor"]))


def oracle_sample_keyed(buf, T, B, K, states, rewards, key):
    """the keyed sample in the oracle: its sample on a copy of the buffer whose header carries (seed, draw_ctr) = key, which by the
    contract draws what the keyed sample draws; `buf` itself is not touched"""
    tmp = buf.copy()
    hdr = tmp[:32].view(P.HEADER)
    hdr["seed"], hdr["draw_ctr"] = np.uint32(key[0]), np.uint32(key[1])
    return P.sample(tmp, T, B, K, states, rewards)


def lib_status(tree):
    """the sticky bits as eaz_priority_status (synchronising) reports them"""
    import torch

    from e_alphazero_b200 import _lib

    f = C.c_int32(-1)
    rc = _lib.load().eaz_priority_status(C.c_void_p(tree.data_ptr()), C.c_size_t(tree.numel()), C.c_void_p(torch.cuda.current_stream().cuda_stream),
                                         C.byref(f))
    assert rc in (0, _abi.EAZ_ERR_UNSUPPORTED)
    return f.value


@pytest.mark.parametrize("kind,kw,B", [("deepsea", dict(size=30), 100), ("subleq", dict(word_size=16), 300),
                                       ("subleq", dict(word_size=256, binary=False), 100)])
def test_replay_handlers_against_ring_and_oracle(shim, kind, kw, B):
    import torch

    from e_alphazero_b200 import ops
    from e_alphazero_b200.replay import PrioritisedReplayRing

    X, lib = shim
    env = H.make_env(kind, seed=81, **kw)
    denv = H.device_env(env)
    T, alpha, seed = 8, 0.6, 0x5EED
    S, N, TB = denv.compact_bytes, T * B, ops.priority_tree_bytes(T, B)
    fields = LEAVES[env.kind]
    attrs = env_attrs(env)
    stream = torch.cuda.current_stream().cuda_stream
    dev = "cuda"
    dummy = torch.zeros(1, dtype=torch.uint8, device=dev)
    amap = denv.action_map if denv.action_map is not None else dummy
    rng = np.random.default_rng(82)

    def call(handler, args, rets, at):
        rc, msg = X.call(lib, handler, args, rets, at, stream)
        assert rc == 0, f"{handler}: {msg}"

    # init: the results start as garbage and must come back zeroed / initialised
    rs = torch.full((T, B, S), 0xAB, dtype=torch.uint8, device=dev)
    rr = torch.full((T, B), float("nan"), dtype=torch.float32, device=dev)
    tree = torch.full((TB,), 0xCD, dtype=torch.uint8, device=dev)
    call("EazReplayInit", [], [X.tbuf(rs), X.tbuf(rr), X.tbuf(tree)], dict(T=T, B=B, priority_exponent=alpha, seed=seed))
    ring = PrioritisedReplayRing(denv, T, B, priority_exponent=alpha, seed=seed)
    buf = P.init(T, B, alpha, seed)

    def check(what):
        torch.cuda.synchronize()
        H.assert_same_bits(host(rs), host(ring.states), f"{what}: ring_states")
        H.assert_same_bits(host(rr), host(ring.rewards), f"{what}: ring_rewards")
        H.assert_same_bits(host(tree), host(ring.tree), f"{what}: tree vs PrioritisedReplayRing")
        H.assert_same_bits(host(tree), buf, f"{what}: tree vs oracle")

    check("init")

    def keyed_sample(K, key):
        key_d = torch.as_tensor(np.asarray(key, np.uint64).astype(np.uint32).view(np.int32)).to(dev)
        out = dict(indices=torch.full((K,), -7, dtype=torch.int32, device=dev), probabilities=torch.full((K,), float("nan"), device=dev))
        first, second = ops.alloc_state(denv, K), ops.alloc_state(denv, K)
        for st in (first, second):
            for v in st.values():
                v.fill_(-3 if v.dtype != torch.uint8 else 9)
        scratch = torch.full((2 * K * (S + 4) + 16,), 0xEE, dtype=torch.uint8, device=dev)
        rets = [out["indices"], out["probabilities"]] + [first[k] for k in fields] + [second[k] for k in fields] + [scratch]
        call("EazReplaySample", [X.tbuf(amap), X.tbuf(rs), X.tbuf(rr), X.tbuf(tree), u32buf(X, key_d.data_ptr(), 2)],
             [X.tbuf(t) for t in rets], dict(attrs, K=K))
        torch.cuda.synchronize()
        got = {k: host(v) for k, v in out.items()}
        got["first"], got["second"] = {k: host(v) for k, v in first.items()}, {k: host(v) for k, v in second.items()}
        sc = host(scratch)
        got["first_records"] = sc[8 * K:8 * K + K * S].reshape(K, S)
        got["second_records"] = sc[8 * K + K * S:8 * K + 2 * K * S].reshape(K, S)
        return got

    def check_sample(K, key, what):
        before, buf_before = host(tree).copy(), buf.copy()
        got = keyed_sample(K, key)
        exp = oracle_sample_keyed(buf, T, B, K, host(rs), host(rr), key)
        H.assert_same_bits(buf, buf_before, f"{what}: the oracle's keyed sample left its buffer alone")
        H.assert_same_bits(host(tree), before, f"{what}: tree bytes unchanged by the keyed sample")
        H.assert_same_bits(got["indices"], exp["indices"], f"{what}: indices")
        H.assert_same_bits(got["probabilities"], exp["probabilities"], f"{what}: probabilities")
        for side in ("first", "second"):
            H.assert_same_bits(got[side + "_records"], exp[side], f"{what}: {side} compact records")
            dec = H.uncompact(env, exp[side])
            for k in fields:
                e = exp[side + "_rewards"].reshape(K, 1) if k == "rewards" else dec[k]
                H.assert_same_bits(got[side][k], e.astype(got[side][k].dtype).reshape(got[side][k].shape), f"{what}: {side}.{k}")
        again = keyed_sample(K, key)
        for k in ("indices", "probabilities", "first_records", "second_records"):
            H.assert_same_bits(again[k], got[k], f"{what}: same key twice, {k}")
        H.assert_same_bits(host(tree), before, f"{what}: tree bytes unchanged by the second keyed sample")
        return got

    # a keyed sample of the empty tree: index 0, probability 0, and (unlike eaz_priority_sample) no EMPTY bit
    got = check_sample(37, (11, 12), "empty tree")
    assert (got["indices"] == 0).all() and (got["probabilities"] == 0).all()
    assert lib_status(tree) == 0

    # T + 3 adds (the ring wraps), each through the aliased handler; one of them without aliasing
    cur = ops.state_to_device(denv, H.random_states(env, B, seed=83))
    for step in range(T + 3):
        lv = [cur[k] for k in fields]
        if step == 2:  # functional form: fresh results, the inputs stay as they were
            rs2, rr2, tree2 = torch.full_like(rs, 0x5A), torch.full_like(rr, -1.0), torch.full_like(tree, 0x77)
            ins = [host(rs).copy(), host(rr).copy(), host(tree).copy()]
            call("EazReplayAdd", [X.tbuf(t) for t in [amap, rs, rr, tree] + lv], [X.tbuf(rs2), X.tbuf(rr2), X.tbuf(tree2)], attrs)
            torch.cuda.synchronize()
            for a, b, n in zip(ins, (rs, rr, tree), ("ring_states", "ring_rewards", "tree")):
                H.assert_same_bits(host(b), a, f"non-aliased add leaves {n} alone")
            rs, rr, tree = rs2, rr2, tree2
        else:
            call("EazReplayAdd", [X.tbuf(t) for t in [amap, rs, rr, tree] + lv], [X.tbuf(rs), X.tbuf(rr), X.tbuf(tree)], attrs)
        ring.add(cur)
        oracle_add_at_cursor(buf, T, B)
        check(f"add {step}")
        cur = ops.env_step(denv, cur, H.to_device(rng.integers(0, env.num_actions, B).astype(np.int32)), auto_reset=True,
                           task_ids=np.ones(B, np.int32) if kind == "subleq" else None)
    hdr = P.header(host(tree))
    assert hdr["cursor"] == (T + 3) % T and hdr["length"] == T

    # set_priorities: duplicates (the last wins), a stale index, a negative priority, an out-of-range index
    stale_row = (int(hdr["cursor"]) - 1) % T  # its pairs end at the slot written next: weight 0
    idx = np.concatenate([rng.integers(0, N, 200), [17, 17, 17], [stale_row * B + 3], [N + 5], [-2]]).astype(np.int32)
    pri = (10.0 ** rng.uniform(-3, 3, idx.size)).astype(np.float32)
    pri[rng.random(idx.size) < 0.1] = 0.0
    pri[-6:-3] = [0.5, 2.0, 7.0]
    pri[5] = -1.0
    d_idx, d_pri = H.to_device(idx), H.to_device(pri)
    call("EazReplaySetPriorities", [X.tbuf(d_idx), X.tbuf(d_pri), X.tbuf(tree)], [X.tbuf(tree)], dict(T=T, B=B))
    ring.set_priorities(d_idx, d_pri)
    P.set_priorities(buf, T, B, idx, pri)
    check("set_priorities")
    assert P.levels(host(tree), T, B)[0][stale_row * B + 3] == 0

    # status: the handler reports the bits eaz_priority_status reports
    flags = torch.full((1,), -1, dtype=torch.int32, device=dev)
    call("EazReplayStatus", [X.tbuf(tree)], [X.tbuf(flags)], {})
    torch.cuda.synchronize()
    expect = _abi.PRIORITY_BAD_PRIORITY | _abi.PRIORITY_BAD_INDEX
    assert int(host(flags)[0]) == lib_status(tree) == int(P.header(buf)["status"]) == expect
    flags.fill_(-1)
    ops.priority_status_async(tree, flags)
    torch.cuda.synchronize()
    assert int(host(flags)[0]) == expect

    # keyed samples; with key = (seed, draw_ctr) they equal eaz_priority_sample on the same tree
    for K in (1, 37, 4096):
        check_sample(K, (rng.integers(0, 2 ** 32), rng.integers(0, 2 ** 32)), f"K={K}")
        hdr = P.header(host(tree))
        key = (int(hdr["seed"]), int(hdr["draw_ctr"]))
        got = check_sample(K, key, f"K={K} header key")
        t2 = tree.clone()
        i2, p2 = torch.empty(K, dtype=torch.int32, device=dev), torch.empty(K, dtype=torch.float32, device=dev)
        f2, s2 = torch.empty((K, S), dtype=torch.uint8, device=dev), torch.empty((K, S), dtype=torch.uint8, device=dev)
        fr2, sr2 = torch.empty(K, device=dev), torch.empty(K, device=dev)
        ops.priority_sample(t2, T, B, i2, p2, rs, rr, f2, fr2, s2, sr2)
        torch.cuda.synchronize()
        H.assert_same_bits(got["indices"], host(i2), f"K={K}: keyed == eaz_priority_sample indices")
        H.assert_same_bits(got["probabilities"], host(p2), f"K={K}: keyed == eaz_priority_sample probabilities")
        H.assert_same_bits(got["first_records"], host(f2), f"K={K}: keyed == eaz_priority_sample first records")
        H.assert_same_bits(got["second_records"], host(s2), f"K={K}: keyed == eaz_priority_sample second records")
        H.assert_same_bits(got["first"]["rewards"].reshape(K), host(fr2), f"K={K}: keyed == eaz_priority_sample first rewards")
        H.assert_same_bits(got["second"]["rewards"].reshape(K), host(sr2), f"K={K}: keyed == eaz_priority_sample second rewards")
        assert P.header(host(t2))["draw_ctr"] == hdr["draw_ctr"] + 1
        # the C entry called directly (ops.priority_sample_keyed), indices and probabilities only
        key_d = torch.as_tensor(np.asarray(key, np.uint64).astype(np.uint32).view(np.int32)).to(dev)
        ops.priority_sample_keyed(tree, T, B, key_d, i2, p2)
        torch.cuda.synchronize()
        H.assert_same_bits(host(i2), got["indices"], f"K={K}: ops.priority_sample_keyed indices")
        H.assert_same_bits(host(p2), got["probabilities"], f"K={K}: ops.priority_sample_keyed probabilities")
    check("after sampling")
    assert P.header(host(tree))["draw_ctr"] == 0
    # and one more set after the samples, through the torch ring and the handler alike
    idx = rng.integers(0, N, 512).astype(np.int32)
    pri = rng.uniform(0, 3, 512).astype(np.float32)
    d_idx, d_pri = H.to_device(idx), H.to_device(pri)
    call("EazReplaySetPriorities", [X.tbuf(d_idx), X.tbuf(d_pri), X.tbuf(tree)], [X.tbuf(tree)], dict(T=T, B=B))
    ring.set_priorities(d_idx, d_pri)
    P.set_priorities(buf, T, B, idx, pri)
    check("second set_priorities")
    check_sample(4096, (5, 6), "after the second set")


def test_replay_add_under_graph_capture():
    """ops.replay_add captured ONCE and replayed T + 2 times with new state contents appends at the advancing device cursor, as
    T + 2 eager calls do; a captured host-cursor add() would rewrite one slot on every replay."""
    import torch

    from e_alphazero_b200 import ops

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    env = H.make_env("subleq", seed=91, word_size=16)
    denv = H.device_env(env)
    T, B, alpha, seed = 8, 300, 0.6, 4
    S = denv.compact_bytes

    def new_ring():
        rs = torch.zeros((T, B, S), dtype=torch.uint8, device="cuda")
        rr = torch.zeros((T, B), dtype=torch.float32, device="cuda")
        tree = torch.zeros(ops.priority_tree_bytes(T, B), dtype=torch.uint8, device="cuda")
        ops.priority_init(tree, T, B, alpha, seed)
        return rs, rr, tree

    warm = new_ring()
    static = ops.state_to_device(denv, H.random_states(env, B, seed=92))
    ops.replay_add(denv, static, *warm)  # loads the kernels outside the capture
    graph_ring, eager_ring = new_ring(), new_ring()
    buf = P.init(T, B, alpha, seed)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g):
            ops.replay_add(denv, static, *graph_ring)
    torch.cuda.current_stream().wait_stream(side)
    for rep in range(T + 2):
        st = ops.state_to_device(denv, H.random_states(env, B, seed=100 + rep))
        for k in static:
            static[k].copy_(st[k])
        g.replay()
        ops.replay_add(denv, st, *eager_ring)
        oracle_add_at_cursor(buf, T, B)
        torch.cuda.synchronize()
        for a, b, n in zip(graph_ring, eager_ring, ("ring_states", "ring_rewards", "tree")):
            H.assert_same_bits(host(a), host(b), f"replay {rep}: {n}")
        H.assert_same_bits(host(graph_ring[2]), buf, f"replay {rep}: tree vs oracle")
        slot = rep % T
        H.assert_same_bits(host(graph_ring[0][slot]), host(ops.env_compact(denv, st)), f"replay {rep}: row {slot} holds this step")
        H.assert_same_bits(host(graph_ring[1][slot]), host(st["rewards"]).reshape(B), f"replay {rep}: rewards row {slot}")
    hdr = P.header(host(graph_ring[2]))
    assert hdr["cursor"] == (T + 2) % T and hdr["length"] == T and hdr["status"] == 0
