"""PrioritisedReplayRing on the GPU (csrc/replay.cu) against the CPU oracle of the sum tree (tests/priority_oracle.c): the whole
tree buffer (every level and the header), the drawn indices, probabilities and decoded pairs bit for bit; validity of every
sampled pair; the sampling distribution; CUDA-graph replay; the status bits."""
import numpy as np
import pytest

from e_alphazero_b200 import _abi
from oracle import oracle as O
from tests import helpers as H
from tests import priority_oracle as P

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from e_alphazero_b200 import ops as _ops

    return _ops


def host(t):
    return t.detach().cpu().numpy()


def assert_tree(ring, buf, what):
    H.assert_same_bits(host(ring.tree), buf, f"tree after {what}")


def assert_sample(ring, got, exp, env, traj, what):
    """got: PrioritisedSample; exp: the oracle's draw from the same tree; traj[t]: host state dict written to slot t."""
    H.assert_same_bits(host(got.indices), exp["indices"], f"{what} indices")
    H.assert_same_bits(host(got.probabilities), exp["probabilities"], f"{what} probabilities")
    for side in ("first", "second"):
        H.assert_same_bits(host(got.compact[side]), exp[side], f"{what} {side} records")
        H.assert_same_bits(host(got.compact[side + "_rewards"]), exp[side + "_rewards"], f"{what} {side} rewards")
        dec = H.uncompact(env, exp[side])
        for k in O.state_fields(env):
            if k != "rewards":
                H.assert_same_bits(host(getattr(got.experience, side)[k]), dec[k], f"{what} {side} {k}")
    # validity: every pair is two consecutive stored states of one env, never through the slot written next
    T, B = ring.T, ring.B
    idx = exp["indices"]
    t, b = idx // B, idx % B
    t1 = (t + 1) % T
    assert (t1 != ring.cursor).all(), what
    assert all(traj[s] is not None for s in np.concatenate([t, t1])), what
    f = {k: host(v) for k, v in got.experience.first.items()}
    s2 = {k: host(v) for k, v in got.experience.second.items()}
    for k in O.state_fields(env):
        H.assert_same_bits(f[k], np.stack([traj[ti][k][bi] for ti, bi in zip(t, b)]), f"{what} first {k} is the stored state")
        H.assert_same_bits(s2[k], np.stack([traj[ti][k][bi] for ti, bi in zip(t1, b)]), f"{what} second {k} is the next stored state")


@pytest.mark.parametrize("kind,kw", [("deepsea", dict(size=30)), ("subleq", dict(word_size=16)), ("subleq", dict(word_size=256, binary=False))])
def test_bit_exact_against_oracle(ops, kind, kw):
    import torch

    from e_alphazero_b200.replay import PrioritisedReplayRing

    env = H.make_env(kind, seed=51, **kw)
    denv = H.device_env(env)
    T, B, alpha, seed = 6, 40, 0.6, 77
    ring = PrioritisedReplayRing(denv, T, B, priority_exponent=alpha, seed=seed)
    buf = P.init(T, B, alpha, seed)
    assert_tree(ring, buf, "init")
    rng = np.random.default_rng(52)
    cur = ops.state_to_device(denv, H.random_states(env, B, seed=53))
    traj = [None] * T
    old_handles = None

    def add():
        nonlocal cur
        slot = ring.cursor
        ring.add(cur)
        traj[slot] = {k: host(v).copy() for k, v in cur.items()}
        P.add_step(buf, T, B, slot)
        assert_tree(ring, buf, f"add slot {slot}")
        cur = ops.env_step(denv, cur, H.to_device(rng.integers(0, env.num_actions, B).astype(np.int32)), auto_reset=True,
                           task_ids=np.ones(B, np.int32) if kind == "subleq" else None)

    def sample(K):
        got = ring.sample(K)
        exp = P.sample(buf, T, B, K, host(ring.states), host(ring.rewards))
        assert_tree(ring, buf, "sample")
        assert_sample(ring, got, exp, env, traj, f"sample {K}")
        return got

    def set_(idx, pri):
        ring.set_priorities(H.to_device(np.asarray(idx, np.int32)), H.to_device(np.asarray(pri, np.float32)))
        P.set_priorities(buf, T, B, idx, pri)
        assert_tree(ring, buf, "set_priorities")

    for _ in range(4):
        add()
    got = sample(96)
    # duplicates (last wins), zeros, a spread of magnitudes over the drawn handles and some never drawn
    idx = np.concatenate([host(got.indices), rng.integers(0, T * B, 64)]).astype(np.int32)
    idx[10:20] = idx[0]
    pri = (10.0 ** rng.uniform(-6, 6, idx.size)).astype(np.float32)
    pri[rng.random(idx.size) < 0.15] = 0
    set_(idx, pri)
    sample(256)
    old_handles = host(got.indices).copy()
    for _ in range(5):  # past the wrap: the handles drawn above go stale one row at a time
        add()
    set_(old_handles, np.full(old_handles.size, 3.5, np.float32))  # stale handles stay at weight 0
    for K in (1, 37, 512):
        sample(K)
    set_(np.arange(T * B, dtype=np.int32)[::-1], rng.uniform(0, 2, T * B).astype(np.float32))
    sample(4096)
    assert ring.numeric_status() == 0
    torch.cuda.synchronize()


def _distribution_ring(ops, B, alpha, seed):
    from e_alphazero_b200.replay import PrioritisedReplayRing

    env = H.make_env("deepsea", seed=1, size=10)
    denv = H.device_env(env)
    ring = PrioritisedReplayRing(denv, 2, B, priority_exponent=alpha, seed=seed)
    st = ops.env_init(denv, B)
    ring.add(st)
    ring.add(st)  # slots 0, 1: the B items of row 0 are valid, row 1 ends at the slot written next
    return ring


@pytest.mark.parametrize("alpha", [0.6, 0.0])
def test_distribution(ops, alpha):
    import torch
    from scipy import stats

    B, K, calls = 4096, 4096, 245  # ~10^6 draws
    ring = _distribution_ring(ops, B, alpha, seed=5)
    rng = np.random.default_rng(6)
    pri = rng.uniform(0.2, 5.0, B).astype(np.float32)
    pri[rng.random(B) < 0.1] = 0
    ring.set_priorities(H.to_device(np.arange(B, dtype=np.int32)), H.to_device(pri))
    idx = torch.empty(K, dtype=torch.int32, device="cuda")
    prob = torch.empty(K, dtype=torch.float32, device="cuda")
    counts = torch.zeros(2 * B, dtype=torch.int64, device="cuda")
    for _ in range(calls):
        ops.priority_sample(ring.tree, ring.T, ring.B, idx, prob)
        counts += torch.bincount(idx.long(), minlength=2 * B)
    counts = host(counts)
    assert counts[B:].sum() == 0, "drew an item of the invalid row"
    c = counts[:B]
    assert c[pri == 0].sum() == 0, "drew a zero-priority item"
    w = np.where(pri > 0, pri.astype(np.float64) ** alpha, 0.0)
    nz = w > 0
    exp = c.sum() * w[nz] / w[nz].sum()
    p = stats.chisquare(c[nz], exp).pvalue
    assert p > 1e-3, p
    assert ring.numeric_status() == 0


def test_graph_capture_equals_eager(ops):
    import torch

    from e_alphazero_b200.replay import PrioritisedReplayRing

    env = H.make_env("subleq", seed=61, word_size=16)
    denv = H.device_env(env)
    T, B, K, reps = 6, 40, 128, 4
    rings = [PrioritisedReplayRing(denv, T, B, priority_exponent=0.6, seed=9) for _ in range(2)]
    st = ops.state_to_device(denv, H.random_states(env, B, seed=62))
    for r in rings:
        for _ in range(T + 2):
            r.add(st)
    pr = H.to_device(np.random.default_rng(63).uniform(0.1, 4.0, K).astype(np.float32))
    bufs = [r.alloc_sample(K) for r in rings]
    c = rings[0].cursor

    def step(r, out):
        r.cursor = c  # a captured add() rewrites the slot it was captured for on every replay; the eager twin does the same
        r.add(st)
        r.sample(K, out=out)
        r.set_priorities(out.indices, pr)

    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g):
            step(rings[0], bufs[0])
    torch.cuda.current_stream().wait_stream(side)
    for rep in range(reps):
        g.replay()
        step(rings[1], bufs[1])
        torch.cuda.synchronize()
        H.assert_same_bits(host(rings[0].tree), host(rings[1].tree), f"tree, replay {rep}")
        H.assert_same_bits(host(bufs[0].indices), host(bufs[1].indices), f"indices, replay {rep}")
        H.assert_same_bits(host(bufs[0].probabilities), host(bufs[1].probabilities), f"probabilities, replay {rep}")
    assert P.header(host(rings[0].tree))["draw_ctr"] == reps


def test_status_bits(ops):
    from e_alphazero_b200._lib import EazError

    ring = _distribution_ring(ops, 64, 0.6, seed=3)
    assert ring.numeric_status() == 0
    ring.set_priorities(H.to_device(np.array([1, 2, 3], np.int32)), H.to_device(np.array([-2.0, np.nan, 1.0], np.float32)))
    with pytest.raises(EazError, match="non-finite"):
        ring.numeric_status()
    leaves = P.levels(host(ring.tree), ring.T, ring.B)[0]
    assert leaves[1] == 0 and leaves[2] == 0 and leaves[3] == 1.0
    assert P.header(host(ring.tree))["status"] == _abi.PRIORITY_BAD_PRIORITY
    # out-of-range device indices are skipped and reported; host indices are refused before anything runs
    ring.set_priorities(H.to_device(np.array([5, 10 ** 6], np.int32)), H.to_device(np.array([1.0, 1.0], np.float32)))
    assert P.header(host(ring.tree))["status"] == _abi.PRIORITY_BAD_PRIORITY | _abi.PRIORITY_BAD_INDEX
    with pytest.raises(EazError, match="outside"):
        ring.set_priorities(np.array([-1]), np.array([1.0]))
