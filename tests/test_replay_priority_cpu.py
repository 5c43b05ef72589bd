"""The prioritised replay sum tree on the CPU oracle (tests/priority_oracle.c): weights and probabilities against a float64
model, the documented descent at child boundaries, zero-weight leaves, duplicate resolution in set, validity across the wrap
of a small ring; and the library's host-side checks of the same entry points (no GPU needed)."""
import ctypes as C
import os

import numpy as np
import pytest

from e_alphazero_b200 import _abi, _lib
from tests import priority_oracle as P


def valid_items(T, B, cursor, length):
    """float64 model of the validity rule: both slots hold data and slot t+1 is not the slot written next."""
    filled = lambda s: (cursor - 1 - s) % T < length
    rows = [(t + 1) % T != cursor and filled(t) and filled((t + 1) % T) for t in range(T)]
    return np.repeat(np.array(rows), B)


def filled_ring(T, B, adds, alpha=0.6, seed=0):
    buf = P.init(T, B, alpha, seed)
    for n in range(adds):
        P.add_step(buf, T, B, n % T)
    return buf


def test_layout_matches_library():
    lib = _lib.load() if os.path.exists(_lib.SO_PATH) else None
    if lib is None:
        _lib.build()
        lib = _lib.load()
    lib.eaz_priority_tree_bytes.restype = C.c_size_t
    for T, B in [(2, 1), (6, 40), (64, 4096), (3, 1000), (1024, 4096)]:
        assert P.tree_bytes(T, B) == lib.eaz_priority_tree_bytes(T, B) > 256 + 4 * 2 * T * B
    assert lib.eaz_priority_tree_bytes(1, 10) == 0 and b"T >= 2" in lib.eaz_last_error()
    assert lib.eaz_priority_tree_bytes(1 << 16, 1 << 15) == 0 and b"below 2^31" in lib.eaz_last_error()
    # host-side argument checks never touch the device
    assert lib.eaz_priority_add_step(None, C.c_size_t(0), 6, 40, 0, None) == _abi.EAZ_ERR_INVALID_ARG
    assert lib.eaz_priority_init(C.c_void_p(1 << 20), C.c_size_t(1 << 20), 6, 40, C.c_float(1.5), 0, None) == _abi.EAZ_ERR_INVALID_ARG
    assert b"priority_exponent" in lib.eaz_last_error()
    assert lib.eaz_priority_sample(C.c_void_p(1 << 20), C.c_size_t(1 << 20), 6, 40, 0, None, None, 0, None, None, None, None, None, None,
                                   None) == _abi.EAZ_ERR_INVALID_ARG


def test_init_header():
    buf = P.init(6, 40, 0.6, seed=123)
    h = P.header(buf)
    assert (h["alpha"], h["seed"], h["draw_ctr"], h["status"], h["cursor"], h["length"], h["max_priority"]) == (np.float32(0.6), 123, 0, 0, 0, 0, 1.0)
    assert (buf[256:256 + 4 * 240].view(np.int32) == -1).all()
    assert all((lv == 0).all() for lv in P.levels(buf, 6, 40))


@pytest.mark.parametrize("alpha", [0.0, 0.6, 1.0])
def test_probabilities_match_float64_model(alpha):
    T, B = 4, 300
    buf = filled_ring(T, B, 3, alpha)
    h = P.header(buf)
    valid = valid_items(T, B, int(h["cursor"]), int(h["length"]))
    rng = np.random.default_rng(5)
    idx = np.flatnonzero(valid)
    pri = rng.lognormal(0.0, 1.5, idx.size).astype(np.float32)
    pri[rng.random(idx.size) < 0.1] = 0
    P.set_priorities(buf, T, B, idx, pri)
    w = np.zeros(T * B)
    w[idx] = np.where(pri > 0, pri.astype(np.float64) ** alpha, 0.0)
    out = P.sample(buf, T, B, 2048)
    i = out["indices"]
    assert (w[i] > 0).all()
    np.testing.assert_allclose(out["probabilities"], w[i] / w.sum(), rtol=1e-6)
    # the tree's levels are sums of their children
    lv = P.levels(buf, T, B)
    np.testing.assert_allclose(lv[0], w, rtol=1e-6)
    for l in range(1, len(lv)):
        np.testing.assert_allclose(lv[l], np.add.reduceat(np.pad(lv[l - 1].astype(np.float64), (0, (-lv[l - 1].size) % 32)),
                                                          np.arange(0, lv[l - 1].size, 32))[: lv[l].size], rtol=1e-6)
    assert P.header(buf)["draw_ctr"] == 1


def test_descent_at_child_boundaries():
    """Two levels of 32 children with exactly representable weights: u just below / at a prefix picks the child whose prefix
    first exceeds u; zero-weight children in between are skipped."""
    T, B = 32, 32  # 1024 leaves: leaves -> 32 nodes -> root
    buf = filled_ring(T, B, T + 1)
    h = P.header(buf)
    valid = valid_items(T, B, int(h["cursor"]), int(h["length"]))
    w = np.zeros(T * B, np.float32)
    w[valid] = 1.0
    w[np.flatnonzero(valid)[::3]] = 0.0  # zero-weight children between non-zero ones
    P.set_priorities(buf, T, B, np.arange(T * B)[valid], w[valid])
    leaves = P.levels(buf, T, B)[0]
    assert (leaves == w).all()
    cum = np.cumsum(w.astype(np.float64))  # exact: integers
    for target in np.flatnonzero(w)[::7]:
        lo, hi = cum[target] - 1.0, cum[target]  # [lo, hi) maps to `target`
        assert P.descend(buf, T, B, lo) == target
        assert P.descend(buf, T, B, np.nextafter(np.float32(hi), np.float32(0))) == target
        assert P.descend(buf, T, B, hi) != target
    # u at or past the total (as rounding can leave it): the last non-zero leaf, never a zero one
    last = np.flatnonzero(w)[-1]
    for u in (cum[-1], cum[-1] * 2, np.inf):
        assert P.descend(buf, T, B, u) == last


def test_zero_weights_never_drawn_with_rounding():
    """Weights of very different magnitudes (sums round), many zeros: no sample ever lands on a zero leaf."""
    T, B = 3, 2000
    buf = filled_ring(T, B, 2, alpha=1.0)
    h = P.header(buf)
    valid = valid_items(T, B, int(h["cursor"]), int(h["length"]))
    idx = np.flatnonzero(valid)
    rng = np.random.default_rng(9)
    pri = (10.0 ** rng.uniform(-30, 30, idx.size)).astype(np.float32)
    pri[rng.random(idx.size) < 0.5] = 0
    pri[-1] = 0  # a zero at the very end, where an overshooting u lands
    P.set_priorities(buf, T, B, idx, pri)
    leaves = P.levels(buf, T, B)[0]
    for _ in range(8):
        out = P.sample(buf, T, B, 4096)
        assert (leaves[out["indices"]] > 0).all()
    for u in (np.float32(P.levels(buf, T, B)[-1][0]), np.float32(3e38)):
        assert leaves[P.descend(buf, T, B, u)] > 0


def test_set_duplicates_last_occurrence_wins():
    T, B = 6, 40
    buf = filled_ring(T, B, 6)
    idx = np.array([3, 7, 3, 3, 7, 11, 3], np.int32)
    pri = np.array([5.0, 1.0, 2.0, 9.0, 4.0, 0.0, 0.25], np.float32)
    P.set_priorities(buf, T, B, idx, pri)
    leaves = P.levels(buf, T, B)[0]
    assert np.isclose(leaves[3], 0.25 ** 0.6, rtol=1e-6) and np.isclose(leaves[7], 4.0 ** 0.6, rtol=1e-6) and leaves[11] == 0
    assert P.header(buf)["max_priority"] == 9.0
    assert (buf[256:256 + 4 * T * B].view(np.int32) == -1).all()


def test_add_step_validity_across_wrap():
    T, B = 4, 3
    buf = P.init(T, B, 0.5)
    for n in range(11):
        c = n % T
        P.add_step(buf, T, B, c)
        h = P.header(buf)
        assert h["cursor"] == (c + 1) % T and h["length"] == min(n + 1, T)
        valid = valid_items(T, B, int(h["cursor"]), int(h["length"]))
        leaves = P.levels(buf, T, B)[0]
        assert ((leaves > 0) == valid).all(), (n, leaves.reshape(T, B))
        assert (leaves[valid] == 1.0).all()  # max priority 1 ** alpha
        # the pair ending at the newest slot is valid, the pair starting there is not
        assert valid[((c - 1) % T) * B] == (n >= 1) and not valid[c * B]
    # a stale handle (its first slot has since become the newest) keeps weight 0 when set
    P.set_priorities(buf, T, B, [c * B, ((c + 1) % T) * B], [3.0, 2.0])
    leaves = P.levels(buf, T, B)[0]
    assert leaves[c * B] == 0 and leaves[((c + 1) % T) * B] > 0
    # a rewrite of the newest slot keeps cursor / length; any other slot is refused with a status bit
    P.add_step(buf, T, B, c)
    assert P.header(buf)["cursor"] == (c + 1) % T and P.header(buf)["status"] == 0
    P.add_step(buf, T, B, (c + 2) % T)
    assert P.header(buf)["status"] == _abi.PRIORITY_BAD_ADD


def test_bad_priorities_and_indices_set_status():
    T, B = 6, 40
    buf = filled_ring(T, B, 6)
    P.set_priorities(buf, T, B, [0, 1, 2, 240, -1], [-1.0, np.nan, np.inf, 1.0, 1.0])
    leaves = P.levels(buf, T, B)[0]
    assert (leaves[:3] == 0).all()
    assert P.header(buf)["status"] == _abi.PRIORITY_BAD_PRIORITY | _abi.PRIORITY_BAD_INDEX
    empty = P.init(T, B)
    out = P.sample(empty, T, B, 4)
    assert (out["indices"] == 0).all() and (out["probabilities"] == 0).all() and P.header(empty)["status"] == _abi.PRIORITY_EMPTY
