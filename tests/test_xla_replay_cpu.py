"""The replay handlers of csrc/xla_ffi_shim.cc without a GPU: the shim still compiles with -Wall -Werror against the XLA-FFI stand-in
(tests/xla_ffi_stub/), exports the five replay handlers, and each handler refuses bad input with kInvalidArgument before anything
touches a device (the buffers below carry no device memory: null or fake pointers that are never dereferenced)."""
import ctypes as C
import os

import pytest

from e_alphazero_b200 import _abi, _lib

INVALID = 3  # xla::ffi::ErrorCode::kInvalidArgument
T, B = 8, 100
FAKE_MISALIGNED = 0x10040  # 64-byte but not 128-byte aligned
U32 = 8  # xla::ffi::DataType::U32 of the stand-in header (tests/xla_ffi_stub/xla/ffi/api/ffi.h)


@pytest.fixture(scope="module")
def shim():
    if not os.path.exists(_lib.SO_PATH):
        _lib.build()
    from tests.xla_ffi_stub import harness as X

    return X, X.load()


def deepsea_attrs():
    return dict(env_kind=_abi.ENV_DEEPSEA, size=30, word_size=0, binary_encoding=0, reward_fn=0)


def tree_bytes(t, b):
    return int(_lib.load().eaz_priority_tree_bytes(t, b))


def leaves(X, n, n_step=None):
    """DeepSea state leaves of n envs (step_count, rewards, terminated, truncated, col); n_step overrides the first leaf's rows"""
    return [X.buf("s32", None, n if n_step is None else n_step), X.buf("f32", None, n, 1), X.buf("pred", None, n), X.buf("pred", None, n),
            X.buf("s32", None, n)]


def u32buf(X, ptr, *dims):
    return X.StubBuf(U32, len(dims), ptr, (C.c_int64 * 4)(*dims))


def test_shim_exports_replay_handlers(shim):
    X, lib = shim
    for h in ("EazReplayInit", "EazReplayAdd", "EazReplaySample", "EazReplaySetPriorities", "EazReplayStatus"):
        assert hasattr(lib, h), h


def test_init_rejects(shim):
    X, lib = shim
    attrs = dict(T=T, B=B, priority_exponent=0.6, seed=3)
    rets = lambda t, b, tree: [X.buf("u8", None, t, b, 4), X.buf("f32", None, t, b), tree]
    ok_tree = X.buf("u8", None, tree_bytes(T, B))
    rc, msg = X.call(lib, "EazReplayInit", [], rets(1, B, ok_tree), dict(attrs, T=1))
    assert rc == INVALID and "T >= 2" in msg, msg
    rc, msg = X.call(lib, "EazReplayInit", [], rets(2, 1 << 30, ok_tree), dict(attrs, T=2, B=1 << 30))
    assert rc == INVALID and "2^31" in msg, msg
    rc, msg = X.call(lib, "EazReplayInit", [], rets(T, B, X.buf("u8", None, tree_bytes(T, B) - 1)), attrs)
    assert rc == INVALID and "tree buffer of" in msg, msg
    rc, msg = X.call(lib, "EazReplayInit", [], rets(T, B, X.buf("u8", FAKE_MISALIGNED, tree_bytes(T, B))), attrs)
    assert rc == INVALID and "128-byte aligned" in msg, msg
    rc, msg = X.call(lib, "EazReplayInit", [], rets(T, B + 1, ok_tree), attrs)  # ring shape does not match (T, B)
    assert rc == INVALID and "ring_states" in msg, msg
    rc, msg = X.call(lib, "EazReplayInit", [], rets(T, B, ok_tree), dict(attrs, priority_exponent=1.5))
    assert rc == INVALID and "priority_exponent" in msg, msg


def test_add_rejects(shim):
    X, lib = shim
    amap = X.buf("u8", None, 30, 30)

    def call(t, b, tree, lv, S=4):
        ring = [X.buf("u8", None, t, b, S), X.buf("f32", None, t, b), tree]
        return X.call(lib, "EazReplayAdd", [amap] + ring + lv, ring, deepsea_attrs())

    ok_tree = X.buf("u8", None, tree_bytes(T, B))
    rc, msg = call(T, B, X.buf("u8", FAKE_MISALIGNED, tree_bytes(T, B)), leaves(X, B))
    assert rc == INVALID and "128-byte aligned" in msg, msg
    rc, msg = call(T, B, X.buf("u8", None, 1024), leaves(X, B))
    assert rc == INVALID and "tree buffer of" in msg, msg
    rc, msg = call(1, B, ok_tree, leaves(X, B))
    assert rc == INVALID and "T >= 2" in msg, msg
    rc, msg = call(2, 1 << 30, ok_tree, leaves(X, 1 << 30))
    assert rc == INVALID and "2^31" in msg, msg
    rc, msg = call(T, B, ok_tree, leaves(X, B, n_step=B - 1))
    assert rc == INVALID and "does not hold" in msg, msg
    rc, msg = call(T, B, ok_tree, leaves(X, B)[:4])
    assert rc == INVALID and "number of state leaves" in msg, msg
    rc, msg = call(T, B, ok_tree, leaves(X, B), S=8)  # DeepSea records are 4 bytes
    assert rc == INVALID and "compact_bytes" in msg, msg


def test_sample_rejects(shim):
    X, lib = shim
    amap = X.buf("u8", None, 30, 30)
    key = u32buf(X, None, 2)

    def call(t, b, tree, K, k_rets=None, key=key):
        kr = K if k_rets is None else k_rets
        args = [amap, X.buf("u8", None, t, b, 4), X.buf("f32", None, t, b), tree, key]
        rets = [X.buf("s32", None, kr), X.buf("f32", None, kr)] + leaves(X, kr) + leaves(X, kr) + [X.buf("u8", None, 2 * kr * 8 + 16)]
        return X.call(lib, "EazReplaySample", args, rets, dict(deepsea_attrs(), K=K))

    ok_tree = X.buf("u8", None, tree_bytes(T, B))
    rc, msg = call(T, B, ok_tree, 0, k_rets=1)
    assert rc == INVALID and "K = 0" in msg, msg
    rc, msg = call(T, B, ok_tree, 37, k_rets=36)
    assert rc == INVALID and "[K]" in msg, msg
    rc, msg = call(T, B, X.buf("u8", FAKE_MISALIGNED, tree_bytes(T, B)), 37)
    assert rc == INVALID and "128-byte aligned" in msg, msg
    rc, msg = call(T, B, X.buf("u8", None, 256), 37)
    assert rc == INVALID and "tree buffer of" in msg, msg
    rc, msg = call(1, B, ok_tree, 37)
    assert rc == INVALID and "T >= 2" in msg, msg
    rc, msg = call(2, 1 << 30, ok_tree, 37)
    assert rc == INVALID and "2^31" in msg, msg
    rc, msg = call(T, B, ok_tree, 37, key=u32buf(X, None, 3))
    assert rc == INVALID and "key" in msg, msg
    rc, msg = call(T, B, ok_tree, 37, key=X.buf("s32", None, 2))  # the key is U32: the binding checks the dtype
    assert rc == INVALID and "dtype" in msg, msg
    # leaf rows that do not match K
    args = [amap, X.buf("u8", None, T, B, 4), X.buf("f32", None, T, B), ok_tree, key]
    rets = [X.buf("s32", None, 37), X.buf("f32", None, 37)] + leaves(X, 37) + leaves(X, 37, n_step=36) + [X.buf("u8", None, 1024)]
    rc, msg = X.call(lib, "EazReplaySample", args, rets, dict(deepsea_attrs(), K=37))
    assert rc == INVALID and "does not hold" in msg, msg


def test_set_priorities_and_status_reject(shim):
    X, lib = shim

    def call(t, b, tree, K=5, Kp=None):
        args = [X.buf("s32", None, K), X.buf("f32", None, K if Kp is None else Kp), tree]
        return X.call(lib, "EazReplaySetPriorities", args, [tree], dict(T=t, B=b))

    ok_tree = X.buf("u8", None, tree_bytes(T, B))
    rc, msg = call(T, B, X.buf("u8", FAKE_MISALIGNED, tree_bytes(T, B)))
    assert rc == INVALID and "128-byte aligned" in msg, msg
    rc, msg = call(T, B, X.buf("u8", None, 512))
    assert rc == INVALID and "tree buffer of" in msg, msg
    rc, msg = call(1, B, ok_tree)
    assert rc == INVALID and "T >= 2" in msg, msg
    rc, msg = call(1 << 16, 1 << 15, ok_tree)
    assert rc == INVALID and "2^31" in msg, msg
    rc, msg = call(T, B, ok_tree, K=5, Kp=4)
    assert rc == INVALID and "differ in length" in msg, msg
    # status: a misaligned or short tree
    rc, msg = X.call(lib, "EazReplayStatus", [X.buf("u8", FAKE_MISALIGNED, tree_bytes(T, B))], [X.buf("s32", None, 1)], {})
    assert rc == INVALID and "128-byte aligned" in msg, msg
    rc, msg = X.call(lib, "EazReplayStatus", [X.buf("u8", None, 16)], [X.buf("s32", None, 1)], {})
    assert rc == INVALID and "short tree" in msg, msg
