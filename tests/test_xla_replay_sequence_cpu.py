"""The sequence add of the replay ring without a GPU: the XLA-FFI shim still compiles with -Wall -Werror against the stand-in
(tests/xla_ffi_stub/) and exports EazReplayAddSequence, which refuses bad shapes with kInvalidArgument, and eaz_replay_add_sequence
refuses bad arguments with EAZ_ERR_INVALID_ARG and a message.  No device memory is touched: the buffers are null or fake pointers that
are never dereferenced, because every check runs before anything is enqueued."""
import ctypes as C
import os

import pytest

from e_alphazero_b200 import _abi, _lib

INVALID = 3  # xla::ffi::ErrorCode::kInvalidArgument
T, B, S = 8, 100, 4  # DeepSea records are 4 bytes
FAKE_ALIGNED = 0x20000  # 128-byte aligned, never dereferenced
FAKE_MISALIGNED = 0x10040  # 64-byte but not 128-byte aligned


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.SO_PATH):
        _lib.build()
    return _lib.load()


@pytest.fixture(scope="module")
def shim(lib):
    from tests.xla_ffi_stub import harness as X

    return X, X.load()


def tree_bytes(lib, t, b):
    return int(lib.eaz_priority_tree_bytes(t, b))


def deepsea_attrs():
    return dict(env_kind=_abi.ENV_DEEPSEA, size=30, word_size=0, binary_encoding=0, reward_fn=0)


def test_shim_exports_sequence_handler(shim):
    X, slib = shim
    assert hasattr(slib, "EazReplayAddSequence")


def test_sequence_handler_rejects(shim, lib):
    X, slib = shim
    amap = X.buf("u8", None, 30, 30)
    ok_tree = X.buf("u8", None, tree_bytes(lib, T, B))

    def call(tree=ok_tree, ring=(T, B, S), compact=(5, B, S), rewards=(5, B), rewards_kind="f32", tree_ret=None):
        rs, rr = X.buf("u8", None, *ring), X.buf("f32", None, *ring[:2])
        args = [amap, rs, rr, tree, X.buf("u8", None, *compact), X.buf(rewards_kind, None, *rewards)]
        return X.call(slib, "EazReplayAddSequence", args, [rs, rr, tree if tree_ret is None else tree_ret], deepsea_attrs())

    rc, msg = call(tree=X.buf("u8", FAKE_MISALIGNED, tree_bytes(lib, T, B)))
    assert rc == INVALID and "128-byte aligned" in msg, msg
    rc, msg = call(tree=X.buf("u8", None, 1024))
    assert rc == INVALID and "tree buffer of" in msg, msg
    rc, msg = call(tree_ret=X.buf("u8", None, tree_bytes(lib, T, B) + 128))
    assert rc == INVALID and "shape of its input" in msg, msg
    # the sequence's B or S does not match the ring
    rc, msg = call(compact=(5, B + 1, S), rewards=(5, B + 1))
    assert rc == INVALID and "compact must be" in msg, msg
    rc, msg = call(compact=(5, B, S + 4))
    assert rc == INVALID and "compact must be" in msg, msg
    rc, msg = call(compact=(5 * B, S), rewards=(5 * B,))
    assert rc == INVALID and "compact must be" in msg, msg
    # the ring's S does not match the env (DeepSea: 4 bytes)
    rc, msg = call(ring=(T, B, 8), compact=(5, B, 8))
    assert rc == INVALID and "compact_bytes" in msg, msg
    # rewards of the wrong shape or dtype
    for bad in ((5, B + 1), (6, B), (5 * B,), (5, B, 1)):
        rc, msg = call(rewards=bad)
        assert rc == INVALID and "rewards must be" in msg, (bad, msg)
    rc, msg = call(rewards_kind="s32")
    assert rc == INVALID and "dtype" in msg, msg
    # shapes that pass reach the library, whose own checks answer for the null buffers without touching a device
    rc, msg = call(tree=X.buf("u8", FAKE_ALIGNED, tree_bytes(lib, T, B)))  # aliased (same buffers in and out): nothing to copy
    assert rc == INVALID and "eaz_replay_add_sequence" in msg and "NULL ring_states" in msg, msg


def test_c_abi_rejects(lib):
    env = _abi.EazEnv(_abi.ENV_DEEPSEA, 30, None, 0, 0, 0)
    nb = tree_bytes(lib, T, B)
    fake = C.c_void_p(FAKE_ALIGNED)

    def call(compact=fake, rewards=fake, steps=3, ring_states=fake, ring_rewards=fake, tree=fake, nbytes=nb, t=T, b=B, s=S, e=env):
        rc = lib.eaz_replay_add_sequence(C.byref(e), compact, rewards, steps, ring_states, ring_rewards, tree, C.c_size_t(nbytes), t, b, s,
                                         None)
        return rc, lib.eaz_last_error().decode()

    rc, msg = call(steps=-1)
    assert rc == _abi.EAZ_ERR_INVALID_ARG and "steps = -1" in msg, msg
    rc, msg = call(s=8)
    assert rc == _abi.EAZ_ERR_INVALID_ARG and "S = 8" in msg and "eaz_env_compact_bytes" in msg, msg
    sub = _abi.EazEnv(_abi.ENV_SUBLEQ, 0, None, 16, 1, 0)  # Subleq-16 records are 56 bytes, not 4
    rc, msg = call(e=sub)
    assert rc == _abi.EAZ_ERR_INVALID_ARG and "S = 4" in msg, msg
    for name in ("ring_states", "ring_rewards"):
        rc, msg = call(**{name: None})
        assert rc == _abi.EAZ_ERR_INVALID_ARG and "NULL ring_states / ring_rewards" in msg, (name, msg)
    for name in ("compact", "rewards"):
        rc, msg = call(**{name: None})
        assert rc == _abi.EAZ_ERR_INVALID_ARG and "NULL compact / rewards" in msg, (name, msg)
    rc, msg = call(tree=None)
    assert rc == _abi.EAZ_ERR_INVALID_ARG and "128-byte aligned" in msg, msg
    rc, msg = call(nbytes=nb - 1)
    assert rc == _abi.EAZ_ERR_INVALID_ARG and "tree buffer of" in msg, msg
    rc, msg = call(t=1)
    assert rc == _abi.EAZ_ERR_INVALID_ARG and "T >= 2" in msg, msg
    bad_env = _abi.EazEnv(_abi.ENV_SUBLEQ, 0, None, 8, 1, 0)  # word_size < 16 (subleq.py:606)
    rc, msg = call(e=bad_env)
    assert rc == _abi.EAZ_ERR_INVALID_ARG and "word_size" in msg, msg


def test_c_abi_zero_steps_enqueues_nothing(lib):
    """steps == 0 returns 0 without a launch: the fake pointers are never touched, and null sequence buffers are accepted"""
    env = _abi.EazEnv(_abi.ENV_DEEPSEA, 30, None, 0, 0, 0)
    fake = C.c_void_p(FAKE_ALIGNED)
    for seq in (fake, None):
        rc = lib.eaz_replay_add_sequence(C.byref(env), seq, seq, 0, fake, fake, fake, C.c_size_t(tree_bytes(lib, T, B)), T, B, S, None)
        assert rc == 0, lib.eaz_last_error()
