"""The evaluation loop's boundary without a GPU: eaz_evaluate_counters matches its ctypes mirror, the workspace size is the search
workspace plus the loop's words, eaz_evaluate refuses what it cannot run before it touches a device, and the XLA-FFI handler EazEvaluate
compiles against the stand-in and checks its argument lists."""
import ctypes as C
import os
import subprocess
import tempfile
import textwrap

import pytest

from e_alphazero_b200 import _abi, _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.SO_PATH):
        _lib.build()
    return _lib.load()


def test_counters_struct_matches_header():
    src = textwrap.dedent("""
        #include <stdio.h>
        #include <stddef.h>
        #include "eaz_b200.h"
        int main(void) {
          printf("%zu %zu %zu %zu\\n", sizeof(eaz_evaluate_counters), offsetof(eaz_evaluate_counters, live),
                 offsetof(eaz_evaluate_counters, ticket), offsetof(eaz_evaluate_counters, cont));
          return 0;
        }""")
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.run(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "t.c"), "-o", os.path.join(d, "t")], check=True)
        got = [int(x) for x in subprocess.run([os.path.join(d, "t")], capture_output=True, text=True, check=True).stdout.split()]
    S = _abi.EazEvaluateCounters
    assert got == [C.sizeof(S), S.live.offset, S.ticket.offset, S.cont.offset]


def test_workspace_bytes(lib):
    env = _abi.EazEnv(_abi.ENV_DEEPSEA, 30, None, 0, 0, 0)
    cfg = _abi.default_search_config(batch=4096, num_simulations=64, gumbel_scale=0.0)
    search = lib.eaz_search_workspace_bytes(C.byref(cfg), C.byref(env))
    got = lib.eaz_evaluate_workspace_bytes(C.byref(cfg), C.byref(env))
    assert got == 256 + 4096 * 2 * 4 + 4096 * 4 + search  # counters, zero noise [B,A], actions [B], search workspace (256-aligned)
    cfg.flags |= _abi.FLAG_REUSE_PREPARED  # the flag does not change the layout
    assert lib.eaz_evaluate_workspace_bytes(C.byref(cfg), C.byref(env)) == got
    bad = _abi.EazEnv(_abi.ENV_SUBLEQ, 0, None, 8, 1, 0)
    assert lib.eaz_evaluate_workspace_bytes(C.byref(cfg), C.byref(bad)) == 0
    cfg.batch = 0
    assert lib.eaz_evaluate_workspace_bytes(C.byref(cfg), C.byref(env)) == 0


def test_evaluate_validates_without_gpu(lib):
    env = _abi.EazEnv(_abi.ENV_DEEPSEA, 10, None, 0, 0, 0)
    fake = C.c_void_p(0x100000)  # never dereferenced: every call below is refused before anything is enqueued
    st = _abi.EazState(step_count=fake, rewards=fake, terminated=fake, truncated=fake, col=fake)
    net = _abi.EazFcParams()
    beta = fake

    def call(cfg, inp=None, states=st, ws_bytes=1 << 30, ws=C.c_void_p(0x200000), max_len=10):
        inp = inp or _abi.EazSearchInputs(None, None, None, beta, None, None, None, C.pointer(env), None, None)
        return lib.eaz_evaluate(C.byref(cfg), C.byref(inp), C.byref(net), C.byref(states), fake, max_len, ws, C.c_size_t(ws_bytes), None)

    cfg = _abi.default_search_config(batch=8, num_simulations=4, gumbel_scale=0.0)
    assert call(_abi.default_search_config(batch=8, num_simulations=4)) == _abi.EAZ_ERR_INVALID_ARG  # gumbel_scale 1
    assert b"gumbel_scale = 0" in lib.eaz_last_error()
    assert call(_abi.default_search_config(batch=8, num_simulations=4, gumbel_scale=0.0, action_sampling=_abi.ACTION_VISITS)) == _abi.EAZ_ERR_INVALID_ARG
    given_root = _abi.EazSearchInputs(fake, fake, fake, beta, None, None, None, C.pointer(env), None, None)
    assert call(cfg, inp=given_root) == _abi.EAZ_ERR_INVALID_ARG
    assert b"must be NULL" in lib.eaz_last_error()
    assert call(cfg, states=_abi.EazState(step_count=fake, rewards=fake, terminated=fake)) == _abi.EAZ_ERR_INVALID_ARG  # DeepSea needs col
    assert call(cfg, ws_bytes=1024) == _abi.EAZ_ERR_WORKSPACE
    assert call(cfg, ws=C.c_void_p(0x200010)) == _abi.EAZ_ERR_WORKSPACE  # not 256-byte aligned
    assert b"256-byte aligned" in lib.eaz_last_error()


def test_shim_evaluate_handler_validates(lib):
    from tests.xla_ffi_stub import harness as X

    shim = X.load()
    assert hasattr(shim, "EazEvaluate")
    f = lambda *d: X.buf("f32", None, *d)
    B = 4
    leaves = [X.buf("s32", None, B), f(B, 1), X.buf("pred", None, B), X.buf("pred", None, B), X.buf("s32", None, B)]
    params = [f(100, 8), f(8)] * 12  # w, b per layer: D = 100, hidden 8
    attrs = dict(env_kind=_abi.ENV_DEEPSEA, size=10, word_size=0, binary_encoding=0, reward_fn=0, num_simulations=4, max_depth=0,
                 max_num_considered_actions=16, discount=0.97, value_scale=0.1, maxvisit_init=50.0, rescale_values=1, flags=7, mlp_mode=0,
                 hash_bits=24, hash_io=0, max_u=1.0, novelty_scale=1.0, max_episode_length=10)
    args = [f(B), X.buf("u8", None, 10, 10), X.buf("u8", None, 1 << 21), X.buf("u8", None, 1)]
    rets = leaves + [f(B), X.buf("u8", None, 1)]
    rc, msg = X.call(shim, "EazEvaluate", args + leaves + params[:23], rets, attrs)
    assert rc == 3 and "24 parameter buffers" in msg, msg
    rc, msg = X.call(shim, "EazEvaluate", args + leaves + params, rets[:-1], attrs)
    assert rc == 3 and "returns and workspace" in msg, msg
    rc, msg = X.call(shim, "EazEvaluate", args + leaves + params, rets, {k: v for k, v in attrs.items() if k != "max_episode_length"})
    assert rc == 3 and "max_episode_length" in msg, msg
    rc, msg = X.call(shim, "EazEvaluate", args + leaves + params, rets, attrs)  # a 1-byte workspace result
    assert rc == 3 and "eaz_evaluate_workspace_bytes" in msg, msg
