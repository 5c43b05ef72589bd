"""The self-play scan's boundary without a GPU: eaz_selfplay_outputs matches its ctypes mirror, the workspace size is the search workspace
plus the loop's words, the staged noise and one step's outputs, eaz_selfplay refuses what it cannot run before it touches a device
(and enqueues nothing for T = 0), and the XLA-FFI handler EazSelfplay compiles against the stand-in and checks its arguments."""
import ctypes as C
import os
import subprocess
import tempfile
import textwrap

import pytest

from e_alphazero_b200 import _abi, _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = C.c_void_p(0x100000)  # never dereferenced: every call below returns before anything is enqueued
WS = C.c_void_p(0x200000)


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.SO_PATH):
        _lib.build()
    return _lib.load()


def test_outputs_struct_matches_header():
    names = [n for n, _ in _abi.EazSelfplayOutputs._fields_]
    offs = ", ".join(f"offsetof(eaz_selfplay_outputs, {n})" for n in names)
    src = textwrap.dedent(f"""
        #include <stdio.h>
        #include <stddef.h>
        #include "eaz_b200.h"
        int main(void) {{
          size_t o[] = {{{offs}}};
          printf("%zu", sizeof(eaz_selfplay_outputs));
          for (size_t i = 0; i < sizeof(o) / sizeof(o[0]); ++i) printf(" %zu", o[i]);
          printf("\\n");
          return 0;
        }}""")
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "t.c"), "w").write(src)
        subprocess.run(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "t.c"), "-o", os.path.join(d, "t")], check=True)
        got = [int(x) for x in subprocess.run([os.path.join(d, "t")], capture_output=True, text=True, check=True).stdout.split()]
    S = _abi.EazSelfplayOutputs
    assert got == [C.sizeof(S)] + [getattr(S, n).offset for n in names]


def test_workspace_bytes(lib):
    al = lambda x: (x + 255) // 256 * 256
    for env, A in ((_abi.EazEnv(_abi.ENV_DEEPSEA, 30, None, 0, 0, 0), 2), (_abi.EazEnv(_abi.ENV_SUBLEQ, 0, None, 40, 1, 0), 40)):
        cfg = _abi.default_search_config(batch=4099, num_simulations=64)
        search = lib.eaz_search_workspace_bytes(C.byref(cfg), C.byref(env))
        got = lib.eaz_selfplay_workspace_bytes(C.byref(cfg), C.byref(env))
        # loop words, staged gumbel + sample_gumbel [B,A], action / value / std / root value / root ube [B], q-value variances [B,A]
        assert got == 256 + 3 * al(4099 * A * 4) + 5 * al(4099 * 4) + search
        cfg.flags |= _abi.FLAG_REUSE_PREPARED  # the flag does not change the layout
        assert lib.eaz_selfplay_workspace_bytes(C.byref(cfg), C.byref(env)) == got
    bad = _abi.EazEnv(_abi.ENV_SUBLEQ, 0, None, 8, 1, 0)
    assert lib.eaz_selfplay_workspace_bytes(C.byref(cfg), C.byref(bad)) == 0
    assert lib.eaz_selfplay_workspace_bytes(C.byref(_abi.default_search_config(batch=0)), C.byref(env)) == 0


def _call(lib, cfg, env, inp=None, states=None, T=8, tasks=None, ws=WS, ws_bytes=1 << 40):
    if states is None:
        states = (_abi.EazState(step_count=FAKE, rewards=FAKE, terminated=FAKE, truncated=FAKE, col=FAKE) if env.kind == _abi.ENV_DEEPSEA else
                  _abi.EazState(step_count=FAKE, rewards=FAKE, terminated=FAKE, truncated=FAKE, memory=FAKE, task=FAKE, solved=FAKE,
                                input_after=FAKE, output_after=FAKE))
    inp = inp or _abi.EazSearchInputs(None, None, None, FAKE, None, None, None, C.pointer(env), None, None)
    out = _abi.EazSelfplayOutputs(*([FAKE] * 9))
    return lib.eaz_selfplay(C.byref(cfg), C.byref(inp), C.byref(_abi.EazFcParams()), C.byref(states), C.c_int32(T), tasks, C.byref(out), ws,
                            C.c_size_t(ws_bytes), None)


def test_selfplay_validates_without_gpu(lib):
    ds = _abi.EazEnv(_abi.ENV_DEEPSEA, 10, None, 0, 0, 0)
    sq = _abi.EazEnv(_abi.ENV_SUBLEQ, 0, None, 256, 1, 0)
    cfg = _abi.default_search_config(batch=8, num_simulations=4)
    err = lambda: lib.eaz_last_error().decode()
    given_root = _abi.EazSearchInputs(FAKE, FAKE, FAKE, FAKE, None, None, None, C.pointer(ds), None, None)
    assert _call(lib, cfg, ds, inp=given_root) == _abi.EAZ_ERR_INVALID_ARG and "must be NULL" in err()
    puct = _abi.default_search_config(batch=8, num_simulations=4, flags=_abi.SEARCH_DEFAULT_FLAGS | _abi.FLAG_PUCT)
    assert _call(lib, puct, ds) == _abi.EAZ_ERR_INVALID_ARG and "EAZ_FLAG_PUCT" in err()
    assert _call(lib, cfg, sq) == _abi.EAZ_ERR_INVALID_ARG and "task_ids" in err()
    assert _call(lib, cfg, ds, T=-1) == _abi.EAZ_ERR_INVALID_ARG and "negative" in err()
    no_beta = _abi.EazSearchInputs(None, None, None, None, None, None, None, C.pointer(ds), None, None)
    assert _call(lib, cfg, ds, inp=no_beta) == _abi.EAZ_ERR_INVALID_ARG and "beta" in err()
    with_obs = _abi.EazState(step_count=FAKE, rewards=FAKE, terminated=FAKE, truncated=FAKE, col=FAKE, observation=FAKE)
    assert _call(lib, cfg, ds, states=with_obs) == _abi.EAZ_ERR_INVALID_ARG and "observation" in err()
    assert _call(lib, cfg, ds, states=_abi.EazState(step_count=FAKE, rewards=FAKE, terminated=FAKE)) == _abi.EAZ_ERR_INVALID_ARG  # needs col
    # T * B rows of max(4 A, S, 16) = 1024 bytes (Subleq-256): 2^31-1 steps x 2^28 envs overflow a 64-bit byte count
    big = _abi.default_search_config(batch=1 << 28, num_simulations=4)
    assert _call(lib, big, sq, T=(1 << 31) - 1, tasks=FAKE) == _abi.EAZ_ERR_INVALID_ARG and "overflows" in err()
    assert _call(lib, cfg, ds, ws_bytes=1024) == _abi.EAZ_ERR_WORKSPACE
    assert _call(lib, cfg, ds, ws=C.c_void_p(0x200010)) == _abi.EAZ_ERR_WORKSPACE and "256-byte aligned" in err()
    assert _call(lib, cfg, ds, ws=None) == _abi.EAZ_ERR_WORKSPACE
    # a scan of length 0 passes every check and enqueues nothing (no device exists here, and the pointers are fake)
    assert _call(lib, cfg, ds, T=0) == 0
    assert _call(lib, cfg, sq, T=0, tasks=FAKE) == 0


def test_shim_selfplay_handler_validates(lib):
    from tests.xla_ffi_stub import harness as X

    shim = X.load()  # (builds the shim with -Wall -Werror against the stand-in)
    assert hasattr(shim, "EazSelfplay")
    f = lambda *d: X.buf("f32", None, *d)
    i = lambda *d: X.buf("s32", None, *d)
    B, T, A = 4, 3, 2
    leaves = [i(B), f(B, 1), X.buf("pred", None, B), X.buf("pred", None, B), i(B)]
    params = [f(100, 8), f(8)] * 12  # w, b per layer: D = 100, hidden 8
    attrs = dict(env_kind=_abi.ENV_DEEPSEA, size=10, word_size=0, binary_encoding=0, reward_fn=0, num_simulations=4, max_depth=0,
                 max_num_considered_actions=16, gumbel_scale=1.0, discount=0.97, two_players_game=0, exploration=0, value_scale=0.1,
                 maxvisit_init=50.0, rescale_values=1, flags=7, mlp_mode=0, hash_bits=24, hash_io=0, max_u=1.0, novelty_scale=1.0, steps=T,
                 root_prior=0, action_sampling=0, temperature=1.0, noise_seed=0, reuse_prepared=0)
    args = [f(B), X.buf("u8", None, 10, 10), X.buf("u8", None, 1 << 21), f(T, B, A), f(1), i(1), X.buf("u8", None, 1)]
    stacked = [i(T, B), f(T, B), f(T, B), f(T, B), f(T, B), f(T, B, A), i(T, B, 4), X.buf("u8", None, T, B, 4), f(T, B)]
    rets = leaves + stacked + [X.buf("u8", None, 1)]

    def call(a=args, r=rets, at=attrs):
        return X.call(shim, "EazSelfplay", a + leaves + params, r, at)

    rc, msg = X.call(shim, "EazSelfplay", args + leaves + params[:23], rets, attrs)
    assert rc == 3 and "24 parameter buffers" in msg, msg
    rc, msg = call(r=rets[:-1])
    assert rc == 3 and "stacked outputs" in msg, msg
    rc, msg = call(at={k: v for k, v in attrs.items() if k != "steps"})
    assert rc == 3 and "steps" in msg, msg
    rc, msg = call(at=dict(attrs, steps=-1))
    assert rc == 3 and "steps must be >= 0" in msg, msg
    rc, msg = call(a=args[:3] + [f(T, B, A + 1)] + args[4:])
    assert rc == 3 and "gumbel must be" in msg, msg
    rc, msg = call(a=args[:5] + [i(T, B + 1)] + args[6:])
    assert rc == 3 and "task_ids must be" in msg, msg
    rc, msg = call(r=leaves + stacked[:5] + [f(T, B, A - 1)] + stacked[6:] + [X.buf("u8", None, 1)])
    assert rc == 3 and "q_values_epistemic_variance" in msg, msg
    rc, msg = call()  # a 1-byte workspace result
    assert rc == 3 and "eaz_selfplay_workspace_bytes" in msg, msg
