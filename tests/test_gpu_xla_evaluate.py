"""EazEvaluate of csrc/xla_ffi_shim.cc, driven through the stand-in call frame of tests/xla_ffi_stub/ with device buffers: the episodes
a JAX caller gets must be bit-identical to eaz_evaluate called directly."""
import pytest

from e_alphazero_b200 import _abi
from tests import helpers as H

pytestmark = pytest.mark.gpu

LEAVES = {_abi.ENV_DEEPSEA: ["step_count", "rewards", "terminated", "truncated", "col"],
          _abi.ENV_SUBLEQ: ["step_count", "rewards", "terminated", "truncated", "memory", "task", "solved", "input_after", "output_after"]}


@pytest.mark.parametrize("kind,kw,B,n,mode,max_len", [("deepsea", dict(size=10), 130, 16, _abi.MLP_TENSOR, 50),
                                                      ("deepsea", dict(size=10), 64, 8, _abi.MLP_EXACT, 4),
                                                      ("subleq", dict(word_size=16), 70, 12, _abi.MLP_EXACT, 50)])
def test_shim_evaluate_equals_abi(kind, kw, B, n, mode, max_len):
    import torch

    from e_alphazero_b200 import _lib, ops
    from tests.xla_ffi_stub import harness as X

    assert torch.cuda.is_available()
    lib = X.load()
    env = H.make_env(kind, seed=301, **kw)
    net = H.make_net(env, seed=302, fill=0.5)
    denv, dnet = H.device_env(env), H.device_net(net)
    tasks = torch.tensor([1, 2, 3] * B, dtype=torch.int32, device="cuda")[:B].contiguous() if kind == "subleq" else None
    init = ops.env_init(denv, B, task_ids=tasks)
    beta = torch.linspace(0, 0.5, B, device="cuda")
    cfg = _abi.default_search_config(batch=B, num_simulations=n, discount=0.97, gumbel_scale=0.0, mlp_mode=mode)

    plan = ops.EvaluatePlan(cfg, denv, dnet)
    direct_states = {k: v.clone() for k, v in init.items()}
    direct_returns = torch.full((B,), float("nan"), device="cuda")
    plan.run(beta, direct_states, direct_returns, max_len)

    import ctypes as C

    ws_bytes = _lib.load().eaz_evaluate_workspace_bytes(C.byref(cfg), C.byref(denv.struct())) + 256
    ws = torch.zeros(ws_bytes, dtype=torch.uint8, device="cuda")
    dummy = torch.zeros(1, dtype=torch.uint8, device="cuda")
    amap = denv.action_map if denv.action_map is not None else dummy
    params = [t for h in range(4) for l in range(3) for t in (dnet.w[h][l], dnet.b[h][l])]
    leaves_in = [init[k] for k in LEAVES[env.kind]]
    leaves_out = [torch.zeros_like(t) for t in leaves_in]
    returns = torch.full((B,), float("nan"), device="cuda")
    attrs = dict(env_kind=env.kind, size=env.size if env.kind == _abi.ENV_DEEPSEA else 0, word_size=env.word_size,
                 binary_encoding=int(env.binary_encoding), reward_fn=int(env.reward_fn), num_simulations=n, max_depth=0,
                 max_num_considered_actions=16, discount=0.97, value_scale=0.1, maxvisit_init=50.0, rescale_values=1,
                 flags=_abi.SEARCH_DEFAULT_FLAGS, mlp_mode=mode, hash_bits=net.hash_bits, hash_io=net.hash_io, max_u=1.0, novelty_scale=1.0,
                 max_episode_length=max_len)
    args = [beta, amap, dnet.binary_set, ws] + leaves_in + params
    rets = leaves_out + [returns, ws]
    stream = torch.cuda.current_stream().cuda_stream
    for call in range(2):  # the second call launches the graph the first one built (same buffers)
        returns.fill_(float("nan"))
        rc, msg = X.call(lib, "EazEvaluate", [X.tbuf(t) for t in args], [X.tbuf(t) for t in rets], attrs, stream)
        assert rc == 0, msg
        torch.cuda.synchronize()
        H.assert_same_bits(returns.cpu().numpy(), direct_returns.cpu().numpy(), f"call {call} returns")
        for k, t in zip(LEAVES[env.kind], leaves_out):
            H.assert_same_bits(t.cpu().numpy(), direct_states[k].cpu().numpy(), f"call {call} state {k}")
    for k, t in zip(LEAVES[env.kind], leaves_in):  # the functional form leaves its inputs alone
        H.assert_same_bits(t.cpu().numpy(), init[k].cpu().numpy(), f"input leaf {k}")
    # a workspace result one byte short of eaz_evaluate_workspace_bytes is refused
    short = torch.zeros(ws_bytes - 257, dtype=torch.uint8, device="cuda")
    rc, msg = X.call(lib, "EazEvaluate", [X.tbuf(t) for t in args], [X.tbuf(t) for t in leaves_out + [returns, short]], attrs, stream)
    assert rc == 3 and "workspace" in msg, msg
