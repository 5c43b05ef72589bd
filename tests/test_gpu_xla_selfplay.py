"""EazSelfplay of csrc/xla_ffi_shim.cc, driven through the stand-in call frame of tests/xla_ffi_stub/ with device buffers: the scan a JAX
caller gets -- final state leaves and every stacked output -- must be bit-identical to eaz_selfplay called directly."""
import pytest

from e_alphazero_b200 import _abi
from tests import helpers as H

pytestmark = pytest.mark.gpu

LEAVES = {_abi.ENV_DEEPSEA: ["step_count", "rewards", "terminated", "truncated", "col"],
          _abi.ENV_SUBLEQ: ["step_count", "rewards", "terminated", "truncated", "memory", "task", "solved", "input_after", "output_after"]}


@pytest.mark.parametrize("kind,kw,B,n,mode,T,noise,sampling", [("deepsea", dict(size=10), 130, 16, _abi.MLP_TENSOR, 12, True, _abi.ACTION_SEARCH),
                                                               ("deepsea", dict(size=10), 64, 8, _abi.MLP_EXACT, 5, False, _abi.ACTION_IMPROVED),
                                                               ("subleq", dict(word_size=16), 70, 12, _abi.MLP_EXACT, 16, True, _abi.ACTION_VISITS)])
def test_shim_selfplay_equals_abi(kind, kw, B, n, mode, T, noise, sampling):
    import ctypes as C

    import torch

    from e_alphazero_b200 import _lib, ops
    from tests.xla_ffi_stub import harness as X

    assert torch.cuda.is_available()
    lib = X.load()
    env = H.make_env(kind, seed=501, **kw)
    net = H.make_net(env, seed=502, fill=0.5)
    denv, dnet = H.device_env(env), H.device_net(net)
    A = denv.num_actions
    g = torch.Generator(device="cuda").manual_seed(503)
    tasks = torch.randint(1, 4, (T, B), dtype=torch.int32, device="cuda", generator=g) if kind == "subleq" else None
    init = ops.env_init(denv, B, task_ids=None if tasks is None else tasks[0].contiguous())
    beta = torch.linspace(0, 0.5, B, device="cuda")
    gumbel = -(-torch.rand((T, B, A), device="cuda", generator=g).clamp_(1e-20, 1 - 1e-7).log()).log() if noise else None
    sample = -(-torch.rand((T, B, A), device="cuda", generator=g).clamp_(1e-20, 1 - 1e-7).log()).log() if noise else None
    cfg = _abi.default_search_config(batch=B, num_simulations=n, discount=0.97, mlp_mode=mode, exploration=1, action_sampling=sampling,
                                     temperature=0.8, noise_seed=12345)

    plan = ops.SelfplayPlan(cfg, denv, dnet)
    direct_states = {k: v.clone() for k, v in init.items()}
    direct = ops.alloc_selfplay_outputs(denv, T, B)
    ws_bytes = _lib.load().eaz_selfplay_workspace_bytes(C.byref(cfg), C.byref(denv.struct())) + 256
    ws = torch.zeros(ws_bytes, dtype=torch.uint8, device="cuda")  # (draw counter at 0, as in the plan's fresh workspace)
    dummy_u8 = torch.zeros(1, dtype=torch.uint8, device="cuda")
    amap = denv.action_map if denv.action_map is not None else dummy_u8
    params = [t for h in range(4) for l in range(3) for t in (dnet.w[h][l], dnet.b[h][l])]
    leaves_in = [init[k] for k in LEAVES[env.kind]]
    leaves_out = [torch.zeros_like(t) for t in leaves_in]
    got = ops.alloc_selfplay_outputs(denv, T, B)
    attrs = dict(env_kind=env.kind, size=env.size if env.kind == _abi.ENV_DEEPSEA else 0, word_size=env.word_size,
                 binary_encoding=int(env.binary_encoding), reward_fn=int(env.reward_fn), num_simulations=n, max_depth=0,
                 max_num_considered_actions=16, gumbel_scale=1.0, discount=0.97, two_players_game=0, exploration=1, value_scale=0.1,
                 maxvisit_init=50.0, rescale_values=1, flags=_abi.SEARCH_DEFAULT_FLAGS, mlp_mode=mode, hash_bits=net.hash_bits, hash_io=net.hash_io,
                 max_u=1.0, novelty_scale=1.0, steps=T, root_prior=0, action_sampling=sampling, temperature=0.8, noise_seed=12345, reuse_prepared=0)
    one_f = torch.zeros(1, device="cuda")
    one_i = torch.zeros(1, dtype=torch.int32, device="cuda")
    args = [beta, amap, dnet.binary_set, gumbel if noise else one_f, sample if noise else one_f, tasks if tasks is not None else one_i, ws]
    args += leaves_in + params
    rets = leaves_out + [got[k] for k in ops.SELFPLAY_OUTPUTS] + [ws]
    stream = torch.cuda.current_stream().cuda_stream
    for call in range(2):  # the second call launches the graph the first one built (same buffers) and draws the next in-search noise
        plan.run(beta, direct_states, T, direct, gumbel=gumbel, sample_gumbel=sample, task_ids=tasks, reuse_prepared=call > 0)
        for t in got.values():
            t.fill_(0x5A)
        if call:
            for a, b in zip(leaves_in, leaves_out):
                a.copy_(b)  # continue from the first call's carry
        rc, msg = X.call(lib, "EazSelfplay", [X.tbuf(t) for t in args], [X.tbuf(t) for t in rets], dict(attrs, reuse_prepared=int(call > 0)), stream)
        assert rc == 0, msg
        torch.cuda.synchronize()
        for k in ops.SELFPLAY_OUTPUTS:
            H.assert_same_bits(got[k].cpu().numpy(), direct[k].cpu().numpy(), f"call {call} {k}")
        for k, t in zip(LEAVES[env.kind], leaves_out):
            H.assert_same_bits(t.cpu().numpy(), direct_states[k].cpu().numpy(), f"call {call} state {k}")
    # a workspace result one byte short of eaz_selfplay_workspace_bytes is refused
    short = torch.zeros(ws_bytes - 257, dtype=torch.uint8, device="cuda")
    rc, msg = X.call(lib, "EazSelfplay", [X.tbuf(t) for t in args], [X.tbuf(t) for t in rets[:-1] + [short]], attrs, stream)
    assert rc == 3 and "workspace" in msg, msg
