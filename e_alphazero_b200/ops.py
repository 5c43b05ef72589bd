"""Thin torch-tensor harness over the C ABI (include/eaz_b200.h).

Tensors supply device pointers and the current CUDA stream; all arithmetic runs
in libeaz_b200.so.  States are dicts of device tensors named like the pgx.State
leaves (``step_count, rewards, terminated, truncated, col | memory, task, solved,
input_after, output_after`` and optionally ``observation``).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

from . import _abi
from ._lib import EazError, check, load, require_cuda

_TORCH_DT = None


def _dt():
    global _TORCH_DT
    if _TORCH_DT is None:
        import torch

        _TORCH_DT = {"i32": torch.int32, "f32": torch.float32, "u8": torch.uint8}
    return _TORCH_DT


def _ptr(t, dtype=None):
    if t is None:
        return None
    if not t.is_cuda:
        raise EazError("expected a CUDA tensor (the C ABI takes device pointers)")
    if not t.is_contiguous():
        raise EazError("expected a contiguous tensor")
    if dtype is not None and t.dtype != dtype:
        raise EazError(f"expected dtype {dtype}, got {t.dtype}")
    return C.c_void_p(t.data_ptr())


def _stream():
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# --------------------------------------------------------------------------- env
@dataclass
class EnvSpec:
    """Static attributes of the pgx.Env instance (deep_sea.py:37-52, subleq.py:599-621)."""

    kind: int
    size: int = 0
    action_map: object = None  # device uint8 [N,N] or None
    word_size: int = 0
    binary_encoding: int = 1
    reward_fn: int = _abi.SUBLEQ_REWARD_SOLVED

    def struct(self) -> _abi.EazEnv:
        return _abi.EazEnv(self.kind, self.size, _ptr(self.action_map), self.word_size, self.binary_encoding, self.reward_fn)

    def _q(self, fn, *a):
        s = self.struct()
        v = getattr(load(), fn)(C.byref(s), *a)
        if v < 0:
            check(-1, fn)
        return v

    @property
    def num_actions(self):
        return self._q("eaz_env_num_actions")

    @property
    def obs_dim(self):
        return self._q("eaz_env_obs_dim")

    @property
    def obs_cols(self):
        return self._q("eaz_env_obs_cols")

    @property
    def compact_bytes(self):
        return self._q("eaz_env_compact_bytes")

    def hash_dim(self, hash_io):
        return self._q("eaz_env_hash_dim", int(hash_io))

    @property
    def obs_shape(self):
        if self.kind == _abi.ENV_DEEPSEA:
            return (self.size, self.size)
        return (self.word_size + 32, self.obs_cols)


def deepsea_spec(size, action_map=None, device="cuda") -> EnvSpec:
    torch = require_cuda()
    am = None
    if action_map is not None:
        am = torch.as_tensor(action_map).to(device=device, dtype=torch.uint8).reshape(size, size).contiguous()
    return EnvSpec(_abi.ENV_DEEPSEA, size=size, action_map=am)


def subleq_spec(word_size, binary_encoding=True, reward_fn=_abi.SUBLEQ_REWARD_SOLVED) -> EnvSpec:
    return EnvSpec(_abi.ENV_SUBLEQ, word_size=word_size, binary_encoding=int(binary_encoding), reward_fn=reward_fn)


_STATE_SHAPES = {
    "step_count": ("i32", lambda e: ()),
    "rewards": ("f32", lambda e: (1,)),
    "terminated": ("u8", lambda e: ()),
    "truncated": ("u8", lambda e: ()),
    "col": ("i32", lambda e: ()),
    "memory": ("i32", lambda e: (e.word_size,)),
    "task": ("i32", lambda e: ()),
    "solved": ("u8", lambda e: ()),
    "input_after": ("i32", lambda e: (8,)),
    "output_after": ("i32", lambda e: (8,)),
}
DEEPSEA_FIELDS = ["step_count", "rewards", "terminated", "truncated", "col"]
SUBLEQ_FIELDS = ["step_count", "rewards", "terminated", "truncated", "memory", "task", "solved", "input_after", "output_after"]


def state_fields(env: EnvSpec):
    return DEEPSEA_FIELDS if env.kind == _abi.ENV_DEEPSEA else SUBLEQ_FIELDS


def alloc_state(env: EnvSpec, B: int, with_obs=False, device="cuda") -> dict:
    torch = require_cuda()
    st = {}
    for name in state_fields(env):
        dt, shp = _STATE_SHAPES[name]
        st[name] = torch.zeros((B,) + shp(env), dtype=_dt()[dt], device=device)
    if with_obs:
        st["observation"] = torch.zeros((B, env.obs_dim), dtype=torch.uint8, device=device)
    return st


def state_to_device(env: EnvSpec, st: dict, device="cuda") -> dict:
    """Upload a host (numpy) state dict."""
    torch = require_cuda()
    out = {}
    for name in state_fields(env):
        dt, _ = _STATE_SHAPES[name]
        out[name] = torch.as_tensor(st[name]).to(device=device, dtype=_dt()[dt]).contiguous()
    return out


def state_struct(env: EnvSpec, st: dict) -> _abi.EazState:
    s = _abi.EazState()
    for name in state_fields(env):
        dt, _ = _STATE_SHAPES[name]
        setattr(s, name, _ptr(st[name], _dt()[dt]))
    if st.get("observation") is not None:
        s.observation = _ptr(st["observation"], _dt()["u8"])
    return s


def _batch(st):
    return st["step_count"].shape[0]


def _tasks(task_ids, B, device):
    torch = require_cuda()
    if task_ids is None:
        return None
    t = torch.as_tensor(task_ids).to(device=device, dtype=torch.int32).contiguous()
    if t.numel() != B:
        raise EazError("task_ids must have one entry per env")
    return t


def env_init(env: EnvSpec, B: int, task_ids=None, with_obs=False, device="cuda") -> dict:
    """vmap(env.init): deep_sea.py:54-57 / subleq.py:623-646 (task ids pre-drawn)."""
    st = alloc_state(env, B, with_obs, device)
    t = _tasks(task_ids, B, device)
    e, s = env.struct(), state_struct(env, st)
    check(load().eaz_env_init(C.byref(e), _ptr(t), C.byref(s), B, _stream()), "eaz_env_init")
    return st


def env_step_(env: EnvSpec, st: dict, action, auto_reset=False, task_ids=None) -> dict:
    """In-place vmap(env.step) (or the reference's auto_reset wrapper, selfplay.py:26-75)."""
    torch = require_cuda()
    B = _batch(st)
    a = torch.as_tensor(action).to(device=st["step_count"].device, dtype=torch.int32).contiguous()
    t = _tasks(task_ids, B, st["step_count"].device)
    e, s = env.struct(), state_struct(env, st)
    check(load().eaz_env_step(C.byref(e), C.byref(s), _ptr(a), int(auto_reset), _ptr(t), B, _stream()), "eaz_env_step")
    return st


def env_step(env: EnvSpec, st: dict, action, auto_reset=False, task_ids=None) -> dict:
    return env_step_(env, {k: v.clone() for k, v in st.items()}, action, auto_reset, task_ids)


def env_observe(env: EnvSpec, st: dict):
    torch = require_cuda()
    B = _batch(st)
    obs = torch.empty((B, env.obs_dim), dtype=torch.uint8, device=st["step_count"].device)
    e, s = env.struct(), state_struct(env, st)
    check(load().eaz_env_observe(C.byref(e), C.byref(s), _ptr(obs), B, _stream()), "eaz_env_observe")
    return obs


def env_compact(env: EnvSpec, st: dict):
    torch = require_cuda()
    B = _batch(st)
    out = torch.empty((B, env.compact_bytes), dtype=torch.uint8, device=st["step_count"].device)
    e, s = env.struct(), state_struct(env, st)
    check(load().eaz_env_compact(C.byref(e), C.byref(s), _ptr(out), B, _stream()), "eaz_env_compact")
    return out


def env_uncompact(env: EnvSpec, compact, rewards=None, with_obs=False, out: dict | None = None) -> dict:
    """eaz_env_uncompact: compact records [B,S] (+ rewards [B]) -> state dict (the decode step of the compact replay ring)."""
    torch = require_cuda()
    B = compact.shape[0]
    st = out if out is not None else alloc_state(env, B, with_obs=with_obs, device=str(compact.device))
    e, s = env.struct(), state_struct(env, st)
    r = None if rewards is None else rewards.reshape(B).to(torch.float32).contiguous()
    check(load().eaz_env_uncompact(C.byref(e), _ptr(compact.contiguous(), torch.uint8), _ptr(r, torch.float32), C.byref(s), B, _stream()),
          "eaz_env_uncompact")
    return st


def trajectory_pack(env: EnvSpec, st: dict, action, out=None):
    """eaz_trajectory_pack: int32 [B,4] replay records {action, reward bits, flags, first compact-state word} in one kernel."""
    torch = require_cuda()
    B = _batch(st)
    if out is None:
        out = torch.empty((B, 4), dtype=torch.int32, device=st["step_count"].device)
    e, s = env.struct(), state_struct(env, st)
    check(load().eaz_trajectory_pack(C.byref(e), C.byref(s), _ptr(action, torch.int32), _ptr(out, torch.int32), B, _stream()), "eaz_trajectory_pack")
    return out


# --------------------------------------------------------------------------- prioritised replay (csrc/replay.cu)
def priority_tree_bytes(T: int, B: int) -> int:
    n = load().eaz_priority_tree_bytes(int(T), int(B))
    if n == 0:
        check(-1, "eaz_priority_tree_bytes")
    return int(n)


def priority_init(tree, T: int, B: int, priority_exponent: float, seed: int = 0) -> None:
    """eaz_priority_init on a uint8 device buffer of priority_tree_bytes(T, B)."""
    check(load().eaz_priority_init(_ptr(tree), C.c_size_t(tree.numel()), int(T), int(B), C.c_float(priority_exponent), C.c_uint32(seed),
                                   _stream()), "eaz_priority_init")


def priority_add_step(tree, T: int, B: int, slot: int) -> None:
    check(load().eaz_priority_add_step(_ptr(tree), C.c_size_t(tree.numel()), int(T), int(B), int(slot), _stream()), "eaz_priority_add_step")


def priority_set(tree, T: int, B: int, indices, priorities) -> None:
    """eaz_priority_set: indices int32 [K], priorities float32 [K], both contiguous device tensors."""
    import torch

    if indices.numel() != priorities.numel():
        raise EazError("set_priorities: indices and priorities differ in length")
    check(load().eaz_priority_set(_ptr(tree), C.c_size_t(tree.numel()), int(T), int(B), _ptr(indices, torch.int32), _ptr(priorities, torch.float32),
                                  int(indices.numel()), _stream()), "eaz_priority_set")


def priority_sample(tree, T: int, B: int, indices, probabilities, states=None, rewards=None, first=None, first_rewards=None, second=None,
                    second_rewards=None) -> None:
    """eaz_priority_sample: K = indices.numel() draws into the given buffers; with `states` ([T,B,S] uint8) the compact records
    (and with `rewards` [T,B] the rewards) of both slots of every drawn pair are gathered into first / second [K,S]."""
    import torch

    S = 0 if states is None else states.shape[-1]
    check(load().eaz_priority_sample(_ptr(tree), C.c_size_t(tree.numel()), int(T), int(B), int(indices.numel()), _ptr(states, torch.uint8),
                                     _ptr(rewards, torch.float32), S, _ptr(indices, torch.int32), _ptr(probabilities, torch.float32),
                                     _ptr(first, torch.uint8), _ptr(first_rewards, torch.float32), _ptr(second, torch.uint8),
                                     _ptr(second_rewards, torch.float32), _stream()), "eaz_priority_sample")


def priority_status(tree) -> int:
    """eaz_priority_status: synchronises; raises EazError if a sticky EAZ_PRIORITY_* bit is set, else returns 0."""
    flags = C.c_int32(0)
    check(load().eaz_priority_status(_ptr(tree), C.c_size_t(tree.numel()), _stream(), C.byref(flags)), "eaz_priority_status")
    return int(flags.value)


def replay_add(env: EnvSpec, st: dict, ring_states, ring_rewards, tree) -> None:
    """eaz_replay_add: one time step of `st` into ring row `cursor` of ring_states [T,B,S] / ring_rewards [T,B], with the cursor read
    and advanced on the device (no host copy of it exists, so a captured call appends at the current cursor on every replay)."""
    import torch

    T, B = ring_states.shape[0], ring_states.shape[1]
    if _batch(st) != B or tuple(ring_rewards.shape) != (T, B) or ring_states.shape[2] != env.compact_bytes:
        raise EazError("replay_add: ring_states must be [T, B, compact_bytes] and ring_rewards [T, B] for the B envs of the state")
    e, s = env.struct(), state_struct(env, st)
    check(load().eaz_replay_add(C.byref(e), C.byref(s), _ptr(ring_states, torch.uint8), _ptr(ring_rewards, torch.float32), _ptr(tree),
                                C.c_size_t(tree.numel()), int(T), int(B), _stream()), "eaz_replay_add")


def priority_sample_keyed(tree, T: int, B: int, key, indices, probabilities, states=None, rewards=None, first=None, first_rewards=None,
                          second=None, second_rewards=None) -> None:
    """eaz_priority_sample_keyed: as priority_sample with (seed, draw counter) = key, a uint32-valued int32 [2] device tensor; the
    tree is only read."""
    import torch

    if key.numel() != 2:
        raise EazError("priority_sample_keyed: key must hold two 32-bit words")
    S = 0 if states is None else states.shape[-1]
    check(load().eaz_priority_sample_keyed(_ptr(tree), C.c_size_t(tree.numel()), int(T), int(B), int(indices.numel()), _ptr(key, torch.int32),
                                           _ptr(states, torch.uint8), _ptr(rewards, torch.float32), S, _ptr(indices, torch.int32),
                                           _ptr(probabilities, torch.float32), _ptr(first, torch.uint8), _ptr(first_rewards, torch.float32),
                                           _ptr(second, torch.uint8), _ptr(second_rewards, torch.float32), _stream()),
          "eaz_priority_sample_keyed")


def priority_status_async(tree, flags) -> None:
    """eaz_priority_status_async: the sticky EAZ_PRIORITY_* word into the int32 [1] device tensor `flags`, without synchronising."""
    import torch

    check(load().eaz_priority_status_async(_ptr(tree), C.c_size_t(tree.numel()), _ptr(flags, torch.int32), _stream()), "eaz_priority_status_async")


def subleq_test_cases(task: int, ws: int):
    import numpy as np

    i, o = np.zeros((3, 8), np.int32), np.zeros((3, 8), np.int32)
    check(load().eaz_subleq_test_cases(int(task), int(ws), i.ctypes.data_as(C.c_void_p), o.ctypes.data_as(C.c_void_p)), "eaz_subleq_test_cases")
    return i, o


# --------------------------------------------------------------------------- hash
def _rows_f32(x):
    torch = require_cuda()
    if x.dtype != torch.float32:
        x = x.to(torch.float32)
    return x.reshape(x.shape[0], -1).contiguous()


def xxhash_indices(x, bits=24):
    """XXHash.get_indices (hashes.py:162-229)."""
    torch = require_cuda()
    x = _rows_f32(x)
    out = torch.empty(x.shape[0], dtype=torch.int32, device=x.device)  # uint32 payload
    check(load().eaz_xxhash_indices(_ptr(x), x.shape[0], x.shape[1], int(bits), _ptr(out), _stream()), "eaz_xxhash_indices")
    return out


def hash_lookup(x, binary_set, bits=24):
    """BaseHash.__call__ (hashes.py:29-38)."""
    torch = require_cuda()
    x = _rows_f32(x)
    out = torch.empty(x.shape[0], dtype=torch.uint8, device=x.device)
    check(load().eaz_hash_lookup(_ptr(x), x.shape[0], x.shape[1], int(bits), _ptr(binary_set, torch.uint8), _ptr(out), _stream()), "eaz_hash_lookup")
    return out


def hash_update_(x, binary_set, bits=24):
    """BaseHash.update (hashes.py:45-50), in place."""
    torch = require_cuda()
    x = _rows_f32(x)
    check(load().eaz_hash_update(_ptr(x), x.shape[0], x.shape[1], int(bits), _ptr(binary_set, torch.uint8), _stream()), "eaz_hash_update")
    return binary_set


# --------------------------------------------------------------------------- network
@dataclass
class FcParams:
    """Device copy of the haiku pytree of EpistemicFullyConnectedAZNet: w[h][l] is [in,out], b[h][l] is [out]
    (heads: value, ube, exploit, explore = fc_az_net/linear{,_1..11} in call order) + the hash state."""

    in_dim: int
    hidden: int
    num_actions: int
    w: list
    b: list
    binary_set: object
    hash_bits: int = 24
    hash_io: int = 0
    word_size: int = 0
    max_u: float = 1.0
    novelty_scale: float = 1.0
    version: int = 0  # bumped by whoever rewrites the device tensors through a path torch does not see (context.as_fc_params)

    def content_token(self):
        """Changes whenever the parameters may have changed: `version` plus torch's in-place update counters of every device
        tensor (optimizer steps, copy_, collectives).  Plans compare it to decide whether their parameter-derived tables
        (weight images, novelty table) are still valid."""
        return (self.version, self.hash_bits, self.hash_io, self.max_u, self.novelty_scale,
                tuple((t.data_ptr(), t._version) for row in self.w + self.b for t in row) + ((self.binary_set.data_ptr(), self.binary_set._version),))

    @staticmethod
    def from_numpy(w, b, binary_set, num_actions, hash_bits=24, hash_io=0, word_size=0, max_u=1.0, novelty_scale=1.0, device="cuda"):
        torch = require_cuda()
        tw = [[torch.as_tensor(w[h][l]).to(device=device, dtype=torch.float32).contiguous() for l in range(3)] for h in range(4)]
        tb = [[torch.as_tensor(b[h][l]).to(device=device, dtype=torch.float32).contiguous() for l in range(3)] for h in range(4)]
        bs = torch.as_tensor(binary_set).to(device=device, dtype=torch.uint8).contiguous()
        return FcParams(tw[0][0].shape[0], tw[0][0].shape[1], num_actions, tw, tb, bs, hash_bits, hash_io, word_size, max_u, novelty_scale)

    @staticmethod
    def from_haiku(params: dict, state: dict, num_actions, prefix="fc_az_net", **kw):
        """params: {'fc_az_net/linear_3': {'w','b'}, ...}; state: {'fc_az_net/xxhash32': {'binary_set'}}."""
        names = [f"{prefix}/linear" + ("" if i == 0 else f"_{i}") for i in range(12)]
        w = [[params[names[h * 3 + l]]["w"] for l in range(3)] for h in range(4)]
        b = [[params[names[h * 3 + l]]["b"] for l in range(3)] for h in range(4)]
        return FcParams.from_numpy(w, b, state[f"{prefix}/xxhash32"]["binary_set"], num_actions, **kw)

    def struct(self) -> _abi.EazFcParams:
        import torch

        s = _abi.EazFcParams()
        s.in_dim, s.hidden, s.num_actions = self.in_dim, self.hidden, self.num_actions
        for h in range(4):
            for l in range(3):
                s.w[h][l] = _ptr(self.w[h][l], torch.float32).value
                s.b[h][l] = _ptr(self.b[h][l], torch.float32).value
        s.binary_set = _ptr(self.binary_set, torch.uint8)
        s.hash_bits, s.hash_io, s.word_size = self.hash_bits, self.hash_io, self.word_size
        s.max_u, s.novelty_scale = self.max_u, self.novelty_scale
        return s


def _mlp_out(B, A, device):
    torch = require_cuda()
    f = lambda *s: torch.empty(s, dtype=torch.float32, device=device)
    return dict(exploit_logits=f(B, A), explore_logits=f(B, A), value=f(B), ube=f(B), novelty=f(B))


def mlp_forward(net: FcParams, observation) -> dict:
    """forward.apply(params, state, observation, is_training=False) on a bool observation batch."""
    torch = require_cuda()
    obs = observation.to(torch.uint8).reshape(observation.shape[0], -1).contiguous()
    B = obs.shape[0]
    out = _mlp_out(B, net.num_actions, obs.device)
    s = net.struct()
    check(load().eaz_mlp_forward(C.byref(s), _ptr(obs), B, _ptr(out["exploit_logits"]), _ptr(out["explore_logits"]), _ptr(out["value"]),
                                 _ptr(out["ube"]), _ptr(out["novelty"]), _stream()), "eaz_mlp_forward")
    return out


def mlp_forward_states(net: FcParams, env: EnvSpec, st: dict) -> dict:
    """Same network, observation derived on the fly from env states."""
    torch = require_cuda()
    B = _batch(st)
    dev = st["step_count"].device
    out = _mlp_out(B, net.num_actions, dev)
    ws = torch.empty(max(B * env.compact_bytes, 16), dtype=torch.uint8, device=dev)
    s, e, ss = net.struct(), env.struct(), state_struct(env, st)
    check(load().eaz_mlp_forward_states(C.byref(s), C.byref(e), C.byref(ss), B, _ptr(out["exploit_logits"]), _ptr(out["explore_logits"]),
                                        _ptr(out["value"]), _ptr(out["ube"]), _ptr(out["novelty"]), _ptr(ws), C.c_size_t(ws.numel()),
                                        _stream()), "eaz_mlp_forward_states")
    return out


# --------------------------------------------------------------------------- convolutional evaluators
class ConvNetParams:
    """EpistemicResidualAZNet / EpistemicMinatarAZNet (network/resnet.py, network/minatar.py) as device tensors.
    `desc`: _abi.convnet_description(params, state, ...) -- numpy / torch leaves are uploaded once."""

    def __init__(self, desc: dict, device="cuda"):
        torch = require_cuda()
        self._keep = []

        def up(x):
            if isinstance(x, dict):
                return {k: up(v) for k, v in x.items()}
            if isinstance(x, (list, tuple)):
                return [up(v) for v in x]
            if hasattr(x, "shape") and not isinstance(x, (int, float)):
                t = torch.as_tensor(x)
                t = t.to(device=device, dtype=torch.uint8 if t.dtype == torch.uint8 else torch.float32).contiguous()
                self._keep.append(t)
                return t
            return x

        self.desc = up(desc)
        self.device = device
        self.struct = _abi.fill_convnet_params(self.desc, lambda t: C.c_void_p(t.data_ptr()))
        self.num_actions = int(desc["num_actions"])

    def forward(self, observation) -> dict:
        """forward.apply(params, state, observation, is_training=False): observation bool [B,H,W,C] on the device."""
        torch = require_cuda()
        obs = observation.to(torch.uint8).reshape(observation.shape[0], -1).contiguous()
        B = obs.shape[0]
        out = _mlp_out(B, self.num_actions, obs.device)
        nbytes = load().eaz_convnet_workspace_bytes(C.byref(self.struct), B)
        if nbytes == 0:
            raise EazError("eaz_convnet_workspace_bytes rejected the configuration: " + load().eaz_last_error().decode())
        ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=obs.device)
        off = (-ws.data_ptr()) % 256
        self._last = (ws, C.c_void_p(ws.data_ptr() + off), C.c_size_t(nbytes), B)
        check(load().eaz_convnet_forward(C.byref(self.struct), _ptr(obs), B, _ptr(out["exploit_logits"]), _ptr(out["explore_logits"]), _ptr(out["value"]),
                                         _ptr(out["ube"]), _ptr(out["novelty"]), self._last[1], self._last[2], _stream()), "eaz_convnet_forward")
        return out

    def numeric_status(self) -> int:
        """eaz_convnet_numeric_status on the workspace of the last forward(): raises EazError if the tensor-core path left its range."""
        _, ptr, nbytes, B = self._last
        flags = C.c_int32(0)
        check(load().eaz_convnet_numeric_status(C.byref(self.struct), B, ptr, nbytes, _stream(), C.byref(flags)), "eaz_convnet_numeric_status")
        return int(flags.value)


# --------------------------------------------------------------------------- search
def alloc_arena(specs, device="cuda", pinned=False):
    """One flat uint8 allocation holding every tensor of `specs` = [(name, shape, torch dtype)] at 256-byte aligned offsets;
    returns (flat, {name: view}).  A host caller moves ALL of them with one copy of `flat` (a pinned host arena built from the
    same specs has the same layout) instead of one small cudaMemcpy per tensor."""
    import math

    import torch

    offs, total = [], 0
    for _, shape, dt in specs:
        nbytes = int(math.prod(shape)) * torch.empty((), dtype=dt).element_size()
        offs.append((total, nbytes))
        total += (nbytes + 255) // 256 * 256
    flat = torch.zeros(max(total, 256), dtype=torch.uint8, device=device)
    if pinned:
        flat = flat.pin_memory()
    views = {name: flat[off : off + nb].view(dt).view(shape) for (name, shape, dt), (off, nb) in zip(specs, offs)}
    return flat, views


def search_output_specs(B, N, A, S, want_tree):
    shp = {"B": (B,), "BA": (B, A), "BN": (B, N), "BNA": (B, N, A), "BNS": (B, N, S)}
    fields = _abi.SUMMARY_FIELDS + (_abi.TREE_FIELDS if want_tree else []) + _abi.ROOT_FIELDS
    return [(name, shp[kind], _dt()[dt]) for name, dt, kind in fields]


def alloc_search_outputs(B, N, A, S, want_tree, device) -> dict:
    require_cuda()
    return alloc_arena(search_output_specs(B, N, A, S, want_tree), device)[1]


@dataclass
class SearchPlan:
    """Pre-allocated workspace + outputs for repeated searches of one shape (no allocation in the hot loop)."""

    cfg: _abi.EazSearchConfig
    env: EnvSpec
    net: FcParams
    want_tree: bool = False
    device: str = "cuda"
    workspace: object = None
    out: dict = field(default_factory=dict)
    out_flat: object = None
    out_specs: object = None
    num_launches: int = 0
    num_launches_reuse: int = 0

    def __post_init__(self):
        torch = require_cuda()
        e = self.env.struct()
        nbytes = load().eaz_search_workspace_bytes(C.byref(self.cfg), C.byref(e))
        if nbytes == 0:
            raise EazError("eaz_search_workspace_bytes rejected the configuration")
        self.workspace = torch.empty(nbytes + 256, dtype=torch.uint8, device=self.device)
        off = (-self.workspace.data_ptr()) % 256
        self._ws_ptr = C.c_void_p(self.workspace.data_ptr() + off)
        self._ws_bytes = C.c_size_t(nbytes)
        B, N, A = self.cfg.batch, self.cfg.num_simulations + 1, self.env.num_actions
        # all outputs in one arena: `out_flat` moves them to the host with one copy (alloc_arena)
        self.out_specs = search_output_specs(B, N, A, self.env.compact_bytes, self.want_tree)
        self.out_flat, self.out = alloc_arena(self.out_specs, self.device)
        self.num_launches = load().eaz_search_num_launches(C.byref(self.cfg), C.byref(e))
        cfg_reuse = _abi.EazSearchConfig.from_buffer_copy(self.cfg)
        cfg_reuse.flags |= _abi.FLAG_REUSE_PREPARED
        self.num_launches_reuse = load().eaz_search_num_launches(C.byref(cfg_reuse), C.byref(e))

    def numeric_status(self) -> int:
        """eaz_search_numeric_status: synchronises, raises EazError if the tensor-core network path left its representable range
        (non-finite weights, clamped hidden activations) since the tables were last rebuilt; returns the flag bits (0)."""
        e = self.env.struct()
        flags = C.c_int32(0)
        check(load().eaz_search_numeric_status(C.byref(self.cfg), C.byref(e), self._ws_ptr, self._ws_bytes, _stream(), C.byref(flags)),
              "eaz_search_numeric_status")
        return int(flags.value)

    PROFILE_CLASSES = ("init", "select", "env_step", "network", "expand_backward", "finalize", "export")

    def run(self, root: dict, profile: bool = False, reuse_prepared: bool | None = False):
        """root: prior_logits [B,A], value [B], value_epistemic_variance [B], beta [B], embedding (state dict),
        gumbel [B,A] pre-drawn standard Gumbel noise (absent / None: drawn inside the search from cfg.noise_seed and the
        workspace's draw counter), optional invalid_actions [B,A] (bool/uint8), optional sample_gumbel [B,A]: the noise of the
        action draw of cfg.action_sampling (absent / None: drawn inside the search like `gumbel`).

        The returned tensors are THIS PLAN'S buffers: the next run() overwrites them (clone what must survive).
        reuse_prepared: False = rebuild the parameter-derived tables, True = the caller promises env / net are unchanged,
        None = decide from `net.content_token()` (rebuild only when the parameters changed since the last run)."""
        import torch

        f32, u8 = torch.float32, torch.uint8
        inv = root.get("invalid_actions")
        if inv is not None and inv.dtype != u8:
            inv = inv.to(u8)
        e, n, s = self.env.struct(), self.net.struct(), state_struct(self.env, root["embedding"])
        inp = _abi.EazSearchInputs(_ptr(root.get("prior_logits"), f32), _ptr(root.get("value"), f32), _ptr(root.get("value_epistemic_variance"), f32),
                                   _ptr(root["beta"], f32), C.pointer(s), _ptr(inv), _ptr(root.get("gumbel"), f32), C.pointer(e), C.pointer(n),
                                   _ptr(root.get("sample_gumbel"), f32))
        o = _abi.EazSearchOutputs()
        for name, _, _ in _abi.SEARCH_OUTPUT_FIELDS:
            setattr(o, name, _ptr(self.out.get(name)))
        # parameter-derived tables (seq-halving table, seen table, weight images) live in the workspace across runs
        # (reuse_prepared=True is the caller's promise that env / net are unchanged since an earlier run on this plan)
        cfg = _abi.EazSearchConfig.from_buffer_copy(self.cfg)
        if reuse_prepared is None:
            tok = (self.net.content_token(), None if self.env.action_map is None else (self.env.action_map.data_ptr(), self.env.action_map._version))
            reuse_prepared = getattr(self, "_prepared", False) and getattr(self, "_prepared_token", None) == tok
            self._prepared_token = tok
        else:
            self._prepared_token = None
        if reuse_prepared:
            if not getattr(self, "_prepared", False):
                raise EazError("reuse_prepared=True before any search built the tables in this plan's workspace")
            cfg.flags |= _abi.FLAG_REUSE_PREPARED
        self._prepared = True
        if profile:  # measurement aid: synchronises; returns (outputs, {class: (ms, launches)})
            ms = (C.c_float * len(self.PROFILE_CLASSES))()
            cnt = (C.c_int32 * len(self.PROFILE_CLASSES))()
            check(load().eaz_search_gumbel_profiled(C.byref(cfg), C.byref(inp), C.byref(o), self._ws_ptr, self._ws_bytes, _stream(), ms, cnt),
                  "eaz_search_gumbel_profiled")
            return self.out, {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(self.PROFILE_CLASSES)}
        check(load().eaz_search_gumbel(C.byref(cfg), C.byref(inp), C.byref(o), self._ws_ptr, self._ws_bytes, _stream()), "eaz_search_gumbel")
        return self.out


def reanalyze_targets(discount, exploration_beta, exploration_ube_target, temperature, action, qvalues, qvalues_epistemic_variance, visit_counts,
                      value, value_epistemic_std, next_state_value, next_rewards, next_terminated, terminated, invalid_actions=None, out=None) -> dict:
    """eaz_reanalyze_targets (reanalyze.py:86-129) on device tensors; `out` may hold pre-allocated result tensors."""
    torch = require_cuda()
    f32, u8, i32 = torch.float32, torch.uint8, torch.int32
    B, A = qvalues.shape
    dev = qvalues.device
    if out is None:
        out = dict(value_target=torch.empty(B, dtype=f32, device=dev), ube_target=torch.empty(B, dtype=f32, device=dev),
                   exploration_policy_target=torch.empty((B, A), dtype=f32, device=dev))
    cfg = _abi.EazReanalyzeConfig(float(discount), float(exploration_beta), int(bool(exploration_ube_target)), float(temperature))
    c = lambda t, dt: t.to(dtype=dt).contiguous()
    keep = [c(action, i32), c(qvalues, f32), c(qvalues_epistemic_variance, f32), c(visit_counts, f32), c(value, f32), c(value_epistemic_std, f32),
            c(next_state_value, f32), c(next_rewards.reshape(B), f32), c(next_terminated, u8), c(terminated, u8),
            c(invalid_actions, u8) if invalid_actions is not None else None]
    check(load().eaz_reanalyze_targets(C.byref(cfg), B, A, *[_ptr(k) for k in keep], _ptr(out["value_target"], f32), _ptr(out["ube_target"], f32),
                                       _ptr(out["exploration_policy_target"], f32), _stream()), "eaz_reanalyze_targets")
    return out


def search(cfg: _abi.EazSearchConfig, env: EnvSpec, net: FcParams, root: dict, want_tree=False) -> dict:
    cfg.batch = root["gumbel"].shape[0]
    plan = SearchPlan(cfg, env, net, want_tree, device=str(root["gumbel"].device))
    return plan.run(root)
