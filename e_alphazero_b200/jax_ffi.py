"""JAX binding of libeaz_b200 through the XLA FFI handlers of csrc/xla_ffi_shim.cc -- what a maintainer of emcts/e-alphazero
imports in place of `emctx` / `pgx` calls inside the jitted `selfplay` / `reanalyze` / `evaluate` functions.

This module needs `jax` (>= 0.4.38: jax.ffi) and `libeaz_xla_ffi.so` (`make -C e_alphazero_b200/csrc xla_ffi`); neither exists in the
image this repository was developed in, so importing it there raises ImportError -- it is integration text, kept importable-by-design
(no torch, no ctypes calls at import time besides loading the two libraries).  The shim itself is compile-checked and driven in
tests through tests/xla_ffi_stub/.

Call shapes mirror the reference (file:line under /root/reference/src):
    epistemic_gumbel_muzero_policy(...)  selfplay.py:107-117, reanalyze.py:77-85, evaluate.py:36-45  (+ epistemic_summary())
    evaluate(...)                        evaluate.py:13-57 (the whole episode loop: one custom call)
    selfplay(...)                        selfplay.py:78-149 (the whole scan of self-play steps: one custom call)
    env_step(...) / env_init(...)        selfplay.py:26-75,135,161,166
    forward_states(...)                  selfplay.py:89, reanalyze.py:67,90
    reanalyze_targets(...)               reanalyze.py:86-129
    hash_update(...)                     train.py:22 (network/hashes.py:45-50)
    make_prioritised_flat_buffer(...)    main.py:217-225 (init / add / sample / set_priorities: main.py:383-385, 413-414, 454);
                                         add also takes selfplay()'s SelfplayOutput.state, the whole scan in one call
                                         (main.py:383-385 with add_sequences=True)
"""
from __future__ import annotations

import ctypes
import os
from typing import NamedTuple

import numpy as np

try:
    import jax
    import jax.numpy as jnp
except ImportError as e:  # pragma: no cover - jax is absent from the development image
    raise ImportError("e_alphazero_b200.jax_ffi needs jax (the torch-side mirror is e_alphazero_b200.emctx / pgx / context)") from e

_HERE = os.path.dirname(os.path.abspath(__file__))
_eaz = ctypes.CDLL(os.path.join(_HERE, "libeaz_b200.so"), mode=ctypes.RTLD_GLOBAL)
_shim = ctypes.CDLL(os.path.join(_HERE, "libeaz_xla_ffi.so"))
for _name, _sym in (("eaz_search", "EazSearch"), ("eaz_env_step", "EazEnvStep"), ("eaz_env_init", "EazEnvInit"),
                    ("eaz_mlp_forward_states", "EazMlpForwardStates"), ("eaz_reanalyze_targets", "EazReanalyzeTargets"),
                    ("eaz_hash_update", "EazHashUpdate"), ("eaz_evaluate", "EazEvaluate"), ("eaz_selfplay", "EazSelfplay"),
                    ("eaz_replay_init", "EazReplayInit"), ("eaz_replay_add", "EazReplayAdd"), ("eaz_replay_add_sequence", "EazReplayAddSequence"),
                    ("eaz_replay_sample", "EazReplaySample"), ("eaz_replay_set_priorities", "EazReplaySetPriorities"),
                    ("eaz_replay_status", "EazReplayStatus")):
    jax.ffi.register_ffi_target(_name, jax.ffi.pycapsule(getattr(_shim, _sym)), platform="CUDA")

i32, f32 = np.int32, np.float32
ENV_DEEPSEA, ENV_SUBLEQ = 0, 1
DEFAULT_FLAGS = 0b111  # EAZ_SEARCH_DEFAULT_FLAGS


class EnvSpec(NamedTuple):
    """Static description of the pgx.Env instance (eaz_env)."""
    kind: int
    size: int = 0                 # DeepSea.size_of_grid
    action_map: object = None     # DeepSea: bool [N,N]
    word_size: int = 0            # Subleq
    binary_encoding: int = 1
    reward_fn: int = 0

    def attrs(self):
        return dict(env_kind=i32(self.kind), size=i32(self.size), word_size=i32(self.word_size),
                    binary_encoding=i32(self.binary_encoding), reward_fn=i32(self.reward_fn))

    def amap(self):
        return self.action_map if self.kind == ENV_DEEPSEA else jnp.zeros((1,), jnp.uint8)

    @property
    def num_actions(self):
        return 2 if self.kind == ENV_DEEPSEA else self.word_size


def state_leaves(env: EnvSpec, s):
    """pgx.State -> the leaves the library reads, in eaz_state order (deep_sea.py:12-22, subleq.py:545-563)."""
    common = [s._step_count, s.rewards, s.terminated, s.truncated]
    if env.kind == ENV_DEEPSEA:
        return common + [s._horizontal_position]
    return common + [s._memory_state, s._task, s._solved, s._example_input_after, s._example_output_after]


def with_leaves(env: EnvSpec, s, leaves):
    names = ["_step_count", "rewards", "terminated", "truncated"] + (
        ["_horizontal_position"] if env.kind == ENV_DEEPSEA else ["_memory_state", "_task", "_solved", "_example_input_after", "_example_output_after"])
    return s.replace(**dict(zip(names, leaves)))


def param_leaves(params, prefix="fc_az_net"):
    """haiku params -> 24 buffers in module order (fully_connected.py:49-81)."""
    out = []
    for i in range(12):
        mod = params[f"{prefix}/linear" + ("" if i == 0 else f"_{i}")]
        out += [mod["w"], mod["b"]]
    return out


def _workspace_bytes(env: EnvSpec, B, num_simulations, flags, mlp_mode):
    """eaz_search_workspace_bytes at trace time (a host-only ctypes call: shapes are static under jit)."""
    from . import _abi  # ctypes mirrors of the POD structs (no torch)

    cfg = _abi.default_search_config(num_simulations=num_simulations, flags=flags, mlp_mode=mlp_mode)
    cfg.batch = B
    e = _abi.EazEnv(env.kind, env.size, None, env.word_size, env.binary_encoding, env.reward_fn)
    _eaz.eaz_search_workspace_bytes.restype = ctypes.c_size_t
    n = _eaz.eaz_search_workspace_bytes(ctypes.byref(cfg), ctypes.byref(e))
    if n == 0:
        raise ValueError("eaz_search_workspace_bytes rejected the configuration")
    return int(n) + 256


class EpistemicSearchSummary(NamedTuple):  # what selfplay.py:119-142 / reanalyze.py:86-116 read
    value: jax.Array
    value_epistemic_std: jax.Array
    visit_counts: jax.Array
    visit_probs: jax.Array
    qvalues: jax.Array
    qvalues_epistemic_variance: jax.Array


class SearchTreeView(NamedTuple):
    summary: EpistemicSearchSummary
    workspace: jax.Array  # thread it into the next call (`workspace=`) to keep the parameter-derived tables

    def epistemic_summary(self):
        return self.summary


class PolicyOutput(NamedTuple):
    action: jax.Array
    action_weights: jax.Array
    search_tree: SearchTreeView


def epistemic_gumbel_muzero_policy(params, rng_key, root, env: EnvSpec, model_state, *, num_simulations, invalid_actions=None,
                                   discount=0.997, exploration=False, two_players_game=False, rescale_values=True, gumbel_scale=1.0,
                                   max_num_considered_actions=16, flags=DEFAULT_FLAGS, mlp_mode=1, workspace=None, reuse_prepared=False,
                                   hash_io=None, hash_bits=24):
    """Drop-in for the call at selfplay.py:107-117: `recurrent_fn` is not passed -- the library runs the fused
    get_epistemic_recurrent_fn(env, forward, ...) of context.py:109-157 for `env` + the FC network in `params`.
    `root` is the reference's EpistemicRootFnOutput (prior_logits, value, value_epistemic_variance, embedding=states, beta)."""
    B, A = root.prior_logits.shape
    _, gumbel_rng = jax.random.split(rng_key)                       # the split mctx's gumbel_muzero_policy performs
    gumbel = jax.random.gumbel(gumbel_rng, (B, A), jnp.float32)     # pre-drawn: the kernel takes the noise, not the key
    inv = jnp.zeros((1,), jnp.bool_) if invalid_actions is None else invalid_actions
    ws_bytes = _workspace_bytes(env, B, num_simulations, flags, mlp_mode)
    ws_in = jnp.zeros((ws_bytes,), jnp.uint8) if workspace is None else workspace
    fB, fBA = jax.ShapeDtypeStruct((B,), jnp.float32), jax.ShapeDtypeStruct((B, A), jnp.float32)
    out_types = [jax.ShapeDtypeStruct((B,), jnp.int32), fBA, fB, fB, fBA, fBA, fBA, fBA, fB, fB, jax.ShapeDtypeStruct((ws_bytes,), jnp.uint8)]
    binary_set = model_state["fc_az_net/xxhash32"]["binary_set"]
    args = [root.beta, gumbel, inv, env.amap(), binary_set, root.prior_logits, root.value, root.value_epistemic_variance, ws_in,
            *state_leaves(env, root.embedding), *param_leaves(params)]
    call = jax.ffi.ffi_call("eaz_search", out_types, input_output_aliases={8: 10})  # workspace_in -> workspace (donated)
    action, weights, value, std, counts, probs, q, qvar, _rv, _ru, ws = call(
        *args, **env.attrs(), num_simulations=i32(num_simulations), max_depth=i32(0), max_num_considered_actions=i32(max_num_considered_actions),
        gumbel_scale=f32(gumbel_scale), discount=f32(discount), two_players_game=i32(two_players_game), exploration=i32(exploration),
        value_scale=f32(0.1), maxvisit_init=f32(50.0), rescale_values=i32(rescale_values), flags=i32(flags), mlp_mode=i32(mlp_mode),
        fused_root=i32(0), draw_gumbel=i32(0), noise_seed=i32(0), reuse_prepared=i32(bool(reuse_prepared) and workspace is not None),
        hash_bits=i32(hash_bits), hash_io=i32(env.kind == ENV_SUBLEQ if hash_io is None else hash_io), max_u=f32(1.0), novelty_scale=f32(1.0))
    return PolicyOutput(action, weights, SearchTreeView(EpistemicSearchSummary(value, std, counts, probs, q, qvar), ws))


def evaluate(params, model_state, env: EnvSpec, states, *, num_simulations, discount, max_episode_length, exploitation_beta=0.0,
             rescale_values=True, mlp_mode=1, hash_io=None, hash_bits=24):
    """evaluate.py:13-57 from `states` = env.init(...) (evaluate.py:52-54; Subleq tasks drawn by the caller): greedy episodes
    (gumbel_scale = 0) until every env has terminated or max_episode_length moves have passed.  The loop runs on the device as one CUDA
    graph whose while condition the device decides.  Returns (mean sum of rewards, sums of rewards [B], final states)."""
    B = states.terminated.shape[0]
    leaves = state_leaves(env, states)
    from . import _abi  # ctypes mirrors of the POD structs (no torch)

    cfg = _abi.default_search_config(batch=B, num_simulations=num_simulations, gumbel_scale=0.0, mlp_mode=mlp_mode)
    e = _abi.EazEnv(env.kind, env.size, None, env.word_size, env.binary_encoding, env.reward_fn)
    _eaz.eaz_evaluate_workspace_bytes.restype = ctypes.c_size_t
    ws_bytes = int(_eaz.eaz_evaluate_workspace_bytes(ctypes.byref(cfg), ctypes.byref(e)))
    if ws_bytes == 0:
        raise ValueError(_eaz_error())
    ws_bytes += 256
    out_types = [jax.ShapeDtypeStruct(x.shape, x.dtype) for x in leaves] + [jax.ShapeDtypeStruct((B,), jnp.float32),
                                                                           jax.ShapeDtypeStruct((ws_bytes,), jnp.uint8)]
    beta = jnp.full((B,), exploitation_beta, jnp.float32)  # evaluate.py:34
    n = len(leaves)
    aliases = {3: n + 1} | {4 + k: k for k in range(n)}  # workspace_in -> workspace, leaves stepped in place
    out = jax.ffi.ffi_call("eaz_evaluate", out_types, input_output_aliases=aliases)(
        beta, env.amap(), model_state["fc_az_net/xxhash32"]["binary_set"], jnp.zeros((ws_bytes,), jnp.uint8), *leaves, *param_leaves(params),
        **env.attrs(), num_simulations=i32(num_simulations), max_depth=i32(0), max_num_considered_actions=i32(16), discount=f32(discount),
        value_scale=f32(0.1), maxvisit_init=f32(50.0), rescale_values=i32(rescale_values), flags=i32(DEFAULT_FLAGS), mlp_mode=i32(mlp_mode),
        hash_bits=i32(hash_bits), hash_io=i32(env.kind == ENV_SUBLEQ if hash_io is None else hash_io), max_u=f32(1.0), novelty_scale=f32(1.0),
        max_episode_length=i32(max_episode_length))
    returns = out[n]
    return returns.mean(), returns, with_leaves(env, states, out[:n])


class SelfplayOutput(NamedTuple):  # selfplay.py:17-23, every field stacked over the steps
    state: tuple                          # the states after each step as (eaz_env_compact records U8[T,B,S], rewards F32[T,B]): the
    root_value: jax.Array                 # replay ring's format (one row per time slot; make_prioritised_flat_buffer(...).add takes it)
    root_epistemic_std: jax.Array
    value_prediction: jax.Array
    ube_prediction: jax.Array
    q_values_epistemic_variance: jax.Array
    action: jax.Array
    trajectory: jax.Array                 # eaz_trajectory_pack records [T,B,4] (what the replay gather of main.py:383-385 sends)


def selfplay(params, model_state, env: EnvSpec, states, rng_key, *, selfplay_steps, num_simulations, discount, exploration_beta=0.0,
             directed_exploration=False, rescale_values=True, tasks=(1,), mlp_mode=1, uniform_prior=False, action_sampling=0, temperature=1.0,
             hash_io=None, hash_bits=24):
    """selfplay.py:78-149 from `states` (the last carry): selfplay_steps steps of the fused-root Gumbel search (the recurrent_fn's policy
    head: exploration = directed_exploration, beta = exploration_beta * linspace(0, 1, B) when directed, selfplay.py:92,105) and the
    auto-reset env step, as one custom call whose loop runs on the device.  The root noise [T,B,A] and the Subleq reset tasks [T,B]
    (jax.random.choice over `tasks`, subleq.py:624) are drawn from rng_key; action_sampling (EAZ_ACTION_*) draws its noise in the
    search.  Returns (final states, SelfplayOutput): lax.scan's (carry, ys) order."""
    B, A, T = states.terminated.shape[0], env.num_actions, int(selfplay_steps)
    leaves = state_leaves(env, states)
    from . import _abi  # ctypes mirrors of the POD structs (no torch)

    flags = DEFAULT_FLAGS
    cfg = _abi.default_search_config(batch=B, num_simulations=num_simulations, mlp_mode=mlp_mode, action_sampling=int(action_sampling))
    e = _abi.EazEnv(env.kind, env.size, None, env.word_size, env.binary_encoding, env.reward_fn)
    _eaz.eaz_selfplay_workspace_bytes.restype = ctypes.c_size_t
    ws_bytes = int(_eaz.eaz_selfplay_workspace_bytes(ctypes.byref(cfg), ctypes.byref(e)))
    S = int(_eaz.eaz_env_compact_bytes(ctypes.byref(e)))
    if ws_bytes == 0 or S <= 0:
        raise ValueError(_eaz_error())
    ws_bytes += 256
    noise_key, task_key = jax.random.split(rng_key)
    gumbel = jax.random.gumbel(noise_key, (T, B, A), jnp.float32)
    task_ids = (jax.random.choice(task_key, jnp.asarray(tasks, jnp.int32), (T, B)) if env.kind == ENV_SUBLEQ else jnp.zeros((1,), jnp.int32))
    beta = (exploration_beta if directed_exploration else 0.0) * jnp.linspace(0.0, 1.0, B, dtype=jnp.float32)
    TB = lambda *s, dt=jnp.float32: jax.ShapeDtypeStruct((T, B) + s, dt)
    out_types = ([jax.ShapeDtypeStruct(x.shape, x.dtype) for x in leaves] +
                 [TB(dt=jnp.int32), TB(), TB(), TB(), TB(), TB(A), TB(4, dt=jnp.int32), TB(S, dt=jnp.uint8), TB(),
                  jax.ShapeDtypeStruct((ws_bytes,), jnp.uint8)])
    n = len(leaves)
    aliases = {6: n + 9} | {7 + k: k for k in range(n)}  # workspace_in -> workspace, leaves stepped in place
    out = jax.ffi.ffi_call("eaz_selfplay", out_types, input_output_aliases=aliases)(
        beta, env.amap(), model_state["fc_az_net/xxhash32"]["binary_set"], gumbel, jnp.zeros((1,), jnp.float32), task_ids,
        jnp.zeros((ws_bytes,), jnp.uint8), *leaves, *param_leaves(params), **env.attrs(), num_simulations=i32(num_simulations), max_depth=i32(0),
        max_num_considered_actions=i32(16), gumbel_scale=f32(1.0), discount=f32(discount), two_players_game=i32(0),
        exploration=i32(directed_exploration), value_scale=f32(0.1), maxvisit_init=f32(50.0), rescale_values=i32(rescale_values),
        flags=i32(flags), mlp_mode=i32(mlp_mode), hash_bits=i32(hash_bits), hash_io=i32(env.kind == ENV_SUBLEQ if hash_io is None else hash_io),
        max_u=f32(1.0), novelty_scale=f32(1.0), steps=i32(T), root_prior=i32(bool(uniform_prior)), action_sampling=i32(action_sampling),
        temperature=f32(temperature), noise_seed=i32(0), reuse_prepared=i32(0))
    action, rv, rstd, vp, up, qvar, traj, compact, rewards = out[n:n + 9]
    return with_leaves(env, states, out[:n]), SelfplayOutput((compact, rewards), rv, rstd, vp, up, qvar, action, traj)


def env_step(env: EnvSpec, states, action, *, auto_reset=False, task_ids=None):
    """jax.vmap(env.step)(states, action) (selfplay.py:135 with auto_reset=True applies selfplay.py:26-75; Subleq resets take
    pre-drawn `task_ids` [B] instead of jax.random.choice, subleq.py:624)."""
    leaves = state_leaves(env, states)
    tasks = jnp.zeros((1,), jnp.int32) if task_ids is None else task_ids
    out_types = [jax.ShapeDtypeStruct(x.shape, x.dtype) for x in leaves]
    aliases = {3 + k: k for k in range(len(leaves))}  # step in place on the donated leaves
    out = jax.ffi.ffi_call("eaz_env_step", out_types, input_output_aliases=aliases)(
        action.astype(jnp.int32), tasks, env.amap(), *leaves, **env.attrs(), auto_reset=i32(auto_reset))
    return with_leaves(env, states, out)


def env_init(env: EnvSpec, template_state, batch, task_ids=None):
    leaves = state_leaves(env, template_state)
    tasks = jnp.zeros((1,), jnp.int32) if task_ids is None else task_ids
    out_types = [jax.ShapeDtypeStruct(x.shape, x.dtype) for x in leaves]
    out = jax.ffi.ffi_call("eaz_env_init", out_types)(tasks, env.amap(), **env.attrs(), batch=i32(batch))
    return with_leaves(env, template_state, out)


def forward_states(params, model_state, env: EnvSpec, states, *, hash_io=None, hash_bits=24):
    """forward.apply(params, state, states.observation, is_training=False) (selfplay.py:89) without materialising observations:
    returns (exploitation_logits, exploration_logits, value, ube, novelty) -- fully_connected.py:101."""
    B, A = states.terminated.shape[0], env.num_actions
    S = 4 if env.kind == ENV_DEEPSEA else 40 + ((env.word_size + 7) & ~7)
    fB, fBA = jax.ShapeDtypeStruct((B,), jnp.float32), jax.ShapeDtypeStruct((B, A), jnp.float32)
    out = jax.ffi.ffi_call("eaz_mlp_forward_states", [fBA, fBA, fB, fB, fB, jax.ShapeDtypeStruct((B * S + 16,), jnp.uint8)])(
        env.amap(), model_state["fc_az_net/xxhash32"]["binary_set"], *state_leaves(env, states), *param_leaves(params), **env.attrs(),
        hash_bits=i32(hash_bits), hash_io=i32(env.kind == ENV_SUBLEQ if hash_io is None else hash_io), max_u=f32(1.0), novelty_scale=f32(1.0))
    return out[:5]


def reanalyze_targets(config, action, summary: EpistemicSearchSummary, next_state_value, next_rewards, next_terminated, terminated,
                      invalid_actions=None):
    """reanalyze.py:86-129: (value_target, ube_target, exploration_policy_target)."""
    B, A = summary.qvalues.shape
    fB = jax.ShapeDtypeStruct((B,), jnp.float32)
    inv = jnp.zeros((1,), jnp.bool_) if invalid_actions is None else invalid_actions
    return jax.ffi.ffi_call("eaz_reanalyze_targets", [fB, fB, jax.ShapeDtypeStruct((B, A), jnp.float32)])(
        action, summary.qvalues, summary.qvalues_epistemic_variance, summary.visit_counts, summary.value, summary.value_epistemic_std,
        next_state_value, next_rewards.reshape(B), next_terminated, terminated, inv, discount=f32(config.discount),
        exploration_beta=f32(config.exploration_beta), exploration_ube_target=i32(config.exploration_ube_target),
        temperature=f32(config.exploration_policy_target_temperature))


def hash_update(binary_set, x, bits=24):
    """BaseHash.update (hashes.py:45-50): sets the bits of the rows of x (float32 [B, D]) in `binary_set` (donated)."""
    return jax.ffi.ffi_call("eaz_hash_update", jax.ShapeDtypeStruct(binary_set.shape, binary_set.dtype), input_output_aliases={1: 0})(
        x.astype(jnp.float32), binary_set, bits=i32(bits))


# ------------------------------------------------------------------------------------------------ prioritised replay
_LEAF_NAMES = {ENV_DEEPSEA: ["_step_count", "rewards", "terminated", "truncated", "_horizontal_position"],
               ENV_SUBLEQ: ["_step_count", "rewards", "terminated", "truncated", "_memory_state", "_task", "_solved", "_example_input_after",
                            "_example_output_after"]}


def _leaf_types(env: EnvSpec, n):
    """ShapeDtypeStructs of the state leaves of n envs, in eaz_state order"""
    s = lambda *shape, dt=jnp.int32: jax.ShapeDtypeStruct((n,) + shape, dt)
    common = [s(), s(1, dt=jnp.float32), s(dt=jnp.bool_), s(dt=jnp.bool_)]
    if env.kind == ENV_DEEPSEA:
        return common + [s()]
    return common + [s(env.word_size), s(), s(dt=jnp.bool_), s(8), s(8)]


class ReplayState(NamedTuple):
    """The buffer state a jitted program threads through its steps: compact records [T,B,S], rewards [T,B] and the sum tree, whose
    header holds the write cursor and length (csrc/replay.cu)."""
    states: jax.Array
    rewards: jax.Array
    tree: jax.Array


class PrioritisedSample(NamedTuple):
    """flashbax's PrioritisedTrajectoryBufferSample: experience = (first, second), each a dict of pgx.State leaves for K envs
    (`template_state.replace(**first)` makes it a pgx.State), indices int32 [K] (handles for set_priorities), probabilities [K]."""
    experience: tuple
    indices: jax.Array
    probabilities: jax.Array


class PrioritisedFlatBuffer(NamedTuple):
    init: object
    add: object
    sample: object
    set_priorities: object
    can_sample: object
    status: object


def make_prioritised_flat_buffer(env: EnvSpec, max_length_time_axis, add_batch_size, sample_batch_size, priority_exponent=0.6):
    """flashbax.make_prioritised_flat_buffer (main.py:217-225) on the compact ring, as pure functions of jax arrays:

        init(template_state, seed) -> ReplayState          (seed: a Python int, it becomes an attribute)
        add(rs, states) -> ReplayState                     one time step of the add_batch_size envs, at the device cursor
        add(rs, (compact, rewards)) -> ReplayState         T' time steps at once, in time order: selfplay()'s SelfplayOutput.state
                                                           (U8[T',B,S], F32[T',B]), so `rs = add(rs, out.state)` is main.py:383-385
        sample(rs, key) -> PrioritisedSample               sample_batch_size pairs drawn from key; rs is only read
        set_priorities(rs, indices, priorities) -> ReplayState
        can_sample(rs) -> bool[]                           at least two time steps stored
        status(rs) -> int32[]                              the sticky EAZ_PRIORITY_* bits (0: nothing went wrong)

    add and set_priorities alias their inputs to their results; donate `rs` at the jit boundary (donate_argnums) so that XLA
    updates the three arrays in place instead of copying them."""
    T, B, K = int(max_length_time_axis), int(add_batch_size), int(sample_batch_size)
    from . import _abi  # ctypes mirrors of the POD structs (no torch)

    e = _abi.EazEnv(env.kind, env.size, None, env.word_size, env.binary_encoding, env.reward_fn)
    _eaz.eaz_priority_tree_bytes.restype = ctypes.c_size_t
    S = int(_eaz.eaz_env_compact_bytes(ctypes.byref(e)))
    tree_bytes = int(_eaz.eaz_priority_tree_bytes(T, B))
    if S <= 0 or tree_bytes == 0:
        raise ValueError(_eaz_error())
    ring_types = [jax.ShapeDtypeStruct((T, B, S), jnp.uint8), jax.ShapeDtypeStruct((T, B), jnp.float32),
                  jax.ShapeDtypeStruct((tree_bytes,), jnp.uint8)]
    names = _LEAF_NAMES[env.kind]

    def init(template_state=None, seed=0):
        del template_state  # the ring stores compact records; its shapes come from env, T and B
        out = jax.ffi.ffi_call("eaz_replay_init", ring_types)(T=i32(T), B=i32(B), priority_exponent=f32(priority_exponent),
                                                              seed=i32(np.uint32(seed).view(np.int32)))
        return ReplayState(*out)

    def add(rs: ReplayState, states):
        if isinstance(states, tuple):  # (compact records [T',B,S], rewards [T',B]): a scan's time steps
            compact, rewards = states
            out = jax.ffi.ffi_call("eaz_replay_add_sequence", ring_types, input_output_aliases={1: 0, 2: 1, 3: 2})(
                env.amap(), rs.states, rs.rewards, rs.tree, compact.astype(jnp.uint8), rewards.astype(jnp.float32), **env.attrs())
            return ReplayState(*out)
        out = jax.ffi.ffi_call("eaz_replay_add", ring_types, input_output_aliases={1: 0, 2: 1, 3: 2})(
            env.amap(), rs.states, rs.rewards, rs.tree, *state_leaves(env, states), **env.attrs())
        return ReplayState(*out)

    def sample(rs: ReplayState, key):
        words = jax.random.bits(key, (2,), jnp.uint32)  # (seed, draw counter) of the contract's stratified draws
        out_types = ([jax.ShapeDtypeStruct((K,), jnp.int32), jax.ShapeDtypeStruct((K,), jnp.float32)] + _leaf_types(env, K) +
                     _leaf_types(env, K) + [jax.ShapeDtypeStruct((2 * K * (S + 4) + 16,), jnp.uint8)])
        out = jax.ffi.ffi_call("eaz_replay_sample", out_types)(env.amap(), rs.states, rs.rewards, rs.tree, words, **env.attrs(), K=i32(K))
        n = len(names)
        first, second = dict(zip(names, out[2:2 + n])), dict(zip(names, out[2 + n:2 + 2 * n]))
        return PrioritisedSample((first, second), out[0], out[1])

    def set_priorities(rs: ReplayState, indices, priorities):
        tree = jax.ffi.ffi_call("eaz_replay_set_priorities", ring_types[2], input_output_aliases={2: 0})(
            indices.astype(jnp.int32).reshape(-1), priorities.astype(jnp.float32).reshape(-1), rs.tree, T=i32(T), B=i32(B))
        return rs._replace(tree=tree)

    def can_sample(rs: ReplayState):
        length = jax.lax.bitcast_convert_type(rs.tree[20:24], jnp.int32)  # PrioHeader.length (bytes 20..23 of the header)
        return length >= 2

    def status(rs: ReplayState):
        return jax.ffi.ffi_call("eaz_replay_status", jax.ShapeDtypeStruct((1,), jnp.int32))(rs.tree)[0]

    return PrioritisedFlatBuffer(init, add, sample, set_priorities, can_sample, status)


def _eaz_error():
    _eaz.eaz_last_error.restype = ctypes.c_char_p
    return _eaz.eaz_last_error().decode("utf-8", "replace")
