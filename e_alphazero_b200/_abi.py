"""ctypes mirror of include/eaz_b200.h (field order and types must match the header).

These are plain POD descriptions; they carry no behaviour.  The product fills
them with CUDA device pointers (``_lib.py``); the CPU oracle's binding reuses the
same layouts with host pointers (``oracle/oracle.py``).
"""
from __future__ import annotations

import ctypes as C

ABI_VERSION = 8

EAZ_OK = 0
EAZ_ERR_INVALID_ARG = -1
EAZ_ERR_WORKSPACE = -2
EAZ_ERR_CUDA = -3
EAZ_ERR_UNSUPPORTED = -4

ENV_DEEPSEA = 0
ENV_SUBLEQ = 1
SUBLEQ_REWARD_SOLVED = 0
SUBLEQ_REWARD_LOWEST_BYTES = 1

HEAD_VALUE, HEAD_UBE, HEAD_EXPLOIT, HEAD_EXPLORE = 0, 1, 2, 3

FLAG_BETA_INTERIOR = 1 << 0
FLAG_BETA_RAW = 1 << 1
FLAG_BETA_FINAL = 1 << 2
FLAG_BACKUP_STD = 1 << 3
FLAG_REUSE_PREPARED = 1 << 4
FLAG_STREAMS_SHIFT = 8
FLAG_PUCT = 1 << 5


def flag_streams(k: int) -> int:
    """EAZ_FLAG_STREAMS(k): search k sub-batches concurrently on auxiliary streams (results unchanged)."""
    return (int(k) & 0xF) << FLAG_STREAMS_SHIFT


SEARCH_DEFAULT_FLAGS = FLAG_BETA_INTERIOR | FLAG_BETA_RAW | FLAG_BETA_FINAL

PRIORITY_BAD_PRIORITY = 1 << 0
PRIORITY_BAD_INDEX = 1 << 1
PRIORITY_EMPTY = 1 << 2
PRIORITY_BAD_ADD = 1 << 3

MLP_EXACT = 0
MLP_TENSOR = 1

# eaz_search_config.root_prior / action_sampling (selfplay.py:92-98, 125-134)
ROOT_PRIOR_GIVEN, ROOT_PRIOR_UNIFORM = 0, 1
ACTION_SEARCH, ACTION_VISITS, ACTION_IMPROVED = 0, 1, 2

_p = C.c_void_p


class EazEnv(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("size", C.c_int32),
        ("action_map", _p),
        ("word_size", C.c_int32),
        ("binary_encoding", C.c_int32),
        ("reward_fn", C.c_int32),
    ]


class EazState(C.Structure):
    _fields_ = [
        ("step_count", _p),
        ("rewards", _p),
        ("terminated", _p),
        ("truncated", _p),
        ("observation", _p),
        ("col", _p),
        ("memory", _p),
        ("task", _p),
        ("solved", _p),
        ("input_after", _p),
        ("output_after", _p),
    ]


class EazFcParams(C.Structure):
    _fields_ = [
        ("in_dim", C.c_int32),
        ("hidden", C.c_int32),
        ("num_actions", C.c_int32),
        ("w", (_p * 3) * 4),
        ("b", (_p * 3) * 4),
        ("binary_set", _p),
        ("hash_bits", C.c_int32),
        ("hash_io", C.c_int32),
        ("word_size", C.c_int32),
        ("max_u", C.c_float),
        ("novelty_scale", C.c_float),
    ]


class EazSearchConfig(C.Structure):
    _fields_ = [
        ("batch", C.c_int32),
        ("num_simulations", C.c_int32),
        ("max_depth", C.c_int32),
        ("max_num_considered_actions", C.c_int32),
        ("gumbel_scale", C.c_float),
        ("discount", C.c_float),
        ("two_players_game", C.c_int32),
        ("exploration", C.c_int32),
        ("value_scale", C.c_float),
        ("maxvisit_init", C.c_float),
        ("rescale_values", C.c_int32),
        ("use_mixed_value", C.c_int32),
        ("epsilon", C.c_float),
        ("flags", C.c_int32),
        ("mlp_mode", C.c_int32),
        ("pb_c_init", C.c_float),
        ("pb_c_base", C.c_float),
        ("temperature", C.c_float),
        ("noise_seed", C.c_uint32),
        ("root_prior", C.c_int32),
        ("action_sampling", C.c_int32),
    ]


CONVNET_RESNET, CONVNET_MINATAR = 0, 1
CONVNET_MAX_BLOCKS = 8


class EazConv(C.Structure):  # hk.Conv2D / hk.Linear: w, b
    _fields_ = [("w", _p), ("b", _p)]


class EazBn(C.Structure):  # hk.BatchNorm in inference: scale, offset (params), mean / var averages (state)
    _fields_ = [("scale", _p), ("offset", _p), ("mean", _p), ("var", _p)]


class EazConvnetParams(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("height", C.c_int32), ("width", C.c_int32), ("in_channels", C.c_int32), ("num_actions", C.c_int32),
        ("num_channels", C.c_int32), ("hidden", C.c_int32), ("num_blocks", C.c_int32), ("resnet_v2", C.c_int32),
        ("stem", EazConv), ("stem_bn", EazBn),
        ("block_bn", (EazBn * 2) * CONVNET_MAX_BLOCKS), ("block_conv", (EazConv * 2) * CONVNET_MAX_BLOCKS),
        ("final_bn", EazBn),
        ("head_conv", EazConv * 4), ("head_bn", EazBn * 4), ("head_fc", EazConv * 4), ("head_out", EazConv * 4),
        ("tower_conv", EazConv * 2), ("tower_fc", (EazConv * 2) * 2), ("mhead_fc", (EazConv * 2) * 4),
        ("binary_set", _p), ("hash_bits", C.c_int32), ("max_u", C.c_float), ("novelty_scale", C.c_float), ("local_unc_scale", C.c_float),
        ("mlp_mode", C.c_int32),
    ]


def fill_convnet_params(desc: dict, ptr) -> EazConvnetParams:
    """desc: the network as nested python data (see `convnet_description`); ptr(array) -> address.  Shared by the CUDA binding
    (device tensors) and the oracle binding (numpy arrays): same struct, different address spaces."""
    s = EazConvnetParams()
    for k in ("kind", "height", "width", "in_channels", "num_actions", "num_channels", "hidden", "num_blocks", "resnet_v2", "hash_bits"):
        setattr(s, k, int(desc[k]))
    for k in ("max_u", "novelty_scale", "local_unc_scale"):
        setattr(s, k, float(desc[k]))
    s.binary_set = ptr(desc["binary_set"])
    s.mlp_mode = int(desc.get("mlp_mode", MLP_EXACT))

    def conv(dst, d):
        dst.w, dst.b = ptr(d["w"]), ptr(d["b"])

    def bn(dst, d):
        dst.scale, dst.offset, dst.mean, dst.var = ptr(d["scale"]), ptr(d["offset"]), ptr(d["mean"]), ptr(d["var"])

    if desc["kind"] == CONVNET_RESNET:
        conv(s.stem, desc["stem"])
        if not desc["resnet_v2"]:
            bn(s.stem_bn, desc["stem_bn"])
        else:
            bn(s.final_bn, desc["final_bn"])
        for i, blk in enumerate(desc["blocks"]):
            for j in range(2):
                bn(s.block_bn[i][j], blk["bn"][j])
                conv(s.block_conv[i][j], blk["conv"][j])
        for h, hd in enumerate(desc["heads"]):
            conv(s.head_conv[h], hd["conv"])
            bn(s.head_bn[h], hd["bn"])
            conv(s.head_fc[h], hd["fc"])
            if h >= 2:
                conv(s.head_out[h], hd["out"])
    else:
        for t in range(2):
            conv(s.tower_conv[t], desc["towers"][t]["conv"])
            for j in range(2):
                conv(s.tower_fc[t][j], desc["towers"][t]["fc"][j])
        for h in range(4):
            for j in range(2):
                conv(s.mhead_fc[h][j], desc["mheads"][h][j])
    return s


def convnet_description(params: dict, state: dict, kind: int, height: int, width: int, in_channels: int, num_actions: int, *, num_channels=None,
                        hidden=64, num_blocks=5, resnet_v2=True, hash_bits=24, max_u=1.0, novelty_scale=1.0, discount=0.9997, prefix=None,
                        hash_name="xxhash32") -> dict:
    """haiku pytrees of EpistemicResidualAZNet (prefix az_resnet, resnet.py:41-135) / EpistemicMinatarAZNet (prefix minatar_az_net,
    minatar.py:11-114) -> the nested description `fill_convnet_params` consumes.  Module names follow haiku's call-order numbering."""
    def cv(name):
        return dict(w=params[name]["w"], b=params[name]["b"])

    def bn(name):
        return dict(scale=params[name]["scale"].reshape(-1), offset=params[name]["offset"].reshape(-1),
                    mean=state[name + "/~/mean_ema"]["average"].reshape(-1), var=state[name + "/~/var_ema"]["average"].reshape(-1))

    def nth(base, i):
        return base if i == 0 else f"{base}_{i}"

    if kind == CONVNET_RESNET:
        p = prefix or "az_resnet"
        C_ = num_channels or 64
        d = dict(kind=kind, height=height, width=width, in_channels=in_channels, num_actions=num_actions, num_channels=C_, hidden=C_,
                 num_blocks=num_blocks, resnet_v2=int(resnet_v2), stem=cv(f"{p}/conv2_d"))
        nbn = 0
        if not resnet_v2:
            d["stem_bn"] = bn(f"{p}/batch_norm")
            nbn = 1
        d["blocks"] = [dict(bn=[bn(f"{p}/block_{i}/batch_norm"), bn(f"{p}/block_{i}/batch_norm_1")],
                            conv=[cv(f"{p}/block_{i}/conv2_d"), cv(f"{p}/block_{i}/conv2_d_1")]) for i in range(num_blocks)]
        if resnet_v2:
            d["final_bn"] = bn(f"{p}/{nth('batch_norm', nbn)}")
            nbn += 1
        heads, nlin = [], 0
        for h in range(4):  # call order: main policy, exploration policy, value, ube (resnet.py:84-124)
            hd = dict(conv=cv(f"{p}/{nth('conv2_d', 1 + h)}"), bn=bn(f"{p}/{nth('batch_norm', nbn + h)}"), fc=cv(f"{p}/{nth('linear', nlin)}"))
            nlin += 1
            if h >= 2:
                hd["out"] = cv(f"{p}/{nth('linear', nlin)}")
                nlin += 1
            heads.append(hd)
        d["heads"] = heads
        d["local_unc_scale"] = 1.0
    else:
        p = prefix or "minatar_az_net"
        C_ = num_channels or 16
        d = dict(kind=kind, height=height, width=width, in_channels=in_channels, num_actions=num_actions, num_channels=C_, hidden=hidden,
                 num_blocks=0, resnet_v2=0)
        # call order (minatar.py:57-95): conv, lin0, lin1 | policy lin2, lin3 | value lin4, lin5 | conv_1, lin6, lin7 | expl lin8, lin9 | ube lin10, lin11
        L = lambda i: cv(f"{p}/{nth('linear', i)}")
        d["towers"] = [dict(conv=cv(f"{p}/conv2_d"), fc=[L(0), L(1)]), dict(conv=cv(f"{p}/conv2_d_1"), fc=[L(6), L(7)])]
        d["mheads"] = [[L(2), L(3)], [L(4), L(5)], [L(8), L(9)], [L(10), L(11)]]  # main policy, value, exploration policy, ube
        d["local_unc_scale"] = 1.0 / (1.0 - min(discount, 0.9997) ** 2)
    d.update(binary_set=state[f"{p}/{hash_name}"]["binary_set"], hash_bits=hash_bits, max_u=max_u, novelty_scale=novelty_scale)
    return d


class EazReanalyzeConfig(C.Structure):
    _fields_ = [
        ("discount", C.c_float),
        ("exploration_beta", C.c_float),
        ("exploration_ube_target", C.c_int32),
        ("exploration_policy_target_temperature", C.c_float),
    ]


class EazSearchInputs(C.Structure):
    _fields_ = [
        ("prior_logits", _p),
        ("value", _p),
        ("value_epistemic_variance", _p),
        ("beta", _p),
        ("embedding", C.POINTER(EazState)),
        ("invalid_actions", _p),
        ("gumbel", _p),
        ("env", C.POINTER(EazEnv)),
        ("net", C.POINTER(EazFcParams)),
        ("sample_gumbel", _p),
    ]


SEARCH_OUTPUT_FIELDS = [
    # name, dtype, shape-kind  (B | BA | BN | BNA | BNS)
    ("action", "i32", "B"),
    ("action_weights", "f32", "BA"),
    ("value", "f32", "B"),
    ("value_epistemic_std", "f32", "B"),
    ("visit_counts", "f32", "BA"),
    ("visit_probs", "f32", "BA"),
    ("qvalues", "f32", "BA"),
    ("qvalues_epistemic_variance", "f32", "BA"),
    ("node_visits", "i32", "BN"),
    ("raw_values", "f32", "BN"),
    ("node_values", "f32", "BN"),
    ("raw_values_epistemic_variance", "f32", "BN"),
    ("node_values_epistemic_variance", "f32", "BN"),
    ("parents", "i32", "BN"),
    ("action_from_parent", "i32", "BN"),
    ("children_index", "i32", "BNA"),
    ("children_prior_logits", "f32", "BNA"),
    ("children_visits", "i32", "BNA"),
    ("children_rewards", "f32", "BNA"),
    ("children_discounts", "f32", "BNA"),
    ("children_values", "f32", "BNA"),
    ("children_rewards_epistemic_variance", "f32", "BNA"),
    ("children_values_epistemic_variance", "f32", "BNA"),
    ("embeddings", "u8", "BNS"),
    ("root_value", "f32", "B"),
    ("root_ube", "f32", "B"),
]
SUMMARY_FIELDS = [f for f in SEARCH_OUTPUT_FIELDS[:8]]
TREE_FIELDS = [f for f in SEARCH_OUTPUT_FIELDS[8:24]]
ROOT_FIELDS = [f for f in SEARCH_OUTPUT_FIELDS[24:]]  # fused-root mode


class EazSearchOutputs(C.Structure):
    _fields_ = [(name, _p) for name, _, _ in SEARCH_OUTPUT_FIELDS]


class EazEvaluateCounters(C.Structure):  # the evaluation loop's device words at the start of the eaz_evaluate workspace
    _fields_ = [("moves", C.c_int32), ("live", C.c_int32), ("ticket", C.c_uint32), ("cont", C.c_int32)]


class EazSelfplayOutputs(C.Structure):  # the stacked per-step outputs of eaz_selfplay: [T,B], [T,B,A], [T,B,4], [T,B,S]
    _fields_ = [(name, _p) for name in ("action", "root_value", "root_epistemic_std", "value_prediction", "ube_prediction",
                                        "q_values_epistemic_variance", "trajectory", "states", "rewards")]


def default_search_config(**kw) -> EazSearchConfig:
    """Defaults of emctx.epistemic_gumbel_muzero_policy /
    epistemic_qtransform_completed_by_mix_value (SURVEY.md Appendix A.1, A.6)."""
    cfg = EazSearchConfig(
        batch=0,
        num_simulations=32,
        max_depth=0,
        max_num_considered_actions=16,
        gumbel_scale=1.0,
        discount=0.997,
        two_players_game=0,
        exploration=0,
        value_scale=0.1,
        maxvisit_init=50.0,
        rescale_values=1,
        use_mixed_value=1,
        epsilon=1e-8,
        flags=SEARCH_DEFAULT_FLAGS,
        mlp_mode=MLP_EXACT,
        pb_c_init=1.25,
        pb_c_base=19652.0,
        temperature=1.0,
        noise_seed=0,
        root_prior=ROOT_PRIOR_GIVEN,
        action_sampling=ACTION_SEARCH,
    )
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise TypeError(f"unknown search config field {k!r}")
        setattr(cfg, k, v)
    return cfg
