"""numpy binding of tests/selfplay_oracle.c, the CPU oracle of the self-play step options (TEST INFRASTRUCTURE ONLY): the uniform root
prior and the played action drawn from the visit counts or the improved policy (eaz_search_config.root_prior / action_sampling).

The library is compiled on first use into the temporary directory (keyed by the sources' contents), so the tests never write into the
repository tree."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from e_alphazero_b200 import _abi
from oracle import oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_SRCS = [os.path.join(_HERE, "selfplay_oracle.c"), os.path.join(_ROOT, "oracle", "eaz_oracle.c"),
         os.path.join(_ROOT, "include", "eaz_b200.h"), os.path.join(_ROOT, "include", "eaz_math.h")]
_lib = None


def lib():
    global _lib
    if _lib is None:
        key = hashlib.sha256(b"".join(open(p, "rb").read() for p in _SRCS)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"eaz_selfplay_oracle_{os.getuid()}_{key}.so")
        if not os.path.exists(so):
            cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"  # the flags of oracle/Makefile
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.run([cc, "-O2", "-std=c11", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                            "-Wno-unused-function", "-o", tmp, _SRCS[0], "-lm"], check=True)
            os.replace(tmp, so)
        _lib = C.CDLL(so)
        _lib.orc_stream_gumbel.restype = C.c_float
        _lib.orc_stream_gumbel.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int32]
        _lib.orc_stream_gumbel_rows.argtypes = [C.c_uint32, C.c_uint32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
        _lib.orc_sample_actions.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_void_p]
    return _lib


def _p(a):
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


def stream_gumbel(seed, ctr, B, A, sample=True, tree0=0) -> np.ndarray:
    """The in-kernel noise [B,A] of trees tree0 .. tree0 + B - 1 at draw counter `ctr`: of the action draw (sample=True) or the root."""
    g = np.zeros((B, A), np.float32)
    lib().orc_stream_gumbel_rows(int(seed) & 0xFFFFFFFF, int(ctr) & 0xFFFFFFFF, int(tree0), int(B), int(A), int(bool(sample)), _p(g))
    return g


def sample_actions(weights, gumbel, temperature=1.0, invalid_actions=None) -> np.ndarray:
    """The draw of EAZ_ACTION_VISITS / IMPROVED from weights [B,A] (visit_probs / action_weights) with the noise gumbel [B,A]."""
    w = np.ascontiguousarray(weights, np.float32)
    g = np.ascontiguousarray(gumbel, np.float32)
    inv = None if invalid_actions is None else np.ascontiguousarray(invalid_actions, np.uint8)
    B, A = w.shape
    assert g.shape == (B, A) and (inv is None or inv.shape == (B, A))
    out = np.zeros(B, np.int32)
    rc = lib().orc_sample_actions(_p(w), _p(inv), _p(g), B, A, C.c_float(temperature), _p(out))
    if rc < 0:
        raise ValueError(f"selfplay oracle sample_actions failed with {rc}")
    return out


def search(cfg: _abi.EazSearchConfig, env, net, root: dict, want_tree=True, fused_root=False) -> dict:
    """oracle.search with the options of `cfg`: root_prior UNIFORM searches from zero root logits; action_sampling replaces the action
    by the draw from this search's visit_probs / action_weights with root["sample_gumbel"].  fused_root: the root value / UBE (and,
    with the given prior, the logits of the recurrent_fn's policy head) come from the oracle network, as the library's fused root."""
    root = dict(root)
    if fused_root:
        ev = O.mlp_forward_states(net, env, root["embedding"])
        root.update(prior_logits=ev["explore_logits" if cfg.exploration else "exploit_logits"], value=ev["value"], value_epistemic_variance=ev["ube"])
    if cfg.root_prior == _abi.ROOT_PRIOR_UNIFORM:
        root["prior_logits"] = np.zeros_like(root["prior_logits"], dtype=np.float32)
    base = _abi.EazSearchConfig.from_buffer_copy(cfg)
    base.root_prior, base.action_sampling = _abi.ROOT_PRIOR_GIVEN, _abi.ACTION_SEARCH
    out = O.search(base, env, net, root, want_tree=want_tree)
    cfg.batch = base.batch
    if fused_root:
        out["root_value"], out["root_ube"] = root["value"].copy(), root["value_epistemic_variance"].copy()
    if cfg.action_sampling != _abi.ACTION_SEARCH:
        w = out["visit_probs"] if cfg.action_sampling == _abi.ACTION_VISITS else out["action_weights"]
        out["search_action"] = out["action"]
        out["action"] = sample_actions(w, root["sample_gumbel"], cfg.temperature, root.get("invalid_actions"))
    return out
