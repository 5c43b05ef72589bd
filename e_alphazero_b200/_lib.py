"""Loader for libeaz_b200.so (the C ABI of include/eaz_b200.h).

There is no fallback: if the shared library is missing, or an op is called
without a CUDA device, this raises.  PyTorch is used only to own device memory
and streams; every computation happens inside the library's CUDA kernels.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

from . import _abi

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("EAZ_LIB_PATH") or os.path.join(_HERE, "libeaz_b200.so")  # (EAZ_LIB_PATH: A/B measurements of two builds)
_lib = None

# every symbol include/eaz_b200.h declares
EXPORTS = [
    "eaz_abi_version", "eaz_last_error",
    "eaz_env_init", "eaz_env_step", "eaz_env_observe", "eaz_env_compact", "eaz_env_uncompact", "eaz_trajectory_pack",
    "eaz_env_num_actions", "eaz_env_obs_dim", "eaz_env_obs_cols", "eaz_env_hash_dim", "eaz_env_compact_bytes",
    "eaz_subleq_test_cases",
    "eaz_xxhash_indices", "eaz_hash_lookup", "eaz_hash_update",
    "eaz_mlp_forward", "eaz_mlp_forward_states",
    "eaz_search_workspace_bytes", "eaz_search_gumbel", "eaz_search_gumbel_profiled", "eaz_search_num_launches", "eaz_search_numeric_status",
    "eaz_reanalyze_targets",
    "eaz_convnet_workspace_bytes", "eaz_convnet_forward", "eaz_convnet_numeric_status",
    "eaz_priority_tree_bytes", "eaz_priority_init", "eaz_priority_add_step", "eaz_priority_set", "eaz_priority_sample", "eaz_priority_status",
    "eaz_replay_add", "eaz_priority_sample_keyed", "eaz_priority_status_async",
]


class EazError(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    """Compile the CUDA sources for sm_100a (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-C", os.path.join(_HERE, "csrc"), "-j4"], capture_output=not verbose, text=True)
    if r.returncode != 0:
        raise EazError("building libeaz_b200.so failed:\n" + (r.stdout or "") + (r.stderr or ""))
    return SO_PATH


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise EazError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(the CUDA library is the only implementation; there is no CPU fallback)")
    lib = C.CDLL(SO_PATH)
    for name in EXPORTS:
        if not hasattr(lib, name):
            raise EazError(f"libeaz_b200.so does not export {name}")
    lib.eaz_last_error.restype = C.c_char_p
    lib.eaz_search_workspace_bytes.restype = C.c_size_t
    lib.eaz_convnet_workspace_bytes.restype = C.c_size_t
    lib.eaz_priority_tree_bytes.restype = C.c_size_t
    if lib.eaz_abi_version() != _abi.ABI_VERSION:
        raise EazError(f"ABI version mismatch: library {lib.eaz_abi_version()} vs bindings {_abi.ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().eaz_last_error().decode("utf-8", "replace")
        raise EazError(f"{what} failed ({rc}): {msg}")


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise EazError("e_alphazero_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch
