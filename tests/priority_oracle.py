"""numpy binding of tests/priority_oracle.c, the CPU oracle of the prioritised replay sum tree (TEST INFRASTRUCTURE ONLY).

The library is compiled on first use into the temporary directory (keyed by the sources' contents), so the tests never write
into the repository tree.  A tree is a uint8 array with the byte layout of the device buffer (csrc/replay.cu)."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_SRCS = [os.path.join(_HERE, "priority_oracle.c"), os.path.join(_ROOT, "oracle", "eaz_oracle.c"),
         os.path.join(_ROOT, "include", "eaz_b200.h"), os.path.join(_ROOT, "include", "eaz_math.h")]
_lib = None

HEADER = np.dtype([("alpha", "<f4"), ("seed", "<u4"), ("draw_ctr", "<u4"), ("status", "<u4"), ("cursor", "<i4"), ("length", "<i4"),
                   ("max_priority", "<f4"), ("reserved", "<u4")])


def lib():
    global _lib
    if _lib is None:
        key = hashlib.sha256(b"".join(open(p, "rb").read() for p in _SRCS)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"eaz_priority_oracle_{os.getuid()}_{key}.so")
        if not os.path.exists(so):
            cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"  # the flags of oracle/Makefile
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.run([cc, "-O2", "-std=c11", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                            "-Wno-unused-function", "-o", tmp, _SRCS[0], "-lm"], check=True)
            os.replace(tmp, so)
        _lib = C.CDLL(so)
        _lib.orc_priority_tree_bytes.restype = C.c_size_t
        _lib.orc_priority_descend.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_float]
    return _lib


def _p(a):
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


def _chk(rc, what):
    if rc < 0:
        raise ValueError(f"priority oracle {what} failed with {rc}")


def tree_bytes(T, B) -> int:
    return int(lib().orc_priority_tree_bytes(int(T), int(B)))


def init(T, B, alpha=0.6, seed=0) -> np.ndarray:
    buf = np.zeros(tree_bytes(T, B), np.uint8)
    _chk(lib().orc_priority_init(_p(buf), int(T), int(B), C.c_float(alpha), C.c_uint32(seed)), "init")
    return buf


def add_step(buf, T, B, slot) -> None:
    _chk(lib().orc_priority_add_step(_p(buf), int(T), int(B), int(slot)), "add_step")


def set_priorities(buf, T, B, indices, priorities) -> None:
    i = np.ascontiguousarray(indices, np.int32)
    p = np.ascontiguousarray(priorities, np.float32)
    assert i.shape == p.shape
    _chk(lib().orc_priority_set(_p(buf), int(T), int(B), _p(i), _p(p), i.size), "set")


def sample(buf, T, B, K, states=None, rewards=None):
    """-> dict(indices [K], probabilities [K]) plus first / second [K,S] and first_rewards / second_rewards [K] when `states`
    ([T,B,S] uint8) and `rewards` ([T,B] float32) are given."""
    out = dict(indices=np.zeros(K, np.int32), probabilities=np.zeros(K, np.float32))
    S = 0
    if states is not None:
        states = np.ascontiguousarray(states, np.uint8)
        S = states.shape[-1]
        out.update(first=np.zeros((K, S), np.uint8), second=np.zeros((K, S), np.uint8))
        if rewards is not None:
            rewards = np.ascontiguousarray(rewards, np.float32)
            out.update(first_rewards=np.zeros(K, np.float32), second_rewards=np.zeros(K, np.float32))
    _chk(lib().orc_priority_sample(_p(buf), int(T), int(B), int(K), _p(states), _p(rewards), int(S), _p(out["indices"]), _p(out["probabilities"]),
                                   _p(out.get("first")), _p(out.get("first_rewards")), _p(out.get("second")), _p(out.get("second_rewards"))),
         "sample")
    return out


def descend(buf, T, B, u) -> int:
    """The leaf one sample with stratified draw `u` lands on (-1: empty tree)."""
    return int(lib().orc_priority_descend(_p(buf), int(T), int(B), float(u)))


def header(buf):
    return buf[:32].view(HEADER)[0]


def levels(buf, T, B) -> list[np.ndarray]:
    """The fp32 levels (leaves first), without their zero padding."""
    N = T * B
    off = (256 + 4 * N + 127) // 128 * 128
    out, n = [], N
    while True:
        out.append(buf[off:off + 4 * n].view(np.float32))
        off += ((n + 31) // 32 * 32 * 4 + 127) // 128 * 128
        if n == 1:
            return out
        n = (n + 31) // 32
