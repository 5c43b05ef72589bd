"""Per-simulation timeline of the 16 tree warps of CTA 0 of the persistent search kernel (psearch.cuh: Trace; globaltimer ns) -- a
measurement aid.
Usage (on a B200): python profiles/trace_psearch.py [c2|c4] [num_simulations]"""
import ctypes as C
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import bench
from e_alphazero_b200 import _lib, ops
from e_alphazero_b200.selfplay import SelfplayRunner

wl = sys.argv[1] if len(sys.argv) > 1 else "c2"
kind, kw, B, n, gamma, desc = bench.WORKLOADS[wl]
if len(sys.argv) > 2:
    n = int(sys.argv[2])
envp, netp = bench.synth_params(kind, kw, 0)
env = ops.deepsea_spec(envp["size"], envp["action_map"])
net = ops.FcParams.from_numpy(netp["w"], netp["b"], netp["binary_set"], netp["num_actions"], 24, netp["hash_io"], netp["word_size"])
runner = SelfplayRunner(env, net, B, n, gamma, exploration_beta=1.0, directed_exploration=True, mlp_mode=1, fused_root=True)
states = ops.env_init(env, B)
for _ in range(4):
    states, _ = runner.step(states)
torch.cuda.synchronize()
buf = torch.zeros(n * 128 + 256, dtype=torch.int64, device="cuda")
lib = _lib.load()
lib.eaz_debug_set_ps_trace(C.c_void_p(buf.data_ptr()))
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
states, _ = runner.step(states)
e1.record()
torch.cuda.synchronize()
lib.eaz_debug_set_ps_trace(None)
raw = buf.cpu().numpy().astype(np.int64)[: n * 128].reshape(n, 16, 8)
L = raw[:, :, 5] & 0xFFFFFFFF
direct = (raw[:, :, 5] >> 32) != 0
# phases of simulation `it` of one warp: table wait + expand = expand done - staging done of it - 1; then backward, refresh, descent
# (the next leaf's table load is issued at its end) and staging; period = descent done of it - descent done of it - 1
ok = ~direct[1:] & ~direct[:-1] & (raw[1:, :, 3] > 0) & (raw[:-1, :, 4] > 0)
cur, prev = raw[1:], raw[:-1]
phases = {
    "expand": cur[:, :, 0] - prev[:, :, 4],
    "backward": cur[:, :, 1] - cur[:, :, 0],
    "refresh": cur[:, :, 2] - cur[:, :, 1],
    "descent": cur[:, :, 3] - cur[:, :, 2],
    "stage": cur[:, :, 4] - cur[:, :, 3],
}
period = cur[:, :, 3] - prev[:, :, 3]
print(f"{desc}: step {e0.elapsed_time(e1):.3f} ms; CTA 0, 16 tree warps x {n} simulations ({int(direct.sum())} warp-steps DIRECT)")
print("per-simulation period and phases of a warp, ns (staged simulations whose predecessor was staged as well): mean / median / p90")
for name, v in [("period", period)] + list(phases.items()):
    x = v[ok]
    print(f"  {name:9s} {x.mean():8.0f} {np.median(x):8.0f} {np.percentile(x, 90):8.0f}")
print("  it  period (mean over warps)  " + " ".join(f"{k:>8s}" for k in phases) + "   Lmax")
for it in range(1, n - 1):
    if it < 6 or it % 8 == 0 or it >= n - 3:
        m = ok[it - 1]
        if not m.any():
            continue
        print(f"{it:4d} {period[it - 1][m].mean():10.0f}              " + " ".join(f"{v[it - 1][m].mean():8.0f}" for v in phases.values()) +
              f"   {int(L[it].max()):4d}")
dd = np.where(raw[:, :, 3] > 0, raw[:, :, 3], np.nan)  # (0: a DIRECT step)
span = np.nanmax(dd, axis=1) - np.nanmin(dd, axis=1)
print(f"spread of 'descent done' across the 16 warps of a simulation: mean {np.nanmean(span[1:-1]):.0f} ns (warps are not synchronised)")
