"""Device time of the per-model DeepSea output table (psearch.cuh: ds_output_table_kernel) and of the persistent search kernel, from a
torch.profiler run of self-play steps that each rebuild the parameter-derived tables -- a measurement aid.
Usage (on a B200): python profiles/time_ds_table.py [c2] [c4] ...   (one JSON line per workload)"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from torch.profiler import ProfilerActivity, profile

import bench
from e_alphazero_b200 import ops
from e_alphazero_b200.selfplay import SelfplayRunner

for wl in sys.argv[1:] or ["c2", "c4"]:
    kind, kw, B, n, gamma, desc = bench.WORKLOADS[wl]
    envp, netp = bench.synth_params(kind, kw, 0)
    env = ops.deepsea_spec(envp["size"], envp["action_map"])
    net = ops.FcParams.from_numpy(netp["w"], netp["b"], netp["binary_set"], netp["num_actions"], 24, netp["hash_io"], netp["word_size"])
    runner = SelfplayRunner(env, net, B, n, gamma, exploration_beta=1.0, directed_exploration=True, mlp_mode=1, fused_root=True, use_graph=False)
    states = ops.env_init(env, B)
    for _ in range(3):
        states, _ = runner.step(states)
    torch.cuda.synchronize()
    steps = 10
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            runner.params_updated()  # every step rebuilds the tables
            states, _ = runner.step(states)
        torch.cuda.synchronize()
    times = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            for name in ("ds_output_table_kernel", "ds_search_kernel"):
                if name in ev.name:
                    times.setdefault(name, []).append(ev.device_time)
    out = {"workload": wl, "desc": desc, "gpu": torch.cuda.get_device_name(), "steps": steps}
    for name, v in times.items():
        out[name] = {"launches": len(v), "mean_us": sum(v) / len(v), "min_us": min(v), "max_us": max(v)}
    print(json.dumps(out))
