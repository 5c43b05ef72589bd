"""Wall time of one self-play scan of T steps: the best host protocol before eaz_selfplay -- T replays of the CUDA graph of
SelfplayRunner(use_graph=True, fused_root=True, device_noise=True), each followed by trajectory() into a [T,B,4] buffer -- against
SelfplayRunner.scan() (one launch of eaz_selfplay's graph; the device runs the T steps and stops the loop).

    python profiles/bench_selfplay_scan.py [--reps 7] [--out profiles/r6_bench_selfplay_scan.jsonl]

Workloads (tensor-core network, random fully connected networks of hidden 256, the reference's linear_layer_size): DeepSea-30 x 4096 x
64 simulations, T = 8; DeepSea-100 x 8192 x 128, T = 8; Subleq-16 x 8192 x 64, T = 32 (selfplay_steps of DeepSea / the default,
config.py:37,105).  Before every scan both runners are told the parameters changed (a learner update separates two scans), so both
rebuild the parameter-derived tables once per scan.  The two paths alternate within one process after a warm-up scan of each; each
sample is host time around one scan ending in a device synchronise.  The warm-up scans start from the same states with the draw
counters at 0, so their DeepSea trajectory records must agree bit for bit (the Subleq reset tasks are drawn differently)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    from bench_evaluate import random_net
    from e_alphazero_b200 import _abi, ops
    from e_alphazero_b200.selfplay import SelfplayRunner

    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    rows = []
    for name, env, B, n, T, tasks in (("deepsea30", ops.deepsea_spec(30, np.random.default_rng(1).random((30, 30)) < 0.5), 4096, 64, 8, (1,)),
                                      ("deepsea100", ops.deepsea_spec(100, np.random.default_rng(2).random((100, 100)) < 0.5), 8192, 128, 8, (1,)),
                                      ("subleq16", ops.subleq_spec(16), 8192, 64, 32, (1, 2, 3))):
        net = random_net(ops, env)
        kw = dict(exploration_beta=0.5, directed_exploration=True, mlp_mode=_abi.MLP_TENSOR, tasks=tasks, fused_root=True, device_noise=True,
                  seed=5)
        host = SelfplayRunner(env, net, B, n, 0.997, use_graph=True, **kw)
        scan = SelfplayRunner(env, net, B, n, 0.997, **kw)
        host.plan.workspace.zero_()  # draw counters at 0 in both (the scan's workspace starts zeroed)
        g = torch.Generator(device="cuda").manual_seed(3)
        init_tasks = torch.tensor(tasks, dtype=torch.int32, device="cuda")[torch.randint(0, len(tasks), (B,), device="cuda", generator=g)]
        init = ops.env_init(env, B, task_ids=init_tasks if env.kind == _abi.ENV_SUBLEQ else None)
        traj = torch.empty((T, B, 4), dtype=torch.int32, device="cuda")
        scan_states = {k: v.clone() for k, v in init.items()}
        host_states = {k: v.clone() for k, v in init.items()}  # (until the first step has made the graph's own state buffers)

        def run_host():
            st = host.static_states() if host.static_states() is not None else host_states
            for t in range(T):
                _, out = host.step(st)
                host.trajectory(st, out, traj[t])

        def reset():
            host.params_updated()
            scan.params_updated()
            if host.static_states() is not None:
                for k, v in host.static_states().items():
                    v.copy_(init[k])
            for k, v in scan_states.items():
                v.copy_(init[k])
            torch.cuda.synchronize()

        reset()
        run_host()
        _, out = scan.scan(scan_states, T)
        torch.cuda.synchronize()
        # (Subleq: the reset tasks come from each runner's generator in different calls -- T draws of [B] against one of [T,B] -- so
        # only the DeepSea records are comparable)
        same = bool(torch.equal(traj, out.trajectory)) if env.kind == _abi.ENV_DEEPSEA else None
        if same is False:
            raise AssertionError(f"{name}: the scan's trajectory records differ from the host protocol's")
        t_host, t_scan = [], []
        for _ in range(a.reps):
            for path in ("host", "scan"):
                reset()
                t0 = time.perf_counter()
                if path == "host":
                    run_host()
                else:
                    scan.scan(scan_states, T)
                torch.cuda.synchronize()
                (t_host if path == "host" else t_scan).append((time.perf_counter() - t0) * 1e3)
        row = dict(workload=name, envs=B, simulations=n, steps=T, mlp_mode="tensor", host_replays_ms=t_host, scan_ms=t_scan,
                   host_replays_median_ms=float(np.median(t_host)), scan_median_ms=float(np.median(t_scan)),
                   speedup=float(np.median(t_host) / np.median(t_scan)), outputs_identical=same, card=card)
        print(json.dumps(row), flush=True)
        rows.append(row)
    if a.out:
        with open(a.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
