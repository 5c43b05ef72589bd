"""Wall time of one evaluate() call: the former per-move host loop (search, env step and `+=` per move, with `terminated.all().item()`
blocking the host before every move) against eaz_evaluate's CUDA graph (one launch; the device decides when the loop stops).

    python profiles/bench_evaluate.py [--reps 5] [--out profiles/r4_bench_evaluate.jsonl]

Workloads: DeepSea-30 x 4096 episodes x 64 simulations (tensor-core network) and Subleq-16 x 8192 episodes x 64 simulations (exact and
tensor-core network), random fully connected networks (hidden 256, the reference's linear_layer_size).  The two paths alternate within one process,
after a warm-up call of each (the graph is built there); each sample is host time around one call ending in a device synchronise.
Both paths must return the same sums of rewards bit for bit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def random_net(ops, env, hidden=256, seed=0):
    rng = np.random.default_rng(seed)
    D, A = env.obs_dim, env.num_actions
    w, b = [], []
    for h in range(4):
        out = A if h >= 2 else 1
        dims = [(D, hidden), (hidden, hidden), (hidden, out)]
        w.append([(rng.standard_normal(d) / np.sqrt(d[0])).astype(np.float32) for d in dims])
        b.append([(0.1 * rng.standard_normal(d[1])).astype(np.float32) for d in dims])
    bset = ((rng.random(1 << 21) < 0.5) * rng.integers(1, 256, 1 << 21)).astype(np.uint8)
    hash_io = int(env.kind == 1)
    return ops.FcParams.from_numpy(w, b, bset, A, hash_io=hash_io, word_size=env.word_size)


def host_loop(torch, _abi, ops, net, env, B, n, discount, max_len, mlp_mode, tasks, seed=0):
    """evaluate() before the device loop (the loop body of the former evaluate.py)."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    task_ids = None
    if env.kind == _abi.ENV_SUBLEQ:
        tt = torch.tensor(list(tasks), dtype=torch.int32, device="cuda")
        task_ids = tt[torch.randint(0, tt.numel(), (B,), device="cuda", generator=gen)].contiguous()
    states = ops.env_init(env, B, task_ids=task_ids)
    cfg = _abi.default_search_config(batch=B, num_simulations=n, discount=discount, exploration=0, gumbel_scale=0.0, mlp_mode=mlp_mode)
    plan = ops.SearchPlan(cfg, env, net, want_tree=False)
    beta = torch.zeros(B, device="cuda")
    gumbel = torch.zeros((B, env.num_actions), device="cuda")
    total = torch.zeros(B, device="cuda")
    counter = 0
    while not bool(states["terminated"].all().item()) and counter <= max_len:
        out = plan.run(dict(beta=beta, embedding=states, gumbel=gumbel), reuse_prepared=counter > 0)
        states = ops.env_step(env, states, out["action"])
        total += states["rewards"][:, 0]
        counter += 1
    return total, counter


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    from e_alphazero_b200 import _abi, ops
    from e_alphazero_b200.evaluate import EvaluateRunner

    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    rows = []
    for name, env, B, mode, tasks in (("deepsea30_tensor", ops.deepsea_spec(30, np.random.default_rng(1).random((30, 30)) < 0.5), 4096,
                                       _abi.MLP_TENSOR, (1,)),
                                      ("subleq16_exact", ops.subleq_spec(16), 8192, _abi.MLP_EXACT, (1, 2, 3)),
                                      ("subleq16_tensor", ops.subleq_spec(16), 8192, _abi.MLP_TENSOR, (1, 2, 3))):
        n, discount, max_len = 64, 0.997, 1000
        net = random_net(ops, env)
        runner = EvaluateRunner(net, env, B, n, discount, max_len, 0.0, True, mode, tasks)
        # warm-up of both paths (graph build, module loads), and the equality of their results
        exp, moves = host_loop(torch, _abi, ops, net, env, B, n, discount, max_len, mode, tasks)
        _, got = runner(0)
        torch.cuda.synchronize()
        assert torch.equal(got, exp) and runner.plan.moves() == moves, name
        t_host, t_graph = [], []
        for _ in range(a.reps):
            for path in ("host", "graph"):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if path == "host":
                    host_loop(torch, _abi, ops, net, env, B, n, discount, max_len, mode, tasks)
                else:
                    runner(0)
                torch.cuda.synchronize()
                (t_host if path == "host" else t_graph).append((time.perf_counter() - t0) * 1e3)
        row = dict(workload=name, episodes=B, simulations=n, moves=moves, host_loop_ms=t_host, graph_ms=t_graph,
                   host_loop_median_ms=float(np.median(t_host)), graph_median_ms=float(np.median(t_graph)),
                   speedup=float(np.median(t_host) / np.median(t_graph)), card=card)
        print(json.dumps(row), flush=True)
        rows.append(row)
    if a.out:
        with open(a.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
