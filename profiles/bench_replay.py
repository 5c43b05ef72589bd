"""Times the prioritised replay ring (csrc/replay.cu) on the GPU with CUDA events: sample(4096) including the gather and the
decode of both states, set_priorities(4096), and add(), each averaged over many calls after warm-up.  As a baseline for the
same draw (the same stratified u values over the same weights) it times torch cumsum + searchsorted over the flat weight
vector.  Rings of T x 4096 DeepSea-30 envs for T = 64, 1024, 4096 (the last tree, with its 64 MB of leaves plus the ring's
states and rewards, is larger than the 126 MB L2).  Prints the card's name and power limit beside the numbers, one JSON line
per ring.

    python profiles/bench_replay.py [--calls 200] [--sizes 64,1024,4096]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch

    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the number is still printed, with the reason the limit is missing
        pl = f"unknown ({e})"
    return torch.cuda.get_device_name(), pl


def timed(fn, calls, warmup=10):
    import torch

    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(calls):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1000.0 / calls  # us per call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--sizes", default="64,1024,4096")
    ap.add_argument("--batch", type=int, default=4096)
    args = ap.parse_args()
    import numpy as np
    import torch

    from e_alphazero_b200 import ops
    from e_alphazero_b200.replay import PrioritisedReplayRing

    assert torch.cuda.is_available(), "bench_replay.py measures on the GPU"
    name, power = card()
    B, K = 4096, args.batch
    env = ops.deepsea_spec(30)
    st = ops.env_init(env, B)
    for T in (int(x) for x in args.sizes.split(",")):
        ring = PrioritisedReplayRing(env, T, B, priority_exponent=0.6, seed=1)
        for _ in range(T):
            ring.add(st)
        N = T * B
        g = torch.Generator(device="cuda").manual_seed(T)
        all_idx = torch.arange(N, dtype=torch.int32, device="cuda")
        ring.set_priorities(all_idx, torch.rand(N, device="cuda", generator=g) * 4)
        out = ring.alloc_sample(K)
        idx = torch.randint(0, N, (K,), dtype=torch.int32, device="cuda", generator=g)
        pri = torch.rand(K, device="cuda", generator=g) * 4
        t_sample = timed(lambda: ring.sample(K, out=out), args.calls)
        t_set = timed(lambda: ring.set_priorities(idx, pri), args.calls)
        t_add = timed(lambda: ring.add(st), args.calls)
        # baseline for the same draw: flat weights, inclusive cumsum, stratified u, searchsorted, probability = w / total
        lv0 = (256 + 4 * N + 127) // 128 * 128
        w = ring.tree[lv0:lv0 + 4 * N].view(torch.float32)
        ks = torch.arange(K, device="cuda", dtype=torch.float32)
        r = torch.rand(K, device="cuda", generator=g)

        def baseline():
            c = torch.cumsum(w, 0)
            total = c[-1]
            u = (ks + r) / K * total
            i = torch.searchsorted(c, u, right=True).clamp_(max=N - 1)
            return i, w[i] / total

        t_base = timed(baseline, args.calls)
        ring.numeric_status()
        print(json.dumps(dict(card=name, power_limit=power, env="deepsea-30", T=T, B=B, items=N, batch=K, calls=args.calls,
                              tree_mb=round(ring.tree.numel() / 2 ** 20, 1),
                              sample_gather_decode_us=round(t_sample, 2), set_priorities_us=round(t_set, 2), add_us=round(t_add, 2),
                              torch_cumsum_searchsorted_us=round(t_base, 2),
                              faster_draw="sum tree" if t_sample < t_base else "cumsum+searchsorted")), flush=True)
        del ring, out, w
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
