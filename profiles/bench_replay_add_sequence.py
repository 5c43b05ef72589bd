"""Times putting one self-play scan's T' time steps into a prioritised replay ring of 1024 slots, three ways, with CUDA events
after warm-up (the ring is full and wrapping when timing starts):

    (a) what a torch caller does without add_sequence: T' x (ops.env_uncompact of row t of the scan's compact records, ring.add)
    (b) T' x ring.add of state dicts that are already decoded
    (c) one ring.add_sequence(dict(compact=[T',B,S], rewards=[T',B])), the scan's SelfplayOutput.state

Each is timed over `--calls` back-to-back repetitions (us per scan, host launch cost included: that is what the caller waits for), the
three alternating for `--rounds` rounds; the medians are reported.  The rows are the states of T' steps of random auto-reset play.
Workloads: DeepSea-30 (T'=8, B=4096), DeepSea-100 (T'=8, B=8192), Subleq-16 (T'=32, B=8192).  Prints the card's name and power limit
beside the numbers, one JSON line per workload.

    python profiles/bench_replay_add_sequence.py [--calls 50] [--rounds 5]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = [("deepsea-30", 8, 4096), ("deepsea-100", 8, 8192), ("subleq-16", 32, 8192)]
T_RING = 1024


def card():
    import torch

    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the number is still printed, with the reason the limit is missing
        pl = f"unknown ({e})"
    return torch.cuda.get_device_name(), pl


def timed(fn, calls):
    import torch

    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(calls):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1000.0 / calls  # us per scan


def env_of(name):
    import numpy as np

    from e_alphazero_b200 import ops

    kind, size = name.split("-")
    if kind == "deepsea":
        n = int(size)
        return ops.deepsea_spec(n, (np.random.default_rng(n).random((n, n)) < 0.5).astype(np.uint8))
    return ops.subleq_spec(int(size))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    import torch

    from e_alphazero_b200 import _abi, ops
    from e_alphazero_b200.replay import PrioritisedReplayRing

    assert torch.cuda.is_available(), "bench_replay_add_sequence.py measures on the GPU"
    name, power = card()
    for env_name, Tp, B in WORKLOADS:
        env = env_of(env_name)
        g = torch.Generator(device="cuda").manual_seed(Tp * B)
        subleq = env.kind == _abi.ENV_SUBLEQ
        tasks = lambda: torch.randint(1, 4, (B,), dtype=torch.int32, device="cuda", generator=g) if subleq else None
        st = ops.env_init(env, B, task_ids=tasks())
        rows = []
        for _ in range(Tp):  # the states after each of T' auto-reset steps of random play
            act = torch.randint(0, env.num_actions, (B,), dtype=torch.int32, device="cuda", generator=g)
            st = ops.env_step(env, st, act, auto_reset=True, task_ids=tasks())
            rows.append(st)
        compact = torch.stack([ops.env_compact(env, r) for r in rows]).contiguous()
        rewards = torch.stack([r["rewards"][:, 0] for r in rows]).contiguous()
        scan_state = dict(compact=compact, rewards=rewards)
        ring = PrioritisedReplayRing(env, T_RING, B, priority_exponent=0.6, seed=1)
        for _ in range(T_RING // Tp + 1):  # full and wrapped before anything is timed
            ring.add_sequence(scan_state)

        def decode_and_add():
            for t in range(Tp):
                ring.add(ops.env_uncompact(env, compact[t], rewards[t]))

        def add_decoded():
            for r in rows:
                ring.add(r)

        ways = dict(a_uncompact_add=decode_and_add, b_add=add_decoded, c_add_sequence=lambda: ring.add_sequence(scan_state))
        for fn in ways.values():  # warm-up: module loads, allocator pools
            for _ in range(3):
                fn()
        got = {k: [] for k in ways}
        for _ in range(args.rounds):
            for k, fn in ways.items():
                got[k].append(timed(fn, args.calls))
        ring.numeric_status()
        med = {k: statistics.median(v) for k, v in got.items()}
        print(json.dumps(dict(card=name, power_limit=power, env=env_name, steps=Tp, B=B, S=env.compact_bytes, T_ring=T_RING,
                              calls=args.calls, rounds=args.rounds, **{f"{k}_us": round(v, 1) for k, v in med.items()},
                              spread_us={k: [round(min(v), 1), round(max(v), 1)] for k, v in got.items()},
                              c_over_a=round(med["c_add_sequence"] / med["a_uncompact_add"], 3),
                              c_over_b=round(med["c_add_sequence"] / med["b_add"], 3))), flush=True)
        del ring, compact, rewards, rows, scan_state
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
