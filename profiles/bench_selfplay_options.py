"""Cost of the self-play step options (uniform root prior, action drawn from the visit counts / improved policy) at the C2 / C3 shapes: the
time of one SelfplayRunner step (CUDA graph, fused root, tables reused) with each option against the options off, from CUDA events --
a measurement aid.  Each setting is timed in rounds that alternate with the options-off runner; the card and its power limit are
printed with the numbers.  Usage (on a B200): python profiles/bench_selfplay_options.py [--steps 50] [--rounds 3]"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from e_alphazero_b200 import _abi, ops
from e_alphazero_b200.selfplay import SelfplayRunner
from tests import helpers as H

OPTIONS = [("off", False, "search"), ("uniform_prior", True, "search"), ("visit_counts", False, "visit_counts"),
           ("improved_policy", False, "improved_policy"), ("uniform+improved", True, "improved_policy")]
SHAPES = {"c2": ("deepsea", dict(size=30), 4096, 64, 0.997, 3), "c3": ("subleq", dict(word_size=16), 8192, 64, 0.97, 3)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def time_steps(r, st, tasks, steps):
    for _ in range(3):
        st, _ = r.step(st, task_ids=tasks)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        st, _ = r.step(st, task_ids=tasks)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--shapes", default="c2,c3")
    args = ap.parse_args()
    print(f"card: {card()}")
    for shape in args.shapes.split(","):
        kind, kw, B, n, gamma, streams = SHAPES[shape]
        env = H.make_env(kind, seed=1, **kw)
        net = H.make_net(env, seed=2, fill=0.5)
        denv, dnet = H.device_env(env), H.device_net(net)
        tasks = torch.ones(B, dtype=torch.int32, device="cuda") if kind == "subleq" else None
        runners = {name: SelfplayRunner(denv, dnet, B, n, gamma, exploration_beta=1.0, directed_exploration=True, mlp_mode=_abi.MLP_TENSOR,
                                        use_graph=True, fused_root=True, streams=streams, device_noise=True, seed=3, uniform_prior=uni,
                                        action_sampling=samp)
                   for name, uni, samp in OPTIONS}
        states = {name: ops.env_init(denv, B, task_ids=tasks) for name in runners}
        ms = {name: [] for name in runners}
        for _ in range(args.rounds):
            for name in runners:
                if name != "off":  # alternate every option with the options-off runner
                    ms["off"].append(time_steps(runners["off"], states["off"], tasks, args.steps))
                ms[name].append(time_steps(runners[name], states[name], tasks, args.steps))
        base = min(ms["off"])
        for name in runners:
            t = ms[name]
            print(f"{shape} {kind} {B} x {n}: {name:17s} min {min(t):.3f} ms / step (runs {', '.join(f'{x:.3f}' for x in t)}), "
                  f"{100 * (min(t) / base - 1):+.1f} % vs off")


if __name__ == "__main__":
    main()
