#!/usr/bin/env python
"""bench.py -- self-play env-steps/s including the E-MCTS search (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2|c1|c3] [--dump-outputs DIR]

One "step" = one self-play move for a whole batch of envs: root network forward -> E-MCTS search
(num_simulations x select/expand/backward with env step, hash probe and network per simulation) ->
auto-reset env step (reference: selfplay.py:86-143).  Default workload = BASELINE config C2
(DeepSea size=30, 4096 envs per GPU, 64 simulations, UBE variance propagation on).

Prints ONE JSON line.  `value` is measured with inputs resident in HBM; `e2e` goes through host
buffers (pinned H2D of the states, D2H of the step's results inside the timed region).
`--impl reference` times the CPU restatement of the reference (oracle/, all host threads) on a
bounded sample of the same workload: JAX/emctx/pgx are not installable in this image, so the
reference's own JAX-CPU path cannot be run (DESIGN.md "CPU baseline").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (env kind, env kwargs, envs per GPU, simulations, discount, description)
    "c1": ("deepsea", dict(size=10), 64, 32, 0.997, "C1: DeepSea size=10, 64 envs, 32 simulations"),
    "c2": ("deepsea", dict(size=30), 4096, 64, 0.997, "C2: DeepSea size=30, 4096 envs/GPU, 64 simulations, UBE variance propagation on"),
    "c3": ("subleq", dict(word_size=16), 8192, 64, 0.97, "C3: Subleq ws=16 binary, 8192 envs/GPU, 64 simulations, hash-count novelty on (IO hash)"),
    "c4": ("deepsea", dict(size=100), 8192, 128, 0.997, "C4: DeepSea size=100, 8192 envs/GPU, 128 simulations"),
}
METRIC = "selfplay_env_steps_per_s_incl_emcts_search"
UNIT = "env-steps/s"


def synth_params(kind, kw, seed=0):
    """Synthetic env + random-init network as host arrays (same generator for both arms)."""
    rng = np.random.default_rng(seed)
    if kind == "deepsea":
        N = kw["size"]
        env = dict(kind="deepsea", size=N, action_map=(rng.random((N, N)) < 0.5).astype(np.uint8))
        D, A, hash_io, ws = N * N, 2, 0, 0
    else:
        ws = kw["word_size"]
        w = (ws - 1).bit_length() + 1
        env = dict(kind="subleq", word_size=ws)
        D, A, hash_io = (ws + 32) * w, ws, 1
    H = 256
    W, Bv = [], []
    for h in range(4):
        outs, ins = [H, H, 1 if h < 2 else A], [D, H, H]
        W.append([np.ascontiguousarray(rng.standard_normal((i, o)).clip(-2, 2) / np.sqrt(i), np.float32) for i, o in zip(ins, outs)])
        Bv.append([np.ascontiguousarray(rng.standard_normal(o) * 0.05, np.float32) for o in outs])
    bset = ((rng.random(1 << 21) < 0.5) * rng.integers(1, 256, 1 << 21)).astype(np.uint8)  # ~half of the states "seen"
    return env, dict(w=W, b=Bv, binary_set=bset, num_actions=A, hash_io=hash_io, word_size=ws, in_dim=D)


class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region (B200_PROFILING.md): an NVML polling thread (about one sample
    per millisecond -- `nvidia-smi -lms` cannot sample a region of a few tens of milliseconds), started a second before the region."""

    REASONS = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40), ("hw_power_brake_slowdown", 0x80),
               ("sw_power_cap", 0x4))

    def __init__(self, torch_device_index):
        self.rows, self.stop_flag, self.thread, self.h, self.nv = [], False, None, None, None
        try:
            import pynvml as nv
            import torch

            nv.nvmlInit()
            try:
                uuid = str(torch.cuda.get_device_properties(torch_device_index).uuid)
                self.h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:  # noqa: BLE001 -- older torch / NVML: fall back to the ordinal
                self.h = nv.nvmlDeviceGetHandleByIndex(torch_device_index)
            self.nv = nv
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def _poll(self):
        nv, h = self.nv, self.h
        while not self.stop_flag:
            try:
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except AttributeError:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((time.time(), nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetPowerUsage(h) / 1000.0, int(reasons)))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.0008)

    def start(self):
        if self.nv is None:
            return
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()

    def stop(self, t0, t1):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable: " + getattr(self, "err", "?")]}
        self.stop_flag = True
        self.thread.join(timeout=1.0)
        rows = [r for r in self.rows if t0 <= r[0] <= t1]
        where = "timed region"
        if not rows:  # region shorter than one polling interval: the samples closest to it
            rows, where = [r for r in self.rows if t0 - 0.05 <= r[0] <= t1 + 0.05], "timed region +- 50 ms"
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(r[1] for r in rows)
        mask = 0
        for r in rows:
            mask |= r[3]
        return {"sm_mhz": float(sm[len(sm) // 2]), "sm_max_mhz": float(self.nv.nvmlDeviceGetMaxClockInfo(self.h, self.nv.NVML_CLOCK_SM)),
                "power_w_max": max(r[2] for r in rows), "samples": len(rows), "sampled": where + " (NVML, ~1 ms period)",
                "reasons": [name for name, bit in self.REASONS if mask & bit]}


def workload_config(desc, B, n):
    """The workload-defining part of `config`, identical in both arms (the driver compares the two lines)."""
    return {"workload": desc, "envs_per_gpu": B, "num_simulations": n, "directed_exploration": True, "beta": "linspace(0,1,B)",
            "l2": "GPU arm: flushed between timed steps (256 MiB write); CPU arm: not applicable"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, "fallback"  # B200_PROFILING.md fallback


# ============================================================================== reference arm / cpu baseline (oracle)
def oracle_step_time(kind, kw, n, gamma, B_sample, seed, repeats=1):
    """Time `repeats` self-play steps of the CPU restatement on B_sample envs; returns seconds per step."""
    from e_alphazero_b200 import _abi
    from oracle import oracle as O

    envp, netp = synth_params(kind, kw, 0)
    env = O.Env.deepsea(envp["size"], envp["action_map"]) if kind == "deepsea" else O.Env.subleq(envp["word_size"], True)
    net = O.FcNet(netp["in_dim"], 256, netp["num_actions"], netp["w"], netp["b"], netp["binary_set"], 24, netp["hash_io"], netp["word_size"])
    rng = np.random.default_rng(seed)
    A = env.num_actions
    st = O.env_init(env, B_sample, rng.integers(1, 2, B_sample))
    for _ in range(3):  # decorrelate depths
        st = O.env_step(env, st, rng.integers(0, A, B_sample), auto_reset=True, task_ids=np.ones(B_sample, np.int32))
    beta = np.linspace(0, 1, B_sample).astype(np.float32)
    cfg = _abi.default_search_config(num_simulations=n, discount=gamma, exploration=1)
    t0 = time.perf_counter()
    for _ in range(repeats):
        ev = O.mlp_forward_states(net, env, st)
        root = dict(prior_logits=ev["explore_logits"], value=ev["value"], value_epistemic_variance=ev["ube"], beta=beta, embedding=st,
                    gumbel=rng.gumbel(size=(B_sample, A)).astype(np.float32))
        out = O.search(cfg, env, net, root, want_tree=False)
        st = O.env_step(env, st, out["action"], auto_reset=True, task_ids=np.ones(B_sample, np.int32))
    return (time.perf_counter() - t0) / repeats


def cpu_baseline(kind, kw, n, gamma, budget_s=12.0):
    from oracle import oracle as O

    O.build()
    cores = O.set_threads(os.cpu_count() or 1)
    probe_B = max(cores * 4, 32)
    t = oracle_step_time(kind, kw, n, gamma, probe_B, seed=1)
    B_sample = int(min(4096, max(probe_B, probe_B * budget_s / max(t, 1e-3))))
    B_sample -= B_sample % max(cores, 1) or 0
    t = oracle_step_time(kind, kw, n, gamma, B_sample, seed=2)
    return {"value": B_sample / t, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{B_sample} envs x 1 self-play step ({n} simulations) of the same workload, {t:.2f} s, OpenMP over envs",
            "simulations_per_s": B_sample * n / t}


def run_reference(args, kind, kw, B, n, gamma, desc):
    """The reference's CPU implementation of the path (the C/OpenMP restatement: JAX / emctx / pgx are not installable here), all host
    threads, on THIS workload at FULL size: every step searches all B envs (the same config as the GPU arm).  At ~1.4 k env-steps/s
    on 16 cores a C2 step takes ~3 s, so K + W steps stay within a few minutes; only if a probe shows that the whole run would take
    longer than ~6 minutes is the per-step batch cut (and `config.envs_per_gpu` then says so)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O

    O.build()
    cores = O.set_threads(os.cpu_count() or 1)
    probe_B = max(cores * 4, 32)
    t = oracle_step_time(kind, kw, n, gamma, probe_B, seed=1)
    est = t / probe_B * B * (args.steps + args.warmup)
    B_sample = B if est <= 360.0 else max(cores, int(B * 360.0 / est) // cores * cores)
    for _ in range(args.warmup):
        oracle_step_time(kind, kw, n, gamma, B_sample, seed=3)
    t0 = time.perf_counter()
    for i in range(args.steps):
        oracle_step_time(kind, kw, n, gamma, B_sample, seed=10 + i)
    dt = time.perf_counter() - t0
    value = B_sample * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(desc, B_sample, n),
            "notes": {"arm": "CPU restatement of the reference (oracle/eaz_oracle.c, OpenMP over envs), not JAX: jax/emctx/pgx are not installable here",
                      "full_batch": B_sample == B},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{B_sample} envs per step x {args.steps} steps ({n} simulations each)"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "simulations_per_s": value * n, "gpu_launches": 0}
    emit(line)


# ============================================================================== B200 arm
def extra_measure(args, name, dev, world, rank, steps=6, B_override=None, n_override=None):
    """Short device-timed measurement of another BASELINE workload for the `extra` block of the JSON line (same runner, same step;
    no e2e / trajectory legs): {"ms_per_step", "value", per-class ms of the search on rank 0}.  Max over ranks like the headline."""
    import torch
    import torch.distributed as dist

    from e_alphazero_b200 import ops
    from e_alphazero_b200.selfplay import SelfplayRunner

    kind, kw, B, n, gamma, desc = WORKLOADS[name]
    B, n = B_override or B, n_override or n
    envp, netp = synth_params(kind, kw, 0)
    env = ops.deepsea_spec(envp["size"], envp["action_map"], dev) if kind == "deepsea" else ops.subleq_spec(envp["word_size"], True)
    net = ops.FcParams.from_numpy(netp["w"], netp["b"], netp["binary_set"], netp["num_actions"], 24, netp["hash_io"], netp["word_size"], device=dev)
    streams = 1 if (kind == "deepsea" and B > 4096) else 3
    runner = SelfplayRunner(env, net, B, n, gamma, exploration_beta=1.0, directed_exploration=True, mlp_mode=args.mlp_mode, device=dev, seed=200 + rank,
                            use_graph=not args.no_graph, fused_root=not args.no_fused_root, streams=streams, device_noise=True)
    gen = torch.Generator(device=dev).manual_seed(17 + rank)
    states = ops.env_init(env, B, task_ids=torch.ones(B, dtype=torch.int32, device=dev) if kind == "subleq" else None, device=dev)
    for _ in range(3):
        states = ops.env_step(env, states, torch.randint(0, env.num_actions, (B,), device=dev, generator=gen, dtype=torch.int32))
    for _ in range(3):
        states, _ = runner.step(states)
    if runner.use_graph:
        states = runner.static_states()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    for i in range(steps):
        flush.zero_()
        ev[i][0].record()
        states, _ = runner.step(states)
        ev[i][1].record()
    torch.cuda.synchronize()
    ms = sum(a.elapsed_time(b) for a, b in ev)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    res = {"workload": desc if not (B_override or n_override) else f"{desc.split(':')[0]} shape at {B} envs/GPU x {n} simulations (self-play step)",
           "envs_per_gpu": B, "num_simulations": n, "steps": steps, "ms_per_step": ms / steps, "value": world * B * steps / (ms * 1e-3), "unit": UNIT,
           "simulations_per_s": world * B * n * steps / (ms * 1e-3), "streams": streams}
    if rank == 0:
        ev0 = ops.mlp_forward_states(net, env, states)
        root = dict(prior_logits=ev0["explore_logits"], value=ev0["value"], value_epistemic_variance=ev0["ube"], beta=runner.beta, embedding=states,
                    gumbel=runner.draw_gumbel())
        _, p = runner.plan.run(root, profile=True)
        res["per_class_ms"] = {k: round(v[0], 4) for k, v in p.items()}
        res["per_class_launches"] = {k: v[1] for k, v in p.items()}
        _, tf_peak, which = measured_peaks()
        D, H, A = netp["in_dim"], 256, env.num_actions
        l1 = 0 if kind == "deepsea" else 2 * D * H
        flops = (3 * (l1 + 2 * H * H) + 2 * (2 * H) + 2 * H * A) * B * n
        net_ms = p["network"][0] if p["network"][1] else p["select"][0]  # (persistent kernel: the network runs inside it)
        res["tensor_roofline"] = {"achieved": flops / (net_ms * 1e-3) / 1e12, "peak": tf_peak, "unit": "TFLOP/s", "frac": flops / (net_ms * 1e-3) / 1e12 / tf_peak,
                                  "peak_source": which, "ms_per_search": net_ms}
    del runner, flush
    torch.cuda.empty_cache()
    return res


def run_b200(args, kind, kw, B, n, gamma, desc):
    import torch
    import torch.distributed as dist

    from e_alphazero_b200 import _abi, ops
    from e_alphazero_b200.selfplay import SelfplayRunner

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl b200) needs a CUDA device: the CUDA library is the only implementation")
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(dev))

    envp, netp = synth_params(kind, kw, 0)
    env = ops.deepsea_spec(envp["size"], envp["action_map"], dev) if kind == "deepsea" else ops.subleq_spec(envp["word_size"], True)
    net = ops.FcParams.from_numpy(netp["w"], netp["b"], netp["binary_set"], netp["num_actions"], 24, netp["hash_io"], netp["word_size"], device=dev)
    if world > 1:  # parameter broadcast (learner -> actors), once per learner update: outside the timed region
        for h in range(4):
            for l in range(3):
                dist.broadcast(net.w[h][l], 0)
                dist.broadcast(net.b[h][l], 0)
        dist.broadcast(net.binary_set, 0)

    # shard = this rank's envs (weak scaling: B per GPU fixed); directed exploration with beta = linspace(0,1,B) (UBE on)
    runner = SelfplayRunner(env, net, B, n, gamma, exploration_beta=1.0, directed_exploration=True, mlp_mode=args.mlp_mode, device=dev, seed=100 + rank,
                            use_graph=not args.no_graph, fused_root=not args.no_fused_root, streams=args.streams, device_noise=True)
    gen = torch.Generator(device=dev).manual_seed(7 + rank)
    states = ops.env_init(env, B, task_ids=torch.ones(B, dtype=torch.int32, device=dev) if kind == "subleq" else None, device=dev)
    A = env.num_actions
    for _ in range(5 if kind == "deepsea" else 3):  # spread the envs over depths with random play (product env kernels)
        act = torch.randint(0, A, (B,), device=dev, generator=gen, dtype=torch.int32)
        keep = torch.rand(B, device=dev, generator=gen) < 0.5
        nxt = ops.env_step(env, states, act)
        for k in states:
            m = keep.reshape((-1,) + (1,) * (states[k].dim() - 1))
            states[k] = torch.where(m, nxt[k], states[k]).contiguous()

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    # Trajectory all-gather into the replay buffer (SURVEY 8e): like the reference, which gathers ONCE per selfplay() scan of
    # selfplay_steps steps (main.py:383-385), every step packs its 16-byte-per-env record into a [T,B,4] scan buffer (one small
    # kernel) and the all-gather of a finished scan runs on a side stream under the next scan's searches (double-buffered).
    T = args.param_refresh
    scan = [torch.empty((T, B, 4), dtype=torch.int32, device=dev) for _ in range(2)]
    gathered = [torch.empty((world, T, B, 4), dtype=torch.int32, device=dev) for _ in range(2)] if world > 1 else None
    side = torch.cuda.Stream(device=dev) if world > 1 else None
    gather_done = [None, None]
    tick = [0]
    record = [None]  # the trajectory record of the latest step (a view into the scan buffer)

    def one_step(st):
        i = tick[0]
        buf, row = (i // T) & 1, i % T
        if world > 1 and row == 0 and gather_done[buf] is not None:
            torch.cuda.current_stream().wait_event(gather_done[buf])  # the gather that last read this scan buffer has finished
        st, out = runner.step(st)
        record[0] = runner.trajectory(st, out, scan[buf][row])
        if world > 1 and row == T - 1:
            ready = torch.cuda.Event()
            ready.record()
            side.wait_event(ready)
            with torch.cuda.stream(side):
                dist.all_gather_into_tensor(gathered[buf].view(-1), scan[buf].view(-1))
                gather_done[buf] = torch.cuda.Event()
                gather_done[buf].record()
        tick[0] = i + 1
        return st, out

    def join_gathers():
        if world > 1:
            torch.cuda.current_stream().wait_stream(side)

    for _ in range(max(args.warmup, 3)):
        states, _ = one_step(states)
    if runner.use_graph:  # step the graph's own state buffers in place from here on (no copies in / out)
        states = runner.static_states()
    torch.cuda.synchronize()

    # ---- timed region: exactly K steps, CUDA events per step, L2 flushed between steps (outside the events)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for k in range(40):  # keep the GPU under this workload's load before the region, so that the sampled clocks are the loaded ones
        states, _ = one_step(states)
        if k % 8 == 7:
            torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_wall0 = time.time()
    for i in range(args.steps):
        flush.zero_()
        if i % args.param_refresh == 0:  # a new selfplay() call = possibly new parameters: rebuild the parameter-derived tables
            runner.params_updated()
        ev[i][0].record()
        states, out = one_step(states)
        ev[i][1].record()
    tail = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    tail[0].record()
    join_gathers()  # any all-gather still in flight is part of the job: its non-overlapped remainder is timed
    tail[1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_wall1 = time.time()
    ms_total = sum(a.elapsed_time(b) for a, b in ev) + tail[0].elapsed_time(tail[1])
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    value = world * B * args.steps / (ms_total * 1e-3)
    if args.dump_outputs:  # before the e2e leg below steps the same state and output buffers again
        arrays = {f"state_{k}": states[k] for k in ops.state_fields(env)}
        arrays.update((k, v) for k, v in vars(out).items() if k != "state")
        arrays["trajectory"] = record[0]
        dump_outputs(args.dump_outputs, arrays, prefix="" if world == 1 else f"rank{rank}_")

    # ---- e2e: host buffers in, host results out, copies inside the timed region (rank-local, max over ranks).
    # A graph runner keeps its state fields in one device arena and the search outputs in another (ops.alloc_arena), so a host caller
    # moves a step's inputs with ONE pinned copy and reads states + results back with two (SelfplayRunner.host_arenas);
    # without the graph the fields are copied one by one.
    fields = ops.state_fields(env)
    res_names = ("action", "root_value", "root_epistemic_std", "value_prediction", "ube_prediction", "q_values_epistemic_variance")
    e2e_ms, d2h = 0.0, 0
    if runner.use_graph and runner.fused_root:  # (with a separate root forward its predictions live outside the output arena)
        dstates = runner.static_states()
        hs_a, hv_a, host_res_flat, host_res = runner.host_arenas()
        hs_b, hv_b, _, _ = runner.host_arenas()
        hs_a.copy_(runner.static_flat)
        torch.cuda.synchronize()
        h2d = hs_a.numel()
        d2h = hs_b.numel() + host_res_flat.numel()
        for i in range(args.steps + 2):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if i >= 2 and (i - 2) % args.param_refresh == 0:
                runner.params_updated()
            a.record()
            runner.static_flat.copy_(hs_a, non_blocking=True)
            dstates, out = one_step(dstates)
            hs_b.copy_(runner.static_flat, non_blocking=True)
            host_res_flat.copy_(runner.plan.out_flat, non_blocking=True)  # action, root value / std, predictions, q variances, visit statistics
            join_gathers()
            b.record()
            torch.cuda.synchronize()
            if i >= 2:
                e2e_ms += a.elapsed_time(b)
            hs_a, hs_b = hs_b, hs_a
    else:
        host_in = {k: states[k].detach().cpu().pin_memory() for k in fields}
        host_out = {k: torch.empty_like(host_in[k]).pin_memory() for k in fields}
        h2d = sum(v.numel() * v.element_size() for v in host_in.values())
        dstates = runner.static_states() if runner.use_graph else {k: torch.empty_like(states[k]) for k in fields}
        host_res = None
        for i in range(args.steps + 2):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if i >= 2 and (i - 2) % args.param_refresh == 0:
                runner.params_updated()
            a.record()
            for k in fields:
                dstates[k].copy_(host_in[k], non_blocking=True)
            dstates, out = one_step(dstates)
            for k in fields:
                host_out[k].copy_(dstates[k], non_blocking=True)
            res = [getattr(out, nme) for nme in res_names]
            if host_res is None:
                host_res = [torch.empty_like(r, device="cpu").pin_memory() for r in res]
                d2h = sum(v.numel() * v.element_size() for v in host_out.values()) + sum(r.numel() * r.element_size() for r in res)
            for hr, r in zip(host_res, res):
                hr.copy_(r, non_blocking=True)
            join_gathers()
            b.record()
            torch.cuda.synchronize()
            if i >= 2:
                e2e_ms += a.elapsed_time(b)
            host_in, host_out = host_out, host_in
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = world * B * args.steps / (e2e_ms * 1e-3)

    # ---- roofline: per-kernel-class CUDA-event times of the search (measured live, rank 0), algorithmic bytes per SURVEY 8(d)
    roofline = None
    if rank == 0:
        ev0 = ops.mlp_forward_states(net, env, states)
        root = dict(prior_logits=ev0["explore_logits"], value=ev0["value"], value_epistemic_variance=ev0["ube"], beta=runner.beta,
                    embedding=states, gumbel=runner.draw_gumbel())
        tplan = ops.SearchPlan(_abi.default_search_config(batch=B, num_simulations=n, discount=gamma, exploration=1, mlp_mode=args.mlp_mode), env, net,
                               want_tree=True, device=dev)
        tout = tplan.run(root)
        V = int(tout["node_visits"][:, 1:].sum().item())  # edge traversals = sum over simulations of path depth
        del tplan
        prof = {}
        reps = 3
        for _ in range(reps):
            _, p = runner.plan.run(root, profile=True)
            for k, (ms, cnt) in p.items():
                prof[k] = (prof.get(k, (0.0, 0))[0] + ms / reps, cnt)
        S = env.compact_bytes
        tree_bytes = V * (32 * A + 68) + B * n * (2 * S + 4 * A + 44)
        io_bytes = B * (8 * A + A + 16 + S) + B * (4 + 20 * A + 8)
        tree_ms = prof["select"][0] + prof["expand_backward"][0] + prof["env_step"][0]
        persistent = kind == "deepsea" and args.mlp_mode == 1 and prof["select"][1] == 1  # ONE launch ran all simulations (psearch.cuh)
        hbm_peak, tf_peak, which = measured_peaks()
        D, H = netp["in_dim"], 256
        l1 = 0 if kind == "deepsea" else 2 * D * H  # one-hot DeepSea layer 1 is a row gather
        flops_fwd = 3 * (l1 + 2 * H * H) + 2 * (2 * H) + 2 * H * A  # 3 heads evaluated per node (value, UBE, one policy head)
        mlp_ms = prof["network"][0] + (tree_ms if persistent else 0.0)  # (persistent: the network runs inside the same kernel)
        tensor_kernel = "mlp_gather_kernel" if kind == "deepsea" else "mlp_tensor_kernel"  # one-hot rows: mlp_gather.cu
        if persistent:
            tensor_kernel = "ds_search_kernel"
        total_ms = sum(v[0] for v in prof.values())
        tree_gbs = (tree_bytes + io_bytes) / (tree_ms * 1e-3) / 1e9
        mlp_tfs = flops_fwd * B * n / (mlp_ms * 1e-3) / 1e12
        # speed-of-light floors of one search: the roof that binds is the one with the larger floor.  The persistent kernel does the
        # tree work AND the network in one launch, so both floors refer to the same duration; otherwise the class that takes longer.
        hbm_floor_us = (tree_bytes + io_bytes) / (hbm_peak * 1e9) * 1e6
        tensor_floor_us = flops_fwd * B * n / (tf_peak * 1e12) * 1e6
        if persistent:
            dominant = "network" if tensor_floor_us >= hbm_floor_us else "tree"
        else:
            dominant = "network" if mlp_ms >= tree_ms else "tree"
        tree_obj = {"bound": "hbm", "achieved": tree_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": tree_gbs / hbm_peak, "traffic": None,
                    "kernels": ("ds_search_kernel (persistent: all simulations of a 128-tree tile in one 4-CTA cluster -- tree steps, DeepSea transition AND "
                                "the tcgen05 network evaluation; its whole duration is charged to the tree bytes)") if persistent else
                               ("tree_step_kernel (expand + backward + action refresh + descent)" + (" + subleq_tree_step_kernel" if kind == "subleq" else "")),
                    "algorithmic_bytes_per_search": tree_bytes + io_bytes, "ms_per_search": tree_ms,
                    "avg_launch_us": 1e3 * tree_ms / max(prof["select"][1] + prof["expand_backward"][1] + prof["env_step"][1], 1),
                    "edge_traversals": V, "peak_source": which, "floor_us_per_search": hbm_floor_us}
        mlp_obj = {"bound": "tensor", "achieved": mlp_tfs, "peak": tf_peak, "unit": "TFLOP/s", "frac": mlp_tfs / tf_peak, "traffic": None,
                   "kernels": "mlp_exact_kernel (fp32 FMA chains, bit-exact mode)" if args.mlp_mode == 0 else f"{tensor_kernel} (tcgen05)",
                   "flops_per_search": flops_fwd * B * n, "ms_per_search": mlp_ms, "avg_launch_us": 1e3 * mlp_ms / max(prof["network"][1], 1),
                   "peak_source": which, "floor_us_per_search": tensor_floor_us}
        try:  # DRAM traffic per launch from the committed ncu --set full captures (profiles/r2_traffic.json, r1_traffic.json)
            traffic = {}
            for name in ("r1_traffic.json", "r2_traffic.json"):
                pth = os.path.join(ROOT, "profiles", name)
                if os.path.exists(pth):
                    traffic.update(json.load(open(pth)).get(args.workload, {}))
            tree_obj["traffic"] = traffic.get("ds_search_kernel" if persistent else "tree_step_kernel")
            mlp_obj["traffic"] = traffic.get(tensor_kernel) if args.mlp_mode == 1 else None
        except (OSError, ValueError):
            pass
        roofline = dict(mlp_obj if dominant == "network" else tree_obj)
        roofline["timing"] = ("CUDA events around every launch in a separate profiled pass of the same search on the same stream (eaz_search_gumbel_profiled)" +
                              ("; the persistent kernel is ONE launch per search, so its event time is its real duration" if persistent else
                               ": the events serialise the PDL chain and the sub-batch streams, so these durations are upper bounds -- in the timed region the "
                               "tree kernel stages its data under the network kernel and sub-batches overlap (value / ms_per_step is the overlapped time)"))
        roofline["dominant"] = dominant
        if persistent:
            roofline["note"] = ("one launch runs the tree steps and the network of all simulations; a simulation is a serial chain network -> backward -> "
                                "refresh -> descent per 128-tree tile (profiles/r2_summary.md 1.1), so the kernel is latency-bound: the tensor roof "
                                "(larger floor) is reported here, the HBM roof of the tree bytes under `other`")
        roofline["share_of_search_time"] = (mlp_ms if dominant == "network" else tree_ms) / total_ms
        roofline["other"] = tree_obj if dominant == "network" else mlp_obj
        roofline["per_class_ms"] = {k: round(v[0], 4) for k, v in prof.items()}
        roofline["per_class_launches"] = {k: v[1] for k, v in prof.items()}

    # ---- extra: the other BASELINE shapes next to the headline (short, device-timed, max over ranks): C4 is the reference's 8-GPU
    # config (8192 envs / GPU), C3 the Subleq config, and one C5 point (Subleq 65 536 envs x 128 simulations)
    extra = None
    if not args.no_extra and args.workload == "c2":
        del flush
        torch.cuda.empty_cache()
        extra = {"c4": extra_measure(args, "c4", dev, world, rank, steps=4)}
        if world == 1:
            extra["c3"] = extra_measure(args, "c3", dev, world, rank, steps=4)
            extra["c5_point"] = extra_measure(args, "c3", dev, world, rank, steps=2, B_override=65536, n_override=128)
    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    cpu = cpu_baseline(kind, kw, n, gamma) if world == 1 and not args.no_cpu_baseline else None
    n_full = (args.steps + args.param_refresh - 1) // args.param_refresh  # steps that rebuilt the parameter-derived tables
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": workload_config(desc, B, n),
            "notes": {"mlp_mode": "exact_fp32" if args.mlp_mode == 0 else "tensor", "cuda_graph": not args.no_graph, "fused_root": not args.no_fused_root,
                      "streams": args.streams, "root_noise": "drawn inside the search (counter-based stream)",
                      "param_refresh": f"weight images / novelty / seq-halving tables rebuilt every {args.param_refresh} steps (selfplay_steps of the reference, config.py:37,105), reused in between",
                      "multi_gpu": (f"envs sharded per rank, params broadcast once, per-step trajectory records packed into a [{args.param_refresh},B,4] scan "
                                    "buffer and all-gathered once per scan on a side stream (main.py:383-385)") if world > 1 else "single GPU"},
            "simulations_per_s": value * n, "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / args.steps,
                    "copies": ("1 pinned H2D copy of the state arena, 2 D2H copies (state arena, search-output arena) per step" if (not args.no_graph and not args.no_fused_root)
                               else "one copy per state field / result tensor")},
            "gpu_launches": n_full * runner.launches_per_step + (args.steps - n_full) * runner.launches_per_step_reuse + args.steps, "roofline": roofline,
            "cpu_baseline": cpu, "extra": extra}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_LIMIT_BYTES = 64 * 10**6


def dump_outputs(out_dir, arrays, prefix=""):
    """Write each [B, ...] tensor of `arrays` to out_dir/<prefix><name>.npy, so that the results of two builds can be compared
    array for array.  Integers of up to 16 bits and floats of up to 32 go out as float32, wider ones as float64: both exact.  Above
    DUMP_LIMIT_BYTES in all, every array keeps the same fixed, seeded sample of rows (envs)."""
    host = {}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        host[name] = a.astype(np.float32 if a.itemsize <= (4 if a.dtype.kind == "f" else 2) else np.float64)
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        B = len(next(iter(host.values())))
        rows = np.sort(np.random.default_rng(0).choice(B, B * DUMP_LIMIT_BYTES // total, replace=False))
        host = {name: a[rows] for name, a in host.items()}
        print(f"bench.py: --dump-outputs keeps {len(rows)} of {B} rows (seed 0) of every array", file=sys.stderr)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), np.ascontiguousarray(a))


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line goes to the process's real stdout; everything else (NCCL banners, warnings) was moved to stderr."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # C-level stdout (e.g. "NCCL version ...") -> stderr
    sys.stdout = os.fdopen(os.dup(2), "w")
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--mlp-mode", type=int, default=1, help="0 = fp32 FMA chains (bit-exact contract), 1 = tcgen05 3xTF32 (default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the short C3 / C4 / C5-point measurements of the `extra` block")
    ap.add_argument("--streams", type=int, default=0,
                    help="EAZ_FLAG_STREAMS: search this many sub-batches concurrently on auxiliary streams (0 = 3, or 1 for DeepSea batches beyond one wave of clusters: C4 then runs as ONE persistent launch over two waves)")
    ap.add_argument("--envs-per-gpu", type=int, default=0, help="override the workload's batch (exploration, not a BASELINE config)")
    ap.add_argument("--sims", type=int, default=0, help="override the workload's simulation count")
    ap.add_argument("--param-refresh", type=int, default=8,
                    help="rebuild the parameter-derived tables every N steps (the reference runs selfplay_steps=8 DeepSea steps per model, config.py:105)")
    ap.add_argument("--no-fused-root", action="store_true", help="evaluate the root network with a separate eaz_mlp_forward_states call")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly instead of replaying a CUDA graph of the step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (states, search outputs, trajectory record) "
                         "to DIR/<name>.npy as float32 / float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 implementation")
    kind, kw, B, n, gamma, desc = WORKLOADS[args.workload]
    if args.envs_per_gpu or args.sims:  # exploration knobs (not the BASELINE configs): the description says so
        B, n = args.envs_per_gpu or B, args.sims or n
        desc += f" [overridden: {B} envs/GPU, {n} simulations]"
    if args.streams <= 0:
        args.streams = 1 if (kind == "deepsea" and B > 4096) else 3  # (C4: one persistent launch, two waves of clusters: psearch.cuh)
    if args.impl == "reference":
        run_reference(args, kind, kw, B, n, gamma, desc)
    else:
        run_b200(args, kind, kw, B, n, gamma, desc)


if __name__ == "__main__":
    main()
