#!/usr/bin/env python
"""bench.py - headline benchmark of the W4A16 QuantLinear hot path (driver contract).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME]

Default workload = BASELINE.json configs[1]: Llama-2-7B int4 g=128 decode, bs=1.  One "step" = one decode
token = the 224 QuantLinear forwards of the model (32 blocks x {q,k,v,o 4096->4096; gate,up 4096->11008;
down 11008->4096}) at M=1, chained through their real data dependencies, on synthetic random-packed
weights (SURVEY.md 8d).  The 3.5 GB weight set is far larger than the 126 MB L2, so every step streams the
weights from HBM.  N>1: one replica per GPU (the 7B model fits one GPU; north_star shards only models that
overflow), no data-path collective, weak scaling; value = tokens/s summed over ranks, time = max over ranks.

    value    device-resident: the token's launches replayed as a CUDA graph, timed with CUDA events.
    e2e      the same token through the public module API with HOST activations: every step copies x from
             pinned host memory to the device, runs the 224 forwards, and copies y back.
    roofline HBM: algorithmic bytes per launch (SURVEY 8d formula) / average launch duration vs the
             measured copy bandwidth in MEASURED_PEAKS.json.
    cpu_baseline  the reference's CPU path (oracle/ref_port_torch.py, a restatement of the python fallback
             qlinear_cuda_old.py:291-355) timed on this box's host cores on one decoder block.

--impl reference times that CPU path alone (rank 0 only) and prints the same JSON shape.

--dump-outputs DIR writes what the timed path returned in its last timed step as DIR/<name>.npy (float32, rank 0): y (the
device-resident step) and y_e2e (the end-to-end step) of the decode workloads, y of the TP workload, one array per layer
of the block the CPU arm times.  All inputs are seeded, so two builds run with the same arguments can be compared
output for output.
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
import torch  # noqa: E402

WORKLOADS = {
    # name: (hidden, intermediate, n_blocks, M, description)
    "llama2-7b-decode-bs1": (4096, 11008, 32, 1, "Llama-2-7B int4 g=128 decode bs=1 (224 QuantLinear forwards/token, M=1)"),
    "llama2-7b-prefill-bs8x2048": (4096, 11008, 32, 16384, "Llama-2-7B int4 g=128 prefill bs=8 seq=2048 (M=16384)"),
}
# tensor-parallel workload (BASELINE.json configs[3]): the ranks of ONE job shard every layer (strong scaling)
TP_WORKLOADS = {
    # name: (hidden, intermediate, kv_dim, n_blocks, M, description)
    "llama2-70b-decode-tp": (8192, 28672, 1024, 80, 1,
                             "Llama-2-70B int4 g=128 decode bs=1, QuantLinear column/row-sharded over the ranks (autogptq_b200.sharding), "
                             "act-order (desc_act) on the column-parallel layers, one all-reduce per row-parallel layer (2 per block) "
                             "fused into the persistent chain kernel over NVLink peer memory"),
}
GROUP = 128


def alg_bytes(M, K, N, g):
    G = -(-K // g)
    return K * N // 2 + G * N * 2 + G * N // 2 + 2 * M * K + 2 * M * N


def block_shapes(hidden, inter):
    # (name, K, N) in execution order; q,k,v read the block input, o reads q's output, gate/up read o's, down reads gate's
    return [("q", hidden, hidden), ("k", hidden, hidden), ("v", hidden, hidden), ("o", hidden, hidden),
            ("gate", hidden, inter), ("up", hidden, inter), ("down", inter, hidden)]


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(outdir, arrays):
    """Save each tensor as float32 outdir/<name>.npy.  One that is larger than its share of DUMP_LIMIT_BYTES keeps a
    fixed, seeded sample of its rows (the same rows on every run of the same workload)."""
    os.makedirs(outdir, exist_ok=True)
    share = DUMP_LIMIT_BYTES // max(1, len(arrays))
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        a = a.reshape(-1, a.shape[-1])
        max_rows = max(1, (share - 4096) // (4 * a.shape[1]))
        if a.shape[0] > max_rows:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], max_rows, replace=False))]
        np.save(os.path.join(outdir, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.thread = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
        except Exception:
            self.proc = None
            return
        def reader():
            for line in self.proc.stdout:
                self.rows.append((time.time(), [c.strip() for c in line.split(",")]))
        self.thread = threading.Thread(target=reader, daemon=True)
        self.thread.start()

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15] or [r for (_, r) in self.rows]
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------- synthetic model
def synth_layer(K, N, g, dev, gen, gain=1.0):
    """Random-packed layer (SURVEY 8d): uniform nibbles, zero nibbles in [0,14]; scales sized for unit gain so
    the 96-deep chain of a token stays O(1) in fp16."""
    from autogptq_b200 import QuantLinear

    lin = QuantLinear(4, g, K, N, False)
    G = -(-K // g)
    lin.qweight = torch.randint(-2**31, 2**31 - 1, (K // 8, N), dtype=torch.int32, device=dev, generator=gen)
    zn = torch.randint(0, 15, (G, N), dtype=torch.int32, device=dev, generator=gen)
    qz = torch.zeros((G, N // 8), dtype=torch.int32, device=dev)
    for j in range(8):
        qz |= zn[:, j::8] << (4 * j)
    lin.qzeros = qz
    # unit gain: rms(q - z) ~ 6.3.  Random SIGN per (group, column): uniform nibbles have mean(q - z) = -0.5, which
    # with all-positive scales adds a coherent offset that grows ~5x per layer and overflows fp16 in a 96-deep
    # chain; signed scales are numerically legal for the kernels and leave traffic / timing unchanged.
    unit = gain * 0.9 / (6.34 * (K ** 0.5))       # x sqrt(E[(0.5+U)^2]) = 1.04 -> per-layer gain ~0.94
    sign = (torch.randint(0, 2, (G, N), device=dev, generator=gen).float() * 2 - 1)
    lin.scales = ((torch.rand((G, N), device=dev, generator=gen) + 0.5) * unit * sign).half()
    lin.g_idx = (torch.arange(K, dtype=torch.int32, device=dev) // g)
    lin = lin.to(dev)
    lin.post_init()
    return lin


def build_model(hidden, inter, n_blocks, dev, seed):
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    return [{name: synth_layer(K, N, GROUP, dev, gen) for (name, K, N) in block_shapes(hidden, inter)}
            for _ in range(n_blocks)]


class Branches:
    """Side streams for the layers of a block that do not depend on each other (k, v next to q; up next to gate).
    Under CUDA-graph capture they become parallel branches, so the three 4096x4096 projections stream together
    instead of paying three serialized launch latencies.  Plain PyTorch stream/event API around the module calls."""

    def __init__(self, device, mode="group"):
        self.mode = mode
        enabled = mode == "branches"
        self.enabled = enabled
        self.side = [torch.cuda.Stream(device=device) for _ in range(2)] if enabled else []

    def run(self, main_fn, side_fns):
        """main_fn() on the current stream, side_fns concurrently; returns main_fn's result after joining."""
        if not self.enabled:
            out = main_fn()
            for f in side_fns:
                f()
            return out
        cur = torch.cuda.current_stream()
        fork = torch.cuda.Event()
        fork.record(cur)
        joins = []
        for st, f in zip(self.side, side_fns):
            st.wait_event(fork)
            with torch.cuda.stream(st):
                f()
                ev = torch.cuda.Event()
                ev.record(st)
                joins.append(ev)
        out = main_fn()
        for ev in joins:
            cur.wait_event(ev)
        return out


def build_chain(model, M, dev):
    """The same token as token_forward (same layers, same dependencies) as ONE persistent launch: autogptq_b200.chain."""
    from autogptq_b200.chain import DecodeChain

    ch = DecodeChain(M=M, dtype=torch.float16, device=dev)
    x = ch.input(model[0]["q"].infeatures)
    t = x
    for blk in model:
        q, _, _ = ch.stage([blk["q"], blk["k"], blk["v"]], t)
        (o,) = ch.stage([blk["o"]], q)
        gate, _ = ch.stage([blk["gate"], blk["up"]], o)
        (t,) = ch.stage([blk["down"]], gate)
    ch.build()
    return ch, x, t


def token_forward(model, x, br):
    """The QuantLinear calls of one forward pass with their true dependencies.  Sibling layers (same input) are
    issued together: one grouped launch (autogptq_b200.forward_group), or parallel graph branches, or serially."""
    from autogptq_b200 import forward_group

    for blk in model:
        if br.mode == "group":
            q, _, _ = forward_group([blk["q"], blk["k"], blk["v"]], x)
            o = blk["o"](q)
            gate, _ = forward_group([blk["gate"], blk["up"]], o)
        else:
            q = br.run(lambda: blk["q"](x), [lambda: blk["k"](x), lambda: blk["v"](x)])
            o = blk["o"](q)
            gate = br.run(lambda: blk["gate"](o), [lambda: blk["up"](o)])
        x = blk["down"](gate)
    return x


# ------------------------------------------------------------------------------------------- CPU baseline (oracle port)
def usable_cpus():
    """Host threads the CPU arm may use: the affinity mask, capped by a cgroup CPU quota (os.cpu_count() reports the
    machine, not the container - oversubscribing 128 torch threads onto a smaller quota made the arm ~10x slower)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                quota, period = txt[0], float(txt[1])
                if quota != "max":
                    n = min(n, max(1, int(float(quota) / period)))
            else:
                quota = float(txt[0])
                period = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    n = min(n, max(1, int(quota / period)))
            break
        except Exception:
            continue
    return max(1, n)


def cpu_block_time(hidden, inter, M, reps, threads, outputs=None):
    """Reference CPU path on one decoder block (7 QuantLinear forwards).  Returns (seconds per block, sample text);
    `outputs`, when given, receives the layers' outputs of the last rep by layer name."""
    from oracle.ref_port_torch import python_fallback_forward

    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(0)
    layers = []
    for (_, K, N) in block_shapes(hidden, inter):
        G = K // GROUP
        layers.append((torch.randint(-2**31, 2**31 - 1, (K // 8, N), dtype=torch.int32, generator=g),
                       torch.randint(0, 2**31 - 1, (G, N // 8), dtype=torch.int32, generator=g),
                       torch.rand((G, N), generator=g) * 0.01 + 0.001, K))
    xs = {K: torch.randn(M, K, generator=g) for K in (hidden, inter)}

    def run_block():
        for (name, _, _), (qw, qz, sc, K) in zip(block_shapes(hidden, inter), layers):
            y = python_fallback_forward(xs[K], qw, qz, sc, GROUP)
            if outputs is not None:
                outputs[name] = y

    run_block()
    t0 = time.perf_counter()
    for _ in range(reps):
        run_block()
    dt = (time.perf_counter() - t0) / reps
    return dt, f"1 of 32 decoder blocks (7 QuantLinear forwards, M={M}), python-fallback port fp32, {reps} reps"


def cpu_block_time_c(hidden, inter, M, reps):
    """Same block on the C / OpenMP restatement (oracle/w4a16_oracle.c: raw nibbles x activations with the zero point
    through sum(x), the formulation of the reference's qigen CPU kernel, qlinear_qigen.py:263,320-338).  None when the
    library has not been built."""
    try:
        from oracle import c_oracle
        if not c_oracle.available():
            return None
        rng = np.random.default_rng(0)
        layers = []
        for (_, K, N) in block_shapes(hidden, inter):
            G = K // GROUP
            layers.append((rng.integers(-2**31, 2**31 - 1, size=(K // 8, N), dtype=np.int64).astype(np.int32),
                           rng.integers(0, 2**31 - 1, size=(G, N // 8), dtype=np.int64).astype(np.int32),
                           (rng.random((G, N), dtype=np.float32) * 0.01 + 0.001), K))
        xs = {K: rng.standard_normal((M, K)).astype(np.float32) for K in (hidden, inter)}

        def run_block():
            for (qw, qz, sc, K) in layers:
                c_oracle.forward(xs[K], qw, qz, sc, None, GROUP, None)

        run_block()
        t0 = time.perf_counter()
        for _ in range(reps):
            run_block()
        return (time.perf_counter() - t0) / reps, c_oracle.threads()
    except Exception:
        return None


def cpu_block_time_qigen(hidden, inter, M, reps, outputs=None):
    """The reference's own compiled CPU kernel (qigen, qlinear_qigen.py:257-338) on one decoder block, through
    oracle/qigen_ref.py around oracle/_ref/cQIGen (built from /root/reference by oracle/build_qigen.py; OpenMP thread count
    baked in at generation time).  None when the library is not there.  `outputs` as in cpu_block_time."""
    try:
        from oracle import qigen_ref
        if not qigen_ref.available():
            return None
        rng = np.random.default_rng(0)
        layers = []
        for (_, K, N) in block_shapes(hidden, inter):
            G = K // GROUP
            zn = rng.integers(0, 15, size=(G, N), dtype=np.int64).astype(np.uint32)
            qz = np.zeros((G, N // 8), dtype=np.uint32)
            for j in range(8):
                qz |= zn[:, j::8] << np.uint32(4 * j)
            layers.append(qigen_ref.QigenLinear(
                rng.integers(-2**31, 2**31 - 1, size=(K // 8, N), dtype=np.int64).astype(np.int32), qz.view(np.int32),
                (rng.random((G, N), dtype=np.float32) * 0.01 + 0.001), GROUP))
        xs = {K: torch.from_numpy(rng.standard_normal((M, K)).astype(np.float32)) for K in (hidden, inter)}

        def run_block():
            for (name, _, _), lin in zip(block_shapes(hidden, inter), layers):
                y = lin.forward(xs[lin.K])
                if outputs is not None:
                    outputs[name] = y

        run_block()
        t0 = time.perf_counter()
        for _ in range(reps):
            run_block()
        return (time.perf_counter() - t0) / reps, qigen_ref.threads()
    except Exception:
        return None


def shared_config(workload, desc, n_calls):
    """The `config` object both arms print (the driver compares them): what is measured, nothing about how."""
    return {"workload": workload, "desc": desc, "group_size": GROUP, "layers_per_step": n_calls,
            "l2": "weight working set 3.5 GB >> 126 MB L2 (no flush needed)"}


def cpu_rows_for(M):
    # bound the CPU sample for the prefill workload: the python path is O(M) in the matmul only
    return min(M, 64)


# ------------------------------------------------------------------------------------------- main arms
def run_reference(args, rank, world):
    if args.workload in TP_WORKLOADS:
        h, i, _, nb, m, d = TP_WORKLOADS[args.workload]
        hidden, inter, n_blocks, M, desc = h, i, nb, m, d
    else:
        hidden, inter, n_blocks, M, desc = WORKLOADS[args.workload]
    if rank != 0:
        return
    threads = usable_cpus()
    Mc = cpu_rows_for(M)
    kind = "port"
    outputs = {}
    probe = cpu_block_time_qigen(hidden, inter, Mc, 1)
    if probe is not None:
        # the reference's own compiled CPU kernel (qigen) - the strongest CPU implementation the reference has for this path
        kind = "reference"
        threads = probe[1]
        times = []
        for _ in range(max(1, args.warmup)):
            cpu_block_time_qigen(hidden, inter, Mc, 1)
        for i in range(args.steps):
            times.append(cpu_block_time_qigen(hidden, inter, Mc, 3, outputs if i == args.steps - 1 else None)[0])
        sample = (f"1 of {n_blocks} decoder blocks (7 QuantLinear forwards, M={Mc}), the reference's qigen kernel "
                  f"(oracle/_ref/cQIGen, forward_gs4, {threads} OpenMP threads baked in), 3 reps per step")
    else:
        for _ in range(max(1, args.warmup)):
            cpu_block_time(hidden, inter, Mc, 1, threads)
        times = []
        sample = ""
        for i in range(args.steps):
            dt, sample = cpu_block_time(hidden, inter, Mc, 1, threads, outputs if i == args.steps - 1 else None)
            times.append(dt)
    t_step = float(np.mean(times))                       # one block
    tokens_per_step = (Mc / n_blocks)                    # a block is 1/32 of a token's linears
    value = tokens_per_step / t_step
    line = {
        "impl": "reference", "metric": "llama2_7b_w4a16_linear_tokens_per_s", "value": value, "unit": "tokens/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_step * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(args.workload, desc, n_blocks * 7),
        "run": {"step": "one decoder block on host cores, scaled to a token (x 1/32)"},
        "cpu_baseline": {"value": value, "unit": "tokens/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)


def run_b200(args, rank, world, local_rank):
    import torch.distributed as dist

    hidden, inter, n_blocks, M, desc = WORKLOADS[args.workload]
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    torch.manual_seed(4321 + rank)                       # activations: the same inputs on every run
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from autogptq_b200 import _lib
    _lib.load()

    model = build_model(hidden, inter, n_blocks, dev, seed=1234 + rank)
    n_calls = n_blocks * 7
    bytes_per_step = n_blocks * sum(alg_bytes(M, K, N, GROUP) for (_, K, N) in block_shapes(hidden, inter))
    flops_per_step = n_blocks * sum(2.0 * M * K * N for (_, K, N) in block_shapes(hidden, inter))

    x_dev = torch.randn(M, hidden, dtype=torch.float16, device=dev)
    x_host = torch.randn(M, hidden, dtype=torch.float16).pin_memory()
    y_host = torch.empty(M, hidden, dtype=torch.float16).pin_memory()
    x_in = torch.empty(M, hidden, dtype=torch.float16, device=dev)

    stream = torch.cuda.Stream(device=dev)
    use_chain = args.siblings == "chain" and M <= 2
    if args.siblings == "chain" and not use_chain:
        args.siblings = "group"
    chain_info = None
    with torch.cuda.stream(stream):
        br = Branches(dev, mode="group" if use_chain else args.siblings)
        y = token_forward(model, x_dev, br)              # eager once: lazy init + finite check
        torch.cuda.synchronize(dev)
        assert torch.isfinite(y.float()).all(), "non-finite activations in the synthetic chain"
        chain_error = None
        if use_chain:
            try:
                chain, ch_x, ch_y = build_chain(model, M, dev)
                chain_info = chain.info()
            except (NotImplementedError, autogptq_b200._lib.B200KernelError) as exc:
                # creation refused (no cooperative launch, not enough shared memory, ...): the per-layer launches are
                # still this repo's kernels; the line says which path ran
                chain_error = str(exc)[:300]
                use_chain = False
                args.siblings = "group"
        if use_chain:
            # the whole token = one persistent cooperative launch (csrc/chain.cuh); checked against the per-layer launches
            ch_x.copy_(x_dev)
            chain.run()
            torch.cuda.synchronize(dev)
            err = (ch_y.float() - y.float()).abs().max().item()
            ref = y.float().abs().max().item()
            # 128 dependent layers, each within 1e-3 of the oracle (tests/test_gpu_7_chain.py), amplify rounding differences
            assert torch.isfinite(ch_y.float()).all() and err <= 0.2 * ref + 1e-3, f"chain vs per-layer launches: {err} (max |y| {ref})"
            chain_info["max_abs_diff_vs_per_layer_launches_after_128_stages"] = err
            chain_info["max_abs_y"] = ref
            dbg = int(os.environ.get("AGB200_CHAIN_DEBUG", "0"))
            g_dev = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_dev, stream=stream):
                chain.run(dbg)
            g_e2e = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_e2e, stream=stream):
                ch_x.copy_(x_host, non_blocking=True)
                chain.run(dbg)
                y_host.copy_(ch_y, non_blocking=True)
        else:
            # device-resident graph
            g_dev = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_dev, stream=stream):
                y_dev = token_forward(model, x_dev, br)
            # end-to-end graph: pinned host -> device, 224 forwards through the module API, device -> pinned host
            g_e2e = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_e2e, stream=stream):
                x_in.copy_(x_host, non_blocking=True)
                y_e2e = token_forward(model, x_in, br)
                y_host.copy_(y_e2e, non_blocking=True)

        def barrier():
            torch.cuda.synchronize(dev)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize(dev)

        def timed(graph, steps, per_step_host=None):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record(stream)
            for i in range(steps):
                if per_step_host is not None:
                    per_step_host(i)
                graph.replay()
                if per_step_host is not None:
                    stream.synchronize()              # the step's result is read on the host
            e1.record(stream)
            e1.synchronize()
            barrier()
            ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            return float(ms.item())

        for _ in range(max(3, args.warmup)):
            g_dev.replay()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
            time.sleep(0.25)
        t0 = time.time()
        ms_dev = timed(g_dev, args.steps)
        t1 = time.time()
        clocks = sampler.stop(t0, t1) if rank == 0 else None
        outputs = {"y": (ch_y if use_chain else y_dev).clone()}      # the e2e graph below overwrites ch_y

        feed = [torch.randn(M, hidden, dtype=torch.float16) for _ in range(4)]
        checksum = [0.0]

        def host_step(i):
            x_host.copy_(feed[i % 4])                 # new input every step
            if i > 0:
                checksum[0] += float(y_host[0, 0])    # device -> host read of the previous result

        for i in range(max(3, args.warmup)):
            host_step(i); g_e2e.replay(); stream.synchronize()
        ms_e2e = timed(g_e2e, args.steps, host_step)
        outputs["y_e2e"] = y_host.clone()

    tokens_per_step = M * world                          # weak scaling: every rank decodes its own stream
    value = tokens_per_step / (ms_dev / args.steps / 1e3)
    e2e_value = tokens_per_step / (ms_e2e / args.steps / 1e3)
    peaks, peak_kind = load_peaks()
    step_s = ms_dev / args.steps / 1e3
    n_launches = 1 if use_chain else (n_blocks * 4 if (args.siblings == "group" and M <= 4) else n_calls)     # kernel launches per step
    if M <= 64:
        achieved = bytes_per_step / step_s / 1e9
        roof = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": None, "peak_kind": peak_kind,
                "kernel": "w4a16_chain_kernel" if use_chain else "w4a16_gemv_kernel", "algorithmic_bytes_per_launch": bytes_per_step / n_launches,
                "avg_launch_us": step_s / n_launches * 1e6, "launches_per_step": n_launches}
    else:
        achieved = flops_per_step / step_s / 1e12
        pk = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
        roof = {"bound": "tensor", "achieved": achieved, "peak": pk, "unit": "TFLOP/s", "frac": achieved / pk,
                "traffic": None, "peak_kind": peak_kind + " (sustained)", "kernel": "w4a16_gemm_kernel",
                "flops_per_launch": flops_per_step / n_launches, "avg_launch_us": step_s / n_launches * 1e6,
                "launches_per_step": n_launches}
    # ncu-derived DRAM traffic per launch, when a profile summary has been committed
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        roof["traffic"] = prof.get(args.workload if use_chain else args.workload + "-per-layer-launch", prof.get(args.workload))
    except Exception:
        pass

    # what a drop-in user without CUDA graphs sees: the same token through eager module calls (host-bound: ~128 launches
    # of python + ctypes), and the prefill configuration (BASELINE configs[2]) on the same weights - sub-records, N = 1 only
    eager_rec, prefill_rec = None, None
    if world == 1 and M == 1:
        with torch.cuda.stream(stream):
            brg = Branches(dev, mode="group")
            for _ in range(2):
                token_forward(model, x_dev, brg)
            torch.cuda.synchronize(dev)
            t_e = time.perf_counter()
            n_e = 5
            for _ in range(n_e):
                token_forward(model, x_dev, brg)
            torch.cuda.synchronize(dev)
            dt_e = (time.perf_counter() - t_e) / n_e
            eager_rec = {"value": 1.0 / dt_e, "unit": "tokens/s", "ms_per_step": dt_e * 1e3,
                         "what": "eager QuantLinear / forward_group calls, no CUDA graph (host-bound), wall clock"}
            try:
                Mp = 16384
                xp = torch.randn(Mp, hidden, dtype=torch.float16, device=dev)
                token_forward(model, xp, Branches(dev, mode="serial"))        # builds the tensor-core copies
                torch.cuda.synchronize(dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                n_p = 2
                for _ in range(n_p):
                    token_forward(model, xp, Branches(dev, mode="serial"))
                e1.record(stream)
                e1.synchronize()
                ms_p = e0.elapsed_time(e1) / n_p
                fl = n_blocks * sum(2.0 * Mp * K * N for (_, K, N) in block_shapes(hidden, inter))
                pk = load_peaks()[0]
                prefill_rec = {"workload": "llama2-7b-prefill-bs8x2048", "M": Mp, "ms_per_step": ms_p, "tflops": fl / ms_p / 1e9,
                               "tokens_per_s": Mp / (ms_p / 1e3), "frac_of_sustained_bf16_peak": fl / ms_p / 1e9 / pk.get("bf16_tflops_sustained", pk["bf16_tflops"]),
                               "kernel": "w4a16_gemm_kernel (tcgen05 / TMEM / TMA)", "steps": n_p}
                del xp
            except Exception as e:
                prefill_rec = {"error": f"{type(e).__name__}: {e}"[:200]}

    # multi-GPU runs also measure the path the ranks SHARE (BASELINE configs[3]): Llama-2-70B decode, tensor-parallel over
    # all ranks of this job - the replica numbers above say nothing about an exchange step
    tp_rec = None
    if world > 1 and M == 1 and os.environ.get("AGB200_BENCH_TP", "1") == "1":
        try:
            tp_rec = tp_chain_record(args, rank, world, local_rank)
        except Exception as e:      # the headline must survive a failure of the extra record
            tp_rec = {"error": f"{type(e).__name__}: {e}"[:300]} if rank == 0 else None

    if rank == 0:
        threads = usable_cpus()
        dt_blk, sample = cpu_block_time(hidden, inter, cpu_rows_for(M), 3, threads)
        cpu_val = (cpu_rows_for(M) / n_blocks) / dt_blk
        line = {
            "metric": "llama2_7b_w4a16_linear_tokens_per_s", "value": value, "unit": "tokens/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_dev / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 (fp32 accumulate)",
            "data": "synthetic",
            "config": shared_config(args.workload, desc, n_calls),
            "run": {"parallelism": f"replica x{world}",
                    "sibling_layers": {"chain": "whole token in ONE persistent cooperative launch (autogptq_b200.chain.DecodeChain): weights streamed by TMA across layer boundaries, 128 dependent stages (q|k|v, o, gate|up, down per block) synchronised by tagged data words", "group": "q|k|v and gate|up each in one grouped launch (forward_group)", "branches": "k,v | up on side streams (graph branches)", "serial": "serial"}[args.siblings],
                    "next_layer_l2_prefetch": bool(args.prefetch), "timing": "CUDA graph replay, CUDA events, max over ranks"},
            "e2e": {"value": e2e_value, "unit": "tokens/s", "h2d_bytes_per_step": M * hidden * 2,
                    "d2h_bytes_per_step": M * hidden * 2, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": n_launches * args.steps,
            "chain": chain_info if chain_error is None else {"refused": chain_error, "fallback": "per-layer grouped launches"},
            "tp70b": tp_rec,
            "eager": eager_rec,
            "prefill": prefill_rec,
            "roofline": roof,
            "cpu_baseline": {"value": cpu_val, "unit": "tokens/s", "cores": threads, "kind": "port", "sample": sample},
            "clocks": clocks,
        }
        q_arm = cpu_block_time_qigen(hidden, inter, cpu_rows_for(M), 3)
        if q_arm is not None:       # the reference's compiled CPU kernel becomes THE cpu baseline; the python fallback stays beside it
            line["cpu_baseline_python"] = line["cpu_baseline"]
            line["cpu_baseline"] = {"value": (cpu_rows_for(M) / n_blocks) / q_arm[0], "unit": "tokens/s", "cores": q_arm[1],
                                    "kind": "reference",
                                    "sample": "1 of 32 decoder blocks (7 QuantLinear forwards), the reference's qigen kernel "
                                              "(oracle/_ref/cQIGen forward_gs4, OpenMP threads baked in at generation), 3 reps"}
        c_arm = cpu_block_time_c(hidden, inter, cpu_rows_for(M), 3)
        if c_arm is not None:       # extra information: a compiled CPU arm next to the reference's python path
            line["cpu_baseline_c"] = {"value": (cpu_rows_for(M) / n_blocks) / c_arm[0], "unit": "tokens/s", "cores": c_arm[1],
                                      "kind": "port", "sample": "same block, C / OpenMP restatement (qigen-style sum(x) formulation), 3 reps"}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def build_tp_blocks(hidden, inter, kv, n_blocks, rank, world, dev, log=None):
    """Llama-2-70B-shaped synthetic blocks, generated unsharded (same seed on every rank) and cut for this rank by
    autogptq_b200.sharding (column-parallel q, k, v, gate, up with act-order g_idx shared by siblings; row-parallel o, down
    with sequential groups - down's act-order permutation is the one that folds into the column order of gate|up offline,
    o_proj's would need the attention heads gathered first and is left sequential).  One full layer lives at a time."""
    from autogptq_b200.sharding import shard_column_parallel, shard_row_parallel, shard_to_module

    gen = torch.Generator(device=dev)
    gen.manual_seed(4321)
    column = ("q", "k", "v", "gate", "up")
    shapes = [("q", hidden, hidden), ("k", hidden, kv), ("v", hidden, kv), ("o", hidden, hidden),
              ("gate", hidden, inter), ("up", hidden, inter), ("down", inter, hidden)]
    blocks = []
    t0 = time.time()
    for bi in range(n_blocks):
        if log and bi % 20 == 0:
            log(f"# building block {bi}/{n_blocks} ({time.time() - t0:.1f} s)")
        blk = {}
        perm_by_k = {}
        for name, K, N in shapes:
            full = synth_layer(K, N, GROUP, dev, gen, gain=1.0)
            g_idx = full.g_idx
            if name in column:                        # GPTQ act-order g_idx (quantization/gptq.py:177-181), shared by sibling layers
                if name in ("q", "gate"):
                    perm_by_k[K] = torch.randperm(K, device=dev, generator=gen)
                g_idx = (torch.arange(K, device=dev, dtype=torch.int32) // GROUP)[torch.argsort(perm_by_k[K])].contiguous()
            fn = shard_column_parallel if name in column else shard_row_parallel
            shard = fn(full.qweight, full.qzeros, full.scales, g_idx, None, group_size=GROUP, rank=rank, world=world)
            blk[name] = shard_to_module(shard, dev)
            blk[name].post_init()
            del full
        blocks.append(blk)
    return blocks


def tp_chain_record(args, rank, world, local_rank, n_blocks=None, steps=None, outputs=None):
    """Llama-2-70B decode, QuantLinears column/row-sharded over `world` ranks (BASELINE configs[3]): one persistent
    chain launch per rank and token, the row-parallel all-reduces fused into it (tagged words over NVLink peer memory,
    autogptq_b200.tp.TPDecodeChain), replayed as a CUDA graph.  Returns the record (rank 0) or None; `outputs`, when
    given, receives the output of the last timed step as "y"."""
    import torch.distributed as dist
    from autogptq_b200.tp import TPDecodeChain

    hidden, inter, kv, nb, M, desc = TP_WORKLOADS["llama2-70b-decode-tp"]
    n_blocks = n_blocks or nb
    steps = steps or max(5, min(args.steps, 20))
    dev = torch.device("cuda", local_rank)
    log = (lambda m: print(m, file=sys.stderr, flush=True)) if rank == 0 else None
    blocks = build_tp_blocks(hidden, inter, kv, n_blocks, rank, world, dev, log)
    shapes = [(hidden, hidden // world), (hidden, kv // world), (hidden, kv // world), (hidden // world, hidden),
              (hidden, inter // world), (hidden, inter // world), (inter // world, hidden)]
    bytes_per_rank_step = n_blocks * sum(alg_bytes(M, K, N, GROUP) for (K, N) in shapes)
    tp = TPDecodeChain(blocks, group=None, M=M, device=dev)
    x = torch.randn(M, hidden, dtype=torch.float16, device=dev)
    stream = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(stream):
        tp.x.copy_(x)
        tp.run()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        y = tp.output()
        assert torch.isfinite(y.float()).all(), "non-finite activations in the TP chain"
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            tp.run()
        for _ in range(3):
            g.replay()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            g.replay()
        e1.record(stream)
        e1.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        if outputs is not None:
            outputs["y"] = tp.output().clone()
    ms = float(ms.item())
    info = tp.chain.info()
    del tp, blocks
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    peaks, peak_kind = load_peaks()
    step_s = ms / steps / 1e3
    achieved = bytes_per_rank_step / step_s / 1e9
    return {
        "metric": "llama2_70b_w4a16_linear_tokens_per_s", "value": M / step_s, "unit": "tokens/s", "n_gpus": world, "steps": steps,
        "ms_per_step": ms / steps, "scaling": "strong", "parallelism": f"tp{world}", "blocks": n_blocks,
        "all_reduces_per_step": 2 * n_blocks if world > 1 else 0, "all_reduce_bytes": M * hidden * 2, "cuda_graph": True,
        "collective": "one-shot all-reduce inside the chain kernel: every rank stores its partial tile as tagged 8-byte words "
                      "into every rank's buffer over NVLink peer memory (cudaIpc), the consuming stage sums the parts",
        "act_order": "q, k, v, gate, up (gather of x in the kernel); down folded offline; o sequential",
        "per_rank_hbm_gbs": achieved, "per_rank_roofline_frac": achieved / peaks["hbm_gbs"], "chain": info,
    }


def run_tp(args, rank, world, local_rank):
    """--workload llama2-70b-decode-tp: the TP chain alone (strong scaling over the ranks of ONE job)."""
    import torch.distributed as dist

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    torch.manual_seed(4321)                              # the TP input: the same on every rank and run
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    t0 = time.time()
    outputs = {}
    rec = tp_chain_record(args, rank, world, local_rank, steps=args.steps, outputs=outputs)
    t1 = time.time()
    if rank == 0:
        clocks = sampler.stop(t0, t1)
        peaks, peak_kind = load_peaks()
        line = {
            "metric": rec["metric"], "value": rec["value"], "unit": "tokens/s", "n_gpus": world, "steps": rec["steps"],
            "warmup": 3, "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16 (fp32 accumulate)", "data": "synthetic",
            "config": {"workload": args.workload, "desc": TP_WORKLOADS[args.workload][5], "group_size": GROUP,
                       "parallelism": rec["parallelism"], "all_reduces_per_step": rec["all_reduces_per_step"],
                       "all_reduce_bytes": rec["all_reduce_bytes"], "cuda_graph": True, "collective": rec["collective"],
                       "act_order": rec["act_order"], "layers_per_step_per_rank": 7 * rec["blocks"]},
            "gpu_launches": rec["steps"], "chain": rec["chain"],
            "roofline": {"bound": "hbm", "achieved": rec["per_rank_hbm_gbs"], "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": rec["per_rank_roofline_frac"], "traffic": None, "peak_kind": peak_kind,
                         "note": "per-rank algorithmic bytes / step time; the step contains the fused all-reduces"},
            "clocks": clocks,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="llama2-7b-decode-bs1", choices=sorted(WORKLOADS) + sorted(TP_WORKLOADS))
    ap.add_argument("--prefetch", action="store_true", help="switch the learned next-layer L2 prefetch of decode launches on (experiment; measured slower)")
    ap.add_argument("--siblings", default="chain", choices=["chain", "group", "branches", "serial"],
                    help="how the token's layers are issued: chain = the whole token as one persistent launch (decode, M <= 2); otherwise per-layer launches with sibling layers (q|k|v, gate|up) as one grouped launch, parallel graph branches, or serially")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed path returned in its last step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: autogptq_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    if args.prefetch:
        import autogptq_b200
        autogptq_b200.set_next_layer_prefetch(True)
    if args.workload in TP_WORKLOADS:
        run_tp(args, rank, world, local_rank)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
