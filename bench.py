#!/usr/bin/env python
"""bench.py -- images/s of the Salience-DETR encoder forward (salience filter + 6 encoder layers) on B200.

Workload (BASELINE.json configs[1]): salience_detr_resnet50_800_1333, bs=2 per GPU, synthetic COCO-shape inputs
(800x1333 padded to 800x1344 -> levels 100x168, 50x84, 25x42, 13x21; Nv=22323, K=11363), fp32, eval, random-init
weights.  A "step" is one encoder-half forward (salience_transformer.py:106-183 of the reference) over one batch.

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's sm_100a path
  python bench.py --impl reference ...                           # the reference's CPU path (oracle port), rank 0 only
  torchrun --nproc-per-node N bench.py --gpus N ...              # one process per GPU, weak scaling (replicas)
  python bench.py ... --dump-outputs DIR                         # also write the last timed step's memory to DIR/memory.npy

Prints ONE JSON line (rank 0).  value = device-resident throughput (CUDA-graph replay, inputs in HBM); e2e =
same metric through EncoderRunner.run_host with pinned HOST buffers (H2D + forward + D2H inside the timed region);
roofline = the dominant kernel (fused MSDA forward) timed alone with CUDA events; cpu_baseline = the oracle port of
the reference's PyTorch CPU path on this host.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

# ONE JSON line on stdout, whatever the libraries print: NCCL writes its version banner (and NCCL_DEBUG output) to file descriptor 1
# from C, past sys.stdout.  The real stdout is kept aside for the result line and descriptor 1 is pointed at stderr for the rest of
# the process.
_RESULT_FD = None


def _claim_stdout():
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: str):
    sys.stdout.flush()
    os.write(_RESULT_FD if _RESULT_FD is not None else 1, (line + "\n").encode())


WORKLOAD = "resnet50_800_1333_bs2"
METRIC = "images/sec encoder-fwd @ 800x1333 bs=2/GPU"
L2_FLUSH_BYTES = 256 << 20


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index, self.start, self.timed_end = [], None, index, 0, None

    def wait_first(self, seconds=3.0):
        """nvidia-smi takes a while to start: block until its first row (so that a short timed region is not missed)."""
        t0 = time.time()
        while not self.rows and time.time() - t0 < seconds and self.proc is not None:
            time.sleep(0.01)

    def mark(self):
        self.start = len(self.rows)

    def mark_end(self):
        self.timed_end = len(self.rows)

    def since_mark(self):
        return len(self.rows) - self.start

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        rows = self.rows[self.start:]
        sm = [int(r[0]) for r in rows if len(r) >= 6 and r[0].isdigit()]
        mx = [int(r[1]) for r in rows if len(r) >= 6 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in rows)]
        out = {"sm_mhz": int(statistics.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
               "reasons": reasons, "samples": len(sm)}
        if self.timed_end is not None:
            out["samples_in_timed_region"] = max(0, self.timed_end - self.start)
            out["note"] = "100 ms sampling; a timed region shorter than that is followed by identical replays of the step until 3 samples exist"
        return out


def msda_algorithmic_bytes(batch, nv, c, heads, levels, points, nq):
    """SURVEY.md 8(d): C_msda = 4*Nv*C + Nq*(12*M*L*P + 4*C) bytes per image (value in; loc+attn in; out)."""
    return batch * (4 * nv * c + nq * (12 * heads * levels * points + 4 * c))


def msda_layer_bytes(runner):
    plan = runner.plan
    b, nv = plan.mask_flat.shape
    m = runner.model.encoder.layers[0].self_attn
    return [msda_algorithmic_bytes(b, nv, m.embed_dim, m.num_heads, m.num_levels, m.num_points, nq)
            for nq in plan.layer_num_query]


def time_msda_in_situ(pkg, runner, reps=20):
    """Roofline leg: the fused MSDA forward launches timed WHERE THEY RUN -- inside the step.  A second runner of the same
    geometry is captured with a CUDA event recorded right before and right after every sampling launch (external event
    nodes of the graph, on the launching stream); the graph is replayed `reps` times with the L2 flushed before each
    replay (as in the timed region) and the per-launch durations are read back.  -> (median ms per layer, how)."""
    from salience_detr_b200.runner import EncoderRunner
    cabi = pkg.cabi
    cabi.KERNEL_TIMERS = {}
    try:
        inst = EncoderRunner(runner.model, runner.feats, runner.masks, runner.pos, use_graph=runner.graph is not None,
                             use_order=runner.use_order, warmup=1)
        pairs = cabi.KERNEL_TIMERS.get("msda", [])[-len(runner.plan.layer_num_query):]
    finally:
        cabi.KERNEL_TIMERS = None
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=runner.dev)
    per_layer = [[] for _ in pairs]
    for _ in range(reps):
        with torch.cuda.stream(inst.stream):
            flush.zero_()
            if inst.graph is None:  # eager: re-record fresh events every step
                cabi.KERNEL_TIMERS = {}
                try:
                    inst.step()
                    pairs = cabi.KERNEL_TIMERS["msda"]
                finally:
                    cabi.KERNEL_TIMERS = None
            else:
                inst.step()
        torch.cuda.synchronize()
        for i, (a, b) in enumerate(pairs):
            per_layer[i].append(a.elapsed_time(b))
    return [statistics.median(x) for x in per_layer], ("in situ: events around each launch inside the captured step"
                                                       if inst.graph is not None else "in situ: events around each eager launch")


def time_msda_kernels(pkg, runner, reps=20):
    """Same launches replayed ALONE after an L2 flush (cold value slice from HBM; the round-1 definition, kept for
    continuity)."""
    cabi = pkg.cabi
    calls = []
    orig = cabi.msda_fused_forward

    def spy(*a, **k):
        calls.append((a, k))
        return orig(*a, **k)

    cabi.msda_fused_forward = spy
    try:
        with torch.no_grad():
            runner.model.forward_encoder(runner.feats, runner.masks, runner.pos, plan=runner.plan,
                                         use_order=runner.use_order)
    finally:
        cabi.msda_fused_forward = orig
    torch.cuda.synchronize()
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=runner.dev)
    per_layer = [[] for _ in calls]
    for _ in range(reps):
        flush.zero_()  # evict L2: the value slice comes from HBM
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(calls) + 1)]
        evs[0].record()
        for i, (a, k) in enumerate(calls):
            orig(*a, **k)
            evs[i + 1].record()
        torch.cuda.synchronize()
        for i in range(len(calls)):
            per_layer[i].append(evs[i].elapsed_time(evs[i + 1]))
    return [statistics.median(x) for x in per_layer]  # ms


def time_gemm_kernels(pkg, runner, reps=10):
    """Secondary (tensor-bound) leg: every dense projection of one step replayed alone with CUDA events.
    -> (total ms per step, logical flops per step, number of GEMM calls)."""
    gemm = pkg.gemm
    calls = []
    orig = gemm.linear

    def spy(x, w, b=None, *a, **k):
        calls.append((x, w, b, a, k))
        return orig(x, w, b, *a, **k)

    # the fused FFN (linear1 -> ReLU -> linear2 -> +residual -> LayerNorm in one tensor-core kernel) counts as its two GEMMs
    ffn_calls = []
    orig_ffn = pkg.cabi.ffn_fused_layernorm

    def spy_ffn(x, *a, **k):
        k2 = dict(k)
        k2.pop("out", None)
        ffn_calls.append((x.clone(), a, k2))
        return orig_ffn(x, *a, **k)

    gemm.linear = spy
    pkg.cabi.ffn_fused_layernorm = spy_ffn
    try:
        with torch.no_grad():
            runner.model.forward_encoder(runner.feats, runner.masks, runner.pos, plan=runner.plan,
                                         use_order=runner.use_order)
    finally:
        gemm.linear = orig
        pkg.cabi.ffn_fused_layernorm = orig_ffn
    torch.cuda.synchronize()
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=runner.dev)
    totals = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for x, w, b, a, k in calls:
            orig(x, w, b, *a, **k)
        for x, a, k in ffn_calls:
            orig_ffn(x, *a, out=x, **k)
        e1.record()
        torch.cuda.synchronize()
        totals.append(e0.elapsed_time(e1))
    flops = sum(2 * (x.numel() // x.shape[-1]) * w.shape[0] * w.shape[1] for x, w, _, _, _ in calls)
    flops += sum(2 * 2 * (x.numel() // 256) * 256 * a[0][0].shape[0] for x, a, _ in ffn_calls)  # a[0] = (W1_hi, W1_lo, scale)
    return statistics.median(totals), flops, len(calls) + 2 * len(ffn_calls)


def use_host_cores():
    """The CPU arm uses every PHYSICAL core this process may run on (torchrun pins OMP_NUM_THREADS=1 by default).  One
    thread per logical CPU was measured on the pool's 64-core / 128-thread hosts: 0.045 images/s at 128 threads against
    0.56 at 64 (gpurun_out/r2_bench_a.json vs BENCH_r01.json) -- SMT siblings fight over the FMA units -- so the faster,
    fairer setting is used and its thread count reported as `cores`."""
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        pass
    smt = 1
    try:
        sib = open("/sys/devices/system/cpu/cpu0/topology/thread_siblings_list").read().strip()
        smt = max(1, len([x for part in sib.split(",") for x in ([part] if "-" not in part else
                                                                  range(int(part.split("-")[0]), int(part.split("-")[1]) + 1))]))
    except Exception:
        smt = 2 if n >= 16 else 1
    torch.set_num_threads(max(1, n // smt))
    return torch.get_num_threads()


def numa_node_cpus():
    """-> list of cpu sets, one per NUMA node that this process may run on."""
    nodes = []
    try:
        allowed = set(os.sched_getaffinity(0))
        base = "/sys/devices/system/node"
        for d in sorted(os.listdir(base)):
            if d.startswith("node") and d[4:].isdigit():
                cpus = set()
                for part in open(f"{base}/{d}/cpulist").read().strip().split(","):
                    if part:
                        lo, _, hi = part.partition("-")
                        cpus.update(range(int(lo), int(hi or lo) + 1))
                if cpus & allowed:
                    nodes.append(cpus & allowed)
    except Exception:
        pass
    return nodes


def best_cpu_setting(step, feats, masks, pos):
    """The CPU arm runs at the FASTEST of two settings (a fair baseline, not a strawman): every physical core of the host,
    or the physical cores of one NUMA node (cross-socket traffic costs this workload more than the second socket's cores
    bring: measured 0.56 images/s on 2 x 32 cores against 0.94 on 32 cores of one node).  One timed forward each."""
    start = set(os.sched_getaffinity(0))
    results = []
    for name, cpus in [("all nodes", start)] + [(f"node {i}", c) for i, c in enumerate(numa_node_cpus()[:1]) if c != start]:
        os.sched_setaffinity(0, cpus)
        n = use_host_cores()
        step(feats, masks, pos)
        t0 = time.time()
        step(feats, masks, pos)
        results.append((time.time() - t0, name, cpus, n))
    dt, name, cpus, n = min(results, key=lambda r: r[0])
    os.sched_setaffinity(0, cpus)
    use_host_cores()
    return n, name, [(r[1], r[3], round(r[0], 3)) for r in results]


def model_cfg(model):
    m = model.encoder.layers[0]
    return dict(heads=m.n_heads, points=m.self_attn.num_points, topk_sa=m.topk_sa, num_layers=model.encoder.num_layers,
                level_filter_ratio=model.level_filter_ratio.tolist(), layer_filter_ratio=model.layer_filter_ratio.tolist())


def reference_step_fn(model, device="cpu"):
    """One encoder-half forward (salience_transformer.py:106-183) of the REFERENCE on `device`, same weights as `model`.
    -> (step(feats, masks, pos) -> memory, kind, description).  kind "reference": the unmodified reference modules
    installed under baseline/_ref (oracle/ref_import.py; on a GPU its pure-PyTorch grid_sample MSDA runs, because its
    CUDA extension does not build against this torch); kind "port": the oracle's torch restatement (fallback when the
    install is absent)."""
    from oracle import ref_import  # reference arm / cpu_baseline / gpu_comparator legs only
    cfg = model_cfg(model)
    if ref_import.available():
        m = model.encoder.layers[0]
        tr = ref_import.build_transformer(
            embed_dim=model.embed_dim, d_ffn=m.linear1.out_features, n_heads=m.n_heads, n_levels=model.num_feature_levels,
            n_points=m.self_attn.num_points, num_layers=model.encoder.num_layers, num_classes=model.num_classes,
            level_filter_ratio=cfg["level_filter_ratio"], layer_filter_ratio=cfg["layer_filter_ratio"], topk_sa=m.topk_sa,
            max_num_embedding=model.encoder.background_embedding.row_embed.num_embeddings)
        sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
        res = tr.load_state_dict(sd, strict=False)
        assert not res.unexpected_keys, res.unexpected_keys  # our parameter names ARE the reference's
        tr = tr.to(device).eval()
        return (lambda f, mk, p: ref_import.run_encoder_half(tr, f, mk, p)[0], "reference",
                "unmodified reference modules (baseline/_ref: models/bricks/salience_transformer.py:106-183 with the "
                "pure-PyTorch grid_sample MSDA, ms_deform_attn.py:159-212), same weights and inputs")
    from oracle import oracle as orc
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}

    def port(f, mk, p):
        with torch.no_grad():
            return orc.encoder_half_forward(sd, f, mk, p, cfg, core="torch")[0]

    return port, "port", "oracle port of the reference PyTorch CPU path (baseline/_ref not installed)"


def cpu_baseline(pkg, model, budget_s=20.0):
    """The reference's CPU path on this host's cores, bounded sample (full bs=2 forwards for about `budget_s`)."""
    from salience_detr_b200.synthetic import make_inputs
    feats, masks, pos = make_inputs(WORKLOAD, seed=0)
    step, kind, desc = reference_step_fn(model, "cpu")
    cores, where, tried = best_cpu_setting(step, feats, masks, pos)
    desc += f"; threads: {cores} on {where} (tried {tried})"
    times = []
    t_end = time.time() + budget_s
    while len(times) < 2 or (time.time() < t_end and len(times) < 10):
        t0 = time.time()
        step(feats, masks, pos)
        times.append(time.time() - t0)
    b = feats[0].shape[0]
    return {"value": round(b / statistics.median(times), 4), "unit": "images/s", "cores": cores, "kind": kind,
            "sample": f"{len(times)} full bs={b} encoder forwards of {WORKLOAD} (median), torch CPU fp32; {desc}"}


def gpu_comparator(model, feats, masks, pos, steps=10, warmup=3):
    """What the reference really executes on this image ON THE B200: its own modules (pure-PyTorch MSDA, ~40 host syncs
    and ~1000 launches per forward), same weights / inputs, CUDA-event timed like tools/benchmark_model.py:44-61."""
    step, kind, desc = reference_step_fn(model, feats[0].device)
    if kind != "reference":
        return {"unavailable": "baseline/_ref not installed"}
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False  # fp32 like the reference's default
    try:
        for _ in range(warmup):
            mem = step(feats, masks, pos)
        torch.cuda.synchronize()
        ts = []
        for _ in range(steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            mem = step(feats, masks, pos)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    b = feats[0].shape[0]
    ms = statistics.median(ts)
    return {"value": round(1000.0 * b / ms, 2), "unit": "images/s", "ms_per_step": round(ms, 3), "steps": steps,
            "impl": desc + "; fp32 (allow_tf32 off), eager, no CUDA graph", "memory_checksum": float(mem.double().abs().mean())}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path, all host cores, rank 0 only."""
    if rank != 0:
        return
    from salience_detr_b200.synthetic import build_model, make_inputs
    model = build_model()
    feats, masks, pos = make_inputs(WORKLOAD, seed=0)
    step, kind, desc = reference_step_fn(model, "cpu")
    cores, where, tried = best_cpu_setting(step, feats, masks, pos)
    desc += f"; threads: {cores} on {where} (tried {tried})"
    for _ in range(args.warmup):
        step(feats, masks, pos)
    t0 = time.time()
    for _ in range(args.steps):
        step(feats, masks, pos)
    dt = time.time() - t0
    b = feats[0].shape[0]
    val = round(args.steps * b / dt, 4)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1000 * dt / args.steps, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "impl": desc},
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": kind,
                             "sample": f"{args.steps} full bs={b} encoder forwards"},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(json.dumps(line))


def run_train(args, rank, world, local):
    """--mode train (BASELINE.json configs[2]: training step, bs=2 per GPU, batch-sharded, NCCL gradient all-reduce):
    encoder-half forward (training path: torch autograd around the MSDA forward / backward kernels) + backward of
    loss = memory.square().mean() + bucketed all-reduce overlapped with the backward (dist.GradientBuckets) + SGD step.
    An extra measurement, not the headline metric."""
    import torch.distributed as dist
    import salience_detr_b200 as pkg
    from salience_detr_b200 import dist as sdist
    from salience_detr_b200.synthetic import build_model, make_inputs
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sdist.bind_to_gpu_numa_node(local)
    sdist.init_from_env("nccl", dev)
    model = build_model().to(dev).train()
    feats, masks, pos = make_inputs(WORKLOAD, seed=sdist.shard_batch_seed(0, rank), device=dev)
    params = [p for p in model.parameters() if p.requires_grad]
    gb = sdist.GradientBuckets(params, bucket_bytes=args.bucket_mb << 20)
    opt = torch.optim.SGD(params, lr=1e-5, foreach=True)
    bsz = feats[0].shape[0]

    with torch.no_grad():
        plan = model.make_plan(masks)   # the masks of the synthetic batch are fixed: one host round trip, outside the step

    def step(comm=True):
        gb.active = comm and world > 1
        gb.zero_()
        mem, _ = model.forward_encoder(feats, masks, pos, plan=plan)
        loss = mem.square().mean()
        loss.backward()
        gb.finish()
        opt.step()
        return loss

    # The eager step is bound by the HOST (~2000 torch launches: 27 ms of CPU per step against 19 ms of device work once the
    # Linear layers are on the tensor cores): capture forward + backward + all-reduce + SGD in one CUDA graph and replay it.
    graphed = None
    eager_step = step
    if not args.no_graph:
        try:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(3):
                    eager_step()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize()
            graphs = {}
            for comm in ([True, False] if world > 1 else [True]):   # the no-all-reduce variant only serves the "exposed" figure
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    static_loss = eager_step(comm)
                graphs[comm] = (g, static_loss)
            graphed = graphs
        except Exception as e:  # capture not possible (e.g. a collective that cannot be captured): eager step
            sys.stderr.write(f"training step not captured ({type(e).__name__}: {str(e)[:300]}): running eagerly\n")
            graphed = None
            torch.cuda.synchronize()
    if graphed is not None:
        def step(comm=True):  # noqa: F811
            g, static_loss = graphed[comm if world > 1 else True]
            g.replay()
            return static_loss

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return sdist.max_over_ranks(e0.elapsed_time(e1), dev)

    steps, warmup = args.steps or 10, max(3, args.warmup or 3)
    with ClockSampler(local) as clk:
        ms = timed(step, steps, warmup)
    ms_nocomm = timed(lambda: step(False), steps, 1) if world > 1 else ms
    n0 = pkg.cabi.launch_count()
    loss = eager_step()              # the launch counter lives on the host side of the C-ABI: count on an eager step
    launches = pkg.cabi.launch_count() - n0
    reached = sum(p.numel() * 4 for p in params if p.grad is not None and bool((p.grad != 0).any()))
    if rank == 0:
        emit(json.dumps({
            "metric": "images/sec encoder fwd+bwd+grad-allreduce+SGD @ 800x1333 bs=2/GPU (training path)",
            "value": round(sdist.aggregate_throughput(bsz, steps, world, ms), 2), "unit": "images/s", "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": round(ms / steps, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD + " training step", "cuda_graph": graphed is not None, "batch_per_gpu": bsz, "global_batch": bsz * world,
                       "parallelism": f"dp{world}: batch-sharded replicas, gradient all-reduce (mean) in {len(gb.buckets)} "
                                      f"bucket(s) of <= {args.bucket_mb} MiB launched from autograd hooks, overlapped with backward",
                       "loss": "memory.square().mean() (the salience-supervision / detection losses are outside the path)"},
            "clocks": clk.summary(),
            "allreduce": {"bytes_per_step": gb.total_bytes, "buckets": len(gb.buckets),
                          "ms_per_step_without_allreduce": round(ms_nocomm / steps, 3),
                          "exposed_ms_per_step": round((ms - ms_nocomm) / steps, 3),
                          "bytes_with_nonzero_gradient": reached},
            "gpu_launches_per_step": launches, "loss": float(loss.detach())}))
    sys.stdout.flush()
    # Tear-down: graphs that captured NCCL kernels must die BEFORE the communicator (a process group destroyed first left the
    # N = 2 run hanging until the timeout killed it), and nothing after the result line may hang the launcher: a watchdog ends the
    # process if the orderly path has not finished in 30 s.
    def _bail():
        time.sleep(30)
        os._exit(0)
    threading.Thread(target=_bail, daemon=True).start()
    if graphed is not None:
        graphed.clear()
        del step, static_loss, g
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, outputs):
    """Write each output the caller of the timed path receives as <out_dir>/<name>.npy in float32, so that two builds can be
    compared output for output on the same seeded inputs.  The encoder memory of the benchmark's workload (2 x 22323 x 256)
    is 45.7 MB and is written whole."""
    import numpy as np
    arrays = {k: v.detach().float().cpu().numpy() for k, v in outputs.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-order", action="store_true")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--gemm", default="auto", choices=["auto", "tcgen05", "3xtf32", "fp32", "tf32"])
    ap.add_argument("--mode", default="forward", choices=["forward", "train"])
    ap.add_argument("--bucket-mb", type=int, default=32)
    ap.add_argument("--e2e-persistent-ctas", type=int, default=0,
                    help="cap of the persistent GEMM / FFN kernels during the e2e (multi-lane) measurement; 0 = one CTA per SM")
    ap.add_argument("--pipeline-depth", type=int, default=4, help="lanes of the host-buffer pipeline (e2e)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last timed step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    _claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        args.steps = args.steps if args.steps is not None else 5
        args.warmup = args.warmup if args.warmup is not None else 1
        return run_reference(args, rank, world)
    if args.mode == "train":
        if not torch.cuda.is_available():
            raise SystemExit("bench.py --mode train needs a GPU")
        return run_train(args, rank, world, local)
    args.steps = args.steps if args.steps is not None else 50
    args.warmup = max(3, args.warmup if args.warmup is not None else 10)

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: the sm_100a path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    import salience_detr_b200 as pkg
    from salience_detr_b200 import dist as sdist
    numa = sdist.bind_to_gpu_numa_node(local)  # before any pinned allocation: host buffers land on the GPU's node
    sdist.init_from_env("nccl", dev)

    from salience_detr_b200.runner import EncoderRunner
    from salience_detr_b200.synthetic import build_model, make_inputs

    torch.backends.cuda.matmul.allow_tf32 = False  # torch default; gemm.linear enables TF32 only for split operands
    pkg.gemm.MODE = args.gemm
    model = build_model().to(dev)
    # the detector's position embedding (configs/salience_detr/salience_detr_resnet50_800_1333.py:32): lets the host-buffer
    # API derive the embedding from the masks on the device instead of shipping 45.7 MB of it per step
    model.attach_position_embedding(pkg.PositionEmbeddingSine(model.embed_dim // 2, temperature=10000, normalize=True, offset=-0.5))
    feats_h, masks_h, pos_h = make_inputs(WORKLOAD, seed=sdist.shard_batch_seed(0, rank))  # weak scaling: replicas
    feats = [t.to(dev) for t in feats_h]
    masks = [t.to(dev) for t in masks_h]
    pos = [t.to(dev) for t in pos_h]
    runner = EncoderRunner(model, feats, masks, pos, use_graph=not args.no_graph, use_order=not args.no_order)
    bsz = feats[0].shape[0]
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    stream = runner.stream

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps, warmup, on_start=None):
        """W untimed + K timed steps; per-step CUDA events on the launching stream; L2 flushed between steps
        (outside the events).  Returns total ms of the K steps (max over ranks)."""
        with torch.cuda.stream(stream):
            for _ in range(warmup):
                fn()
        barrier()
        if on_start is not None:
            on_start()
        pairs = []
        with torch.cuda.stream(stream):
            for _ in range(steps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                fn()
                e1.record(stream)
                pairs.append((e0, e1))
        barrier()
        return sdist.max_over_ranks(sum(a.elapsed_time(b) for a, b in pairs), dev)

    with ClockSampler(local) as clk:
        clk.wait_first()
        total_ms = timed(runner.step, args.steps, args.warmup, on_start=clk.mark)
        clk.mark_end()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"memory": runner.memory})
        t_probe = time.time()
        while clk.proc is not None and clk.since_mark() < 3 and time.time() - t_probe < 3.0:  # same step, same flush, untimed
            with torch.cuda.stream(stream):
                for _ in range(20):
                    flush.zero_()
                    runner.step()
            torch.cuda.synchronize()
    clocks = clk.summary()
    value = sdist.aggregate_throughput(bsz, args.steps, world, total_ms)

    # end to end through the public host-buffer API (the detector-side boundary, salience_detr.py:172-203: feature maps and
    # padding masks in, memory out; the sine position embedding is a function of the masks and is derived on the device).
    # Every step copies its feature maps from pinned host memory and its result back.  serial = one stream; pipelined =
    # HostPipeline, double-buffered, copies overlap compute.  Every timed leg runs --steps steps; 20 steps (60 ms) proved
    # too short for a stable e2e figure, so use >= 200 when e2e matters.
    from salience_detr_b200.runner import HostPipeline
    e2e_steps = args.steps
    host_runner = EncoderRunner(model, feats, masks, None, use_graph=not args.no_graph, use_order=not args.no_order)
    host_runner.bind_host(feats_h)
    stream_keep, stream = stream, host_runner.stream
    e2e_serial_ms = timed(host_runner.run_host, args.steps, 3)
    stream = stream_keep
    pkg.cabi.lib().sdetr_set_persistent_ctas(args.e2e_persistent_ctas)  # grid sizes are fixed when the lanes' graphs are captured
    pipe = HostPipeline(model, feats, masks, None, depth=args.pipeline_depth, use_graph=not args.no_graph, use_order=not args.no_order)
    host_batch = ([t.pin_memory() for t in feats_h], None)
    pipe.run([host_batch] * 4)  # warm-up
    barrier()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    pipe.h2d.wait_event(t0)
    pipe.run([host_batch] * e2e_steps)  # returns when the last output is in host memory
    t1.record()
    barrier()
    e2e_ms = sdist.max_over_ranks(t0.elapsed_time(t1), dev)
    pkg.cabi.lib().sdetr_set_persistent_ctas(0)
    e2e_val = sdist.aggregate_throughput(bsz, e2e_steps, world, e2e_ms)

    # fresh masks every step: nothing derived from the masks is reused -- masks H2D, plan (two launches + one host
    # round trip), position tokens, an EAGER forward (top-k sizes are host integers of the plan, so a captured graph
    # cannot be replayed for new masks), memory D2H.  The honest cost of a batch whose padding was never seen before.
    masks_pin = [m.pin_memory() for m in masks_h]
    feats_pin = host_batch[0]
    out_pin = torch.empty(host_runner.memory.shape, dtype=torch.float32, pin_memory=True)

    def fresh_step():
        f = [t.to(dev, non_blocking=True) for t in feats_pin]
        m = [t.to(dev, non_blocking=True) for t in masks_pin]
        with torch.no_grad():
            mem, _ = model.forward_encoder(f, m, None, plan=None, use_order=not args.no_order)
        out_pin.copy_(mem, non_blocking=True)

    stream_keep, stream = stream, torch.cuda.current_stream(dev)
    fresh_ms = timed(fresh_step, args.steps, 3)
    fresh_serial_val = sdist.aggregate_throughput(bsz, args.steps, world, fresh_ms)
    stream = stream_keep
    # the same, pipelined: copies, plan (own stream) and eager forwards of consecutive batches overlap; every batch still pays
    # its own plan and an eager forward
    from salience_detr_b200.runner import FreshMaskPipeline
    fpipe = FreshMaskPipeline(model, feats, masks, depth=3, use_order=not args.no_order)
    fresh_batch = (feats_pin, masks_pin)
    fpipe.run([fresh_batch] * 6)
    barrier()
    fresh_steps = args.steps
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    fpipe.h2d.wait_event(t0)
    fpipe.run([fresh_batch] * fresh_steps)
    t1.record()
    barrier()
    fresh_val = sdist.aggregate_throughput(bsz, fresh_steps, world, sdist.max_over_ranks(t0.elapsed_time(t1), dev))

    line = None
    if rank == 0:
        byts = msda_layer_bytes(runner)
        cold = time_msda_kernels(pkg, runner)
        try:
            med, how = time_msda_in_situ(pkg, runner)
            assert len(med) == len(byts) and all(x > 0 for x in med)
        except Exception as e:  # external event nodes unavailable: fall back to the isolated replay
            med, how = cold, f"isolated replay after an L2 flush (in-situ timing failed: {type(e).__name__}: {e})"
        peak, peak_src = peaks()
        achieved = sum(byts) / (sum(med) / 1000.0) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "msda_traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("dram_bytes_per_launch_mean")
            except Exception:
                traffic = None
        gemm_ms, gemm_flops, gemm_calls = time_gemm_kernels(pkg, runner)
        f16 = pkg.gemm.MODE == "auto" and pkg.gemm.OWN_KERNEL == "f16x3"
        try:
            tf32_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"] / (1.0 if f16 else 2.0)
            gemm_peak_src = "MEASURED_PEAKS.json bf16_tflops" + ("" if f16 else " / 2 (TF32 dense = half the bf16 rate)")
        except Exception:
            tf32_peak = 1590.0 / (1.0 if f16 else 2.0)  # B200_PROFILING.md fallback
            gemm_peak_src = "fallback (B200_PROFILING.md)"
        passes = 1 if pkg.gemm.MODE in ("fp32", "tf32") else 3
        gemm_exec = passes * gemm_flops / (gemm_ms / 1000.0) / 1e12
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(total_ms / args.steps, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": bsz, "global_batch": bsz * world,
                       "parallelism": f"dp{world} (independent replicas, no forward collective)",
                       "weights": "random init (seed 0) + N(0,0.02) sampling-offset weights",
                       "gemm": {"auto": ("3xFP16 (fp32-class accuracy, 22-bit operands: hi/lo fp16 split with exact power-of-two range scaling): "
                                         "hand-written persistent tcgen05.mma.kind::f16 GEMM" if pkg.gemm.OWN_KERNEL == "f16x3" else
                                         "3xTF32 (fp32-class accuracy): hand-written persistent tcgen05.mma.kind::tf32 GEMM") +
                                        " (TMA, pre-split weight, activation split in the kernel into tensor memory, double-buffered TMEM "
                                        "accumulator, TMA-store epilogue) for every projection; linear1 -> ReLU -> linear2 -> +residual -> LayerNorm of the encoder "
                                        "layers as ONE tensor-core kernel with the hidden activations in tensor memory; GEMMs of <= 2304 rows "
                                        "(latency-bound) on cuBLAS fp32 or the two-launch small-level predictor kernels",
                                "tcgen05": "hand-written tcgen05.mma.kind::tf32 GEMM (TMA, in-kernel 3xTF32 split, TMEM accumulator; fp32-class accuracy)",
                                "3xtf32": "cuBLAS TF32 tensor cores on 3-way split operands (3xTF32, fp32-class accuracy)",
                                "fp32": "cuBLAS fp32 SIMT", "tf32": "cuBLAS TF32 (reduced precision)"}[pkg.gemm.MODE], "cuda_graph": runner.graph is not None,
                       "msda_order": "spatial tiles" if runner.use_order else "score order",
                       "l2": "256 MiB flush between timed steps (outside the events)"},
            "clocks": clocks,
            "e2e": {"value": round(e2e_val, 2), "unit": "images/s", "h2d_bytes_per_step": host_runner.h2d_bytes,
                    "d2h_bytes_per_step": host_runner.d2h_bytes, "ms_per_step": round(e2e_ms / e2e_steps, 4), "steps": e2e_steps,
                    "pipeline_depth": args.pipeline_depth, "persistent_ctas": args.e2e_persistent_ctas or "one per SM",
                    "api": "salience_detr_b200.runner.HostPipeline.run (pinned host feature maps in, memory out, double-buffered: "
                           "H2D, forward and D2H of consecutive batches overlap; the sine position embedding is derived from "
                           "the padding masks on the device, as in the detector, salience_detr.py:172-176)",
                    "serial_value": round(sdist.aggregate_throughput(bsz, args.steps, world, e2e_serial_ms), 2),
                    "serial_api": "EncoderRunner.run_host (one stream: H2D -> forward -> D2H per step)",
                    "fresh_masks_value": round(fresh_val, 2),
                    "fresh_masks_serial_value": round(fresh_serial_val, 2),
                    "fresh_masks_api": "runner.FreshMaskPipeline (3 lanes; _serial_: one stream): per step feats + masks H2D, make_plan (sdetr_mask_plan + one host round trip), position "
                                       "tokens, EAGER forward_encoder (no CUDA graph), memory D2H",
                    "numa": numa},
            "gpu_launches": runner.launches_per_step * args.steps,
            "gpu_launches_per_step": runner.launches_per_step,
            "roofline": {"bound": "hbm (SURVEY.md 8(d) denominator; measured: the gather is bound by the L1 tag stage, ~2 clk per "
                                  "128-byte line, DESIGN.md 3.1)",
                         "kernel": "sdetr::msda_fwd_kernel<32,4,4,fused> (6 launches/step)",
                         "achieved": round(achieved, 1), "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                         "frac": round(achieved / peak, 4), "traffic": traffic,
                         "algorithmic_bytes_per_step": int(sum(byts)), "kernel_ms_per_step": round(sum(med), 4),
                         "per_layer_us": [round(1000 * x, 1) for x in med], "timing": how,
                         "isolated_cold": {"kernel_ms_per_step": round(sum(cold), 4),
                                           "frac": round(sum(byts) / (sum(cold) / 1000.0) / 1e9 / peak, 4),
                                           "per_layer_us": [round(1000 * x, 1) for x in cold],
                                           "how": "the same six launches replayed alone after an L2 flush (round-1 definition)"}},
            # secondary leg: the dense projections (tensor-bound; 3xTF32 issues 3 TF32 MMA passes per logical product)
            "roofline_gemm": {"bound": "tensor (measured: the kernel is bound by L2<->SM operand/result traffic, DESIGN.md 3.4)",
                              "kernels": ("sdetr::gemm_f16x3_kernel + sdetr::ffn_fused_kernel (3xFP16, tcgen05.mma.kind::f16; the FFN keeps its hidden activations in tensor memory)" if f16 else
                                          "sdetr::gemm_3xtf32_p_kernel<presplit>") + " (+ cuBLAS fp32 for <= 2304-row GEMMs)",
                              "achieved": round(gemm_exec, 1), "peak": round(tf32_peak, 1), "peak_source": gemm_peak_src,
                              "unit": "TFLOP/s", "frac": round(gemm_exec / tf32_peak, 4),
                              "logical_tflops": round(gemm_flops / (gemm_ms / 1000.0) / 1e12, 1),
                              "mma_passes": passes, "gemm_calls_per_step": gemm_calls,
                              "kernel_ms_per_step": round(gemm_ms, 4)},
        }
        if world == 1 and not args.skip_cpu_baseline:
            line["gpu_comparator"] = gpu_comparator(model, feats, masks, pos)
            line["cpu_baseline"] = cpu_baseline(pkg, model)
        emit(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
