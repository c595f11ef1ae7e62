#!/usr/bin/env python
"""Benchmark of the ALIGNN edge-gated conv hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--norm batchnorm|layernorm]
                    [--dump-outputs DIR]

A "step" is one forward + backward + optimizer update of ALIGNN (4 ALIGNN + 4 GCN layers, hidden
256, the `ALIGNN` class of alignn/models/alignn.py, L1 loss as in train.py:240) on one synthetic
JARVIS-DFT-shaped batch of 64 crystals per GPU (30 atoms, k=12: N=1920, E=23 040, T=276 480).
Weak scaling: every rank owns its own 64 graphs; the only collective is the gradient all-reduce.

Prints ONE JSON line (rank 0).  Keys follow the driver contract; extra keys:
  roofline      dominant kernel (fused edge kernel on L(g)): compulsory bytes / CUDA-event time
  step_hbm      whole-step compulsory bytes (SURVEY.md section 8d: 10.04 GB per batch fwd+bwd) / step time
  cpu_baseline  the oracle (torch-CPU restatement of the reference DGL path) on this box's cores
  e2e           same metric with the batch starting in pinned HOST memory every step and the loss read back
`--impl reference` times that CPU oracle alone (the reference's own implementation needs DGL, which
cannot be installed offline; see DESIGN.md).
`--dump-outputs DIR` writes what the last timed step of `value` returned as float32 .npy files (rank 0): out.npy
(predictions), loss.npy, grad.npy (the flat gradient buffer) and state.npy (every floating-point tensor of the model's
state_dict after the optimizer update, flattened in state_dict order), 32 MB for the default model.  Inputs,
initialisation and the number of steps before it are fixed by the arguments, so two builds run with the same
arguments can be compared output for output.
"""
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

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "graphs/sec fwd+bwd"
UNIT = "graphs/s"
WORKLOAD = "configs[2]: ALIGNN training fwd+bwd+AdamW, batch=64 JARVIS-shaped graphs/GPU (30 atoms, k=12), 4+4 layers d=256"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--norm", default="batchnorm", choices=["batchnorm", "layernorm"])
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--atoms", type=int, default=30)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying CUDA graphs")
    ap.add_argument("--cpu-sample-graphs", type=int, default=0, help="0 = calibrate (~4 s of CPU work per step)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


# ---------------------------------------------------------------------------------------------
# shared: byte model (SURVEY.md section 8d / BASELINE.md section 3)
# ---------------------------------------------------------------------------------------------
def conv_bytes_train(Nn, Ne, d):
    fwd = 4 * d * (2 * Nn + 2 * Ne) + 8 * Ne + 4 * d * Ne          # inference fwd + save m
    bwd = 4 * d * (5 * Nn + 4 * Ne) + 8 * Ne
    return fwd + bwd


def step_bytes(N, E, T, d, n_alignn, n_gcn):
    return n_alignn * (conv_bytes_train(N, E, d) + conv_bytes_train(E, T, d)) + n_gcn * conv_bytes_train(N, E, d)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            j = json.load(fh)
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------
# CPU oracle arm (cpu_baseline and --impl reference)
# ---------------------------------------------------------------------------------------------
def _oracle_setup(args, graphs):
    """One fwd+bwd+AdamW step of the oracle on `graphs` crystals.  Inputs come from oracle/synthetic_inputs.py (the same
    generator as the product's, restated with oracle types): nothing of alignn_b200 is imported on this arm."""
    from oracle import alignn_oracle as O
    from oracle import synthetic_inputs as SI
    og, olg, lat, tgt = SI.make_batch(batch_size=graphs, atoms=args.atoms, k=12, seed=123)
    torch.manual_seed(123)
    model = O.ALIGNN(norm=args.norm)
    model.train()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)

    def step():
        opt.zero_grad(set_to_none=True)
        out = model((og, olg, lat))
        loss = (out - tgt).abs().mean()
        loss.backward()
        opt.step()
    return step


def cpu_calibrate(args, graphs):
    """Host thread count the oracle runs fastest with, measured on the SAME `graphs`-crystal step that is then timed
    (more threads is not faster for these gather/index_add-heavy ops on a 100+ core box)."""
    ncpu = os.cpu_count() or 1
    cands = sorted({min(ncpu, c) for c in (16, 32, 64)})
    step = _oracle_setup(args, graphs)
    best = None
    for th in cands:
        torch.set_num_threads(th)
        step()
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if best is None or dt < best[1]:
            best = (th, dt)
    return best


def cpu_oracle_run(args, graphs, steps, warmup, threads):
    """graphs/s of the oracle (fwd+bwd+AdamW) on `graphs` crystals per step with `threads` host threads."""
    torch.set_num_threads(threads)
    step = _oracle_setup(args, graphs)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    return graphs * len(times) / total, total / len(times) * 1e3


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    graphs = args.cpu_sample_graphs if args.cpu_sample_graphs > 0 else args.batch     # the full 64-graph batch by default
    threads, dt = cpu_calibrate(args, graphs)
    warm = max(1, min(args.warmup, 3))
    if args.cpu_sample_graphs <= 0 and (args.steps + warm) * dt > 150.0:
        # keep the whole run within a few minutes: a bounded sample of the batch per step (time per graph is flat in the
        # batch size for this path: block-diagonal graphs)
        graphs = int(max(8, min(args.batch, args.batch * 150.0 / ((args.steps + warm) * dt))))
    gps, ms = cpu_oracle_run(args, graphs, args.steps, warm, threads)
    line = {
        "impl": "reference", "metric": METRIC, "value": gps, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the workload keys are the same in both arms (the reference arm times a bounded sample of it: cpu_baseline.sample)
        "config": {"workload": WORKLOAD, "norm": args.norm, "global_batch": args.batch * args.gpus, "per_gpu_batch": args.batch,
                   "parallelism": f"dp{args.gpus}", "optimizer": "AdamW", "loss": "L1",
                   "l2": "not applicable (host cores)"},
        "run": {"device": "host cores (reference arm)",
                "sample": f"{graphs} graphs per step" + ("" if graphs == args.batch else " (bounded CPU sample of the 64-graph batch)")},
        "cpu_baseline": {"value": gps, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{args.steps} steps x {graphs} graphs, torch-CPU restatement of the reference DGL path "
                                   f"(DGL is not installable offline); thread count calibrated on the same step over "
                                   f"{os.cpu_count()} cores"},
        "e2e": {"value": gps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# clocks sampler
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([t.strip() for t in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 6:
                continue
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except ValueError:
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def dump_outputs(directory, out, loss, grad, model):
    """One step's predictions, loss, flat gradient buffer and resulting model state as float32 .npy files."""
    os.makedirs(directory, exist_ok=True)
    state = torch.cat([t.reshape(-1).float() for t in model.state_dict().values() if t.is_floating_point()])
    for name, t in (("out", out), ("loss", loss), ("grad", grad), ("state", state)):
        np.save(os.path.join(directory, name + ".npy"), t.detach().float().cpu().numpy())


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def run_ours(args):
    from alignn_b200 import _lib, dp, ops, synthetic
    from alignn_b200.alignn import ALIGNN, ALIGNNConfig

    rank, local, world = dp.init_from_env("nccl")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU path")
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.load()

    # ---- model ------------------------------------------------------------------------------
    torch.manual_seed(123)                                   # reference default seed, config.py:164
    cfg = ALIGNNConfig(name="alignn")
    if args.norm == "layernorm":
        from alignn_b200 import alignn_atomwise as AW

        class Model(ALIGNN):
            _mlp, _alignn_conv, _gcn_conv = AW.MLPLayer, AW.ALIGNNConv, AW.EdgeGatedGraphConv
        model = Model(cfg)
    else:
        model = ALIGNN(cfg)
    model.to(dev).train()
    dp.broadcast_parameters(model)
    use_graph = not args.no_graph
    reducer = dp.FlatGradAllReducer(model.parameters())
    opt = None            # dp.FlatAdamW, built after the first backward has shown which parameters train

    # ---- data: each rank owns its own batches (weak scaling); 4 distinct batches rotate ------
    nb = 4
    host = []
    for b in range(nb):
        g, lg, lat, tgt = synthetic.make_batch(batch_size=args.batch, atoms=args.atoms, k=12,
                                               seed=123 + 1000 * rank + b)
        host.append((g.pin_memory(), lg.pin_memory(), lat.pin_memory(), tgt.pin_memory()))
    N, E, T = host[0][0].num_nodes(), host[0][0].num_edges(), host[0][1].num_edges()
    resident = [(g.to(dev), lg.to(dev), lat.to(dev), tgt.to(dev)) for g, lg, lat, tgt in host]
    h2d_bytes = host[0][0].nbytes() + host[0][1].nbytes() + host[0][2].numel() * 4 + host[0][3].numel() * 4

    def step(batch):
        g, lg, lat, tgt = batch
        reducer.zero_grad()
        out = model((g, lg, lat))
        loss = (out - tgt).abs().mean()                      # nn.L1Loss, train.py:240
        with reducer.deferring():                            # weight-gradient GEMMs queued: one batched launch in gather()
            loss.backward()
        reducer.all_reduce()
        opt.step()
        return out, loss

    def h2d(i):
        g, lg, lat, tgt = host[i % nb]
        return (g.to(dev, non_blocking=True), lg.to(dev, non_blocking=True), lat.to(dev, non_blocking=True),
                tgt.to(dev, non_blocking=True))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=cpu_group_ref[0]) if cpu_group_ref[0] is not None else dist.barrier()
        torch.cuda.synchronize()

    cpu_group_ref = [None]

    # everything below (warm-up, capture, every timed region) runs on ONE side stream: the autograd accumulators are
    # created on the stream that later replays them
    work = torch.cuda.Stream()
    work.wait_stream(torch.cuda.current_stream())

    def timed(fn, steps):
        """EXACTLY `steps` calls between two events on the launching stream, barrier + synchronize on both sides,
        max over ranks.  Returns (ms, what the last call returned)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(work):
            e0.record()
            for i in range(steps):
                last = fn(i)
            e1.record()
        barrier()
        if world > 1 and cpu_group_ref[0] is not None:
            ms = torch.tensor([e0.elapsed_time(e1)])
            dist.all_reduce(ms, op=dist.ReduceOp.MAX, group=cpu_group_ref[0])
            return ms.item(), last
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), last

    # ---- warm-up (also builds the flat gradient buffer, the flat optimizer and the operand-image tables) ------------
    with torch.cuda.stream(work):
        g0, lg0, lat0, tgt0 = resident[0]
        reducer.zero_grad()
        (model((g0, lg0, lat0)) - tgt0).abs().mean().backward()
        reducer.gather()
        opt = dp.FlatAdamW(reducer, lr=1e-3, capturable=use_graph)
        for i in range(max(args.warmup, 3)):
            step(resident[i % nb])
    barrier()

    # ---- CUDA graphs: one per resident batch and one per host batch (H2D copies inside the graph) --------
    # The step is a few hundred launches of which most are small (g-graph convs, norms, optimizer); replaying them as
    # a graph removes the host launch cost.  Shapes are static here; a variable-size loader buckets (DESIGN.md).
    # The gradient all-reduce stays OUTSIDE the graphs: per step = replay(zero_grad + forward + backward) -> eager flat
    # all-reduce -> replay(optimizer).
    graphs_res, graphs_e2e, graph_opt, launches_per_step = [], [], None, None

    # ALIGNN_B200_NCCL_IN_GRAPH=1: capture the all-reduce and the optimizer into the same graph as forward + backward
    # (one replay per step).  Round 1 reported a hang: the capture and the replays are fine (tools/nccl_in_graph_probe.py,
    # capture_error_mode="thread_local" keeps the process-group watchdog out of the capture); what hangs on this stack is
    # an eager NCCL barrier AFTER captured collectives were replayed, so the rank barrier of the timed regions is a
    # gloo (CPU) barrier in this mode.  Opt-in until it has run at 8 GPUs.
    nccl_in_graph = use_graph and world > 1 and os.environ.get("ALIGNN_B200_NCCL_IN_GRAPH", "0") == "1"
    cpu_group_ref[0] = dist.new_group(backend="gloo") if nccl_in_graph else None

    def fwd_bwd(batch):
        g, lg, lat, tgt = batch
        reducer.zero_grad()
        out = model((g, lg, lat))
        loss = (out - tgt).abs().mean()
        with reducer.deferring():
            loss.backward()
        reducer.gather()                                      # batched weight gradients + the other gradients -> flat buffer
        if nccl_in_graph:
            reducer.reduce_flat()
            opt.step()
        return out, loss

    if use_graph:
        pool = None
        for b in range(nb):
            gr = torch.cuda.CUDAGraph()
            l0 = _lib.launch_count()
            with torch.cuda.graph(gr, pool=pool, stream=work, capture_error_mode="thread_local" if nccl_in_graph else "global"):
                out_b, loss_b = fwd_bwd(resident[b])
            launches_per_step = _lib.launch_count() - l0
            pool = pool or gr.pool()
            graphs_res.append((gr, out_b, loss_b))
        if not nccl_in_graph:
            graph_opt = torch.cuda.CUDAGraph()
            l0 = _lib.launch_count()
            with torch.cuda.graph(graph_opt, pool=pool, stream=work):
                opt.step()
            launches_per_step += _lib.launch_count() - l0         # the flat AdamW launch is one of the library's kernels
        barrier()

    def run_resident(i):
        """One step on resident batch i % nb; returns (predictions, loss), valid until that batch's next step."""
        if use_graph:
            gr, out, loss = graphs_res[i % nb]
            gr.replay()
            if not nccl_in_graph:
                reducer.reduce_flat()
                graph_opt.replay()
            return out, loss
        return step(resident[i % nb])

    # End to end = what a training loop with a prefetching loader does (train.py's DataLoader has pin_memory and
    # worker prefetch): while the GPU works on batch i, a copy stream moves batch i+1 from pinned host memory into the
    # device buffers of its slot; the loss of every step is copied back to pinned memory and read by the host one step
    # later (the step itself never waits for the host).  Every timed step still pays its own H2D copy and D2H read: the
    # first step of a region copies its own inputs serially if nobody prefetched them.
    from alignn_b200.runtime import BucketedForward
    copy_stream = torch.cuda.Stream()
    copy_done = [torch.cuda.Event() for _ in range(nb)]
    compute_done = [torch.cuda.Event() for _ in range(nb)]
    loss_host = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ready = [torch.cuda.Event() for _ in range(2)]
    pf = {"slot_has": None, "last_loss": 0.0}

    def prefetch(i):
        b = i % nb
        g_h, lg_h, lat_h, tgt_h = host[b]
        g_d, lg_d, lat_d, tgt_d = resident[b]
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(compute_done[b])           # the previous step that read this slot has finished
            BucketedForward._copy_graph(g_d, g_h)
            BucketedForward._copy_graph(lg_d, lg_h)
            lat_d.copy_(lat_h, non_blocking=True)
            tgt_d.copy_(tgt_h, non_blocking=True)
            copy_done[b].record(copy_stream)
        pf["slot_has"] = i

    def run_e2e(i):
        if not use_graph:
            return step(h2d(i))[1].item()                     # D2H + sync, as train.py:300-305 does
        b = i % nb
        if pf["slot_has"] != i:
            prefetch(i)                                       # nobody copied this step's inputs yet: do it now
        work.wait_event(copy_done[b])
        gr, _, loss_b = graphs_res[b]
        gr.replay()
        if not nccl_in_graph:
            reducer.reduce_flat()
            graph_opt.replay()
        compute_done[b].record(work)
        loss_host[i % 2].copy_(loss_b.detach(), non_blocking=True)
        loss_ready[i % 2].record(work)
        prefetch(i + 1)                                       # overlaps with the step just launched
        if i > 0:
            loss_ready[(i - 1) % 2].synchronize()             # the host reads every step's loss, one step late
            pf["last_loss"] = float(loss_host[(i - 1) % 2])
        return pf["last_loss"]

    with torch.cuda.stream(work):
        for i in range(2):
            run_resident(i)

    # ---- timed: resident inputs -------------------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count()
    ms_total, (out_last, loss_last) = timed(run_resident, args.steps)
    launches = (launches_per_step * args.steps) if use_graph else (_lib.launch_count() - l0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out_last, loss_last, reducer.flat, model)

    # ---- timed: end to end from pinned host memory, loss read back every step ----------------
    with torch.cuda.stream(work):
        for i in range(2):
            run_e2e(i)
    ms_e2e, _ = timed(run_e2e, args.steps)
    clocks = sampler.stop() if rank == 0 else None

    # ---- per-kernel table: CUDA events around every library call in an eager replay of the same steps (events inside
    #      a graph replay carry no timestamps); the roofline entry is the kernel with the largest total time ----------
    with torch.cuda.stream(work):
        for i in range(2):                                    # eager allocations settle on this stream
            step(resident[i % nb])
    ops.TIMER = ops.KernelTimer()
    ms_eager, _ = timed(lambda i: step(resident[i % nb]), args.steps)
    ksum = ops.TIMER.summary()
    ops.TIMER = None

    if world > 1 and cpu_group_ref[0] is not None:
        lt = torch.tensor([launches], dtype=torch.float64)
        dist.all_reduce(lt, group=cpu_group_ref[0])
    else:
        lt = torch.tensor([launches], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(lt)
    if rank != 0:
        if world > 1:
            _finish(nccl_in_graph)
        return

    graphs_per_step = args.batch * world
    value = graphs_per_step * args.steps / (ms_total / 1e3)
    e2e_value = graphs_per_step * args.steps / (ms_e2e / 1e3)
    peak, peak_src = peaks()
    d = cfg.hidden_features
    sbytes = step_bytes(N, E, T, d, cfg.alignn_layers, cfg.gcn_layers)
    ms_step = ms_total / args.steps
    traffic_tab = {}
    tpath = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")     # dram bytes per launch from `ncu --set full` captures
    if os.path.exists(tpath) and args.norm == "batchnorm" and (N, E, T) == (1920, 23040, 276480):
        with open(tpath) as fh:
            traffic_tab = json.load(fh)

    def entry(name, k):
        # the kernel's L(g)-sized launches: algorithmic bytes / event time
        ach = k["big_bytes"] / (k["big_ms"] * 1e-3) / 1e9 if k["big_ms"] > 0 else 0.0
        tr = traffic_tab.get(name)
        return {"kernel": name, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": (tr or {}).get("dram_bytes_per_launch"), "traffic_source": (tr or {}).get("source"),
                "share_of_eager_step": k["total_ms"] / ms_eager, "ms_per_step": k["total_ms"] / args.steps,
                "launches_per_step": k["launches"] / args.steps, "big_launches_per_step": k["big_launches"] / args.steps,
                "avg_big_launch_ms": k["big_ms"] / max(k["big_launches"], 1),
                "algorithmic_bytes_per_big_launch": k["big_bytes"] / max(k["big_launches"], 1)}
    table = sorted((entry(n, k) for n, k in ksum.items()), key=lambda e: -e["ms_per_step"])
    roofline = None
    if table:
        roofline = dict(table[0])
        roofline["peak_source"] = peak_src
        roofline["note"] = ("dominant kernel by total time in the step; achieved = algorithmic bytes (DESIGN.md section 4) of its "
                            "L(g)-sized launches / CUDA-event time on the launching stream")
        roofline["extra"] = table[1:8]
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "norm": args.norm, "global_batch": graphs_per_step, "per_gpu_batch": args.batch,
                   "parallelism": f"dp{world}", "optimizer": "AdamW", "loss": "L1",
                   "l2": f"no explicit flush: per-step working set ~{sbytes / 1e9:.1f} GB >> 126 MB L2; 4 batches rotate"},
        "run": {"device": "B200", "N": N, "E": E, "T": T,
                "optimizer_impl": "one launch over one flat parameter (alignn_b200.dp.FlatAdamW -> alignn_b200_adamw_flat)",
                "cuda_graph": use_graph, "allreduce_in_graph": bool(nccl_in_graph), "eager_ms_per_step": ms_eager / args.steps,
                "timing": f"exactly {args.steps} steps between two events on the launching stream, barrier + synchronize "
                          f"on both sides, max over ranks"},
        "roofline": roofline,
        "step_hbm": {"algorithmic_bytes_per_step": sbytes, "achieved": sbytes / (ms_step * 1e-3) / 1e9, "peak": peak,
                     "unit": "GB/s", "frac": sbytes / (ms_step * 1e-3) / 1e9 / peak,
                     "note": "conv-stack compulsory bytes per batch (SURVEY 8d) / whole step time incl. embeddings, GEMMs, optimizer"},
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": 4,
                "how": ("every step: inputs pinned host -> device (copy stream, issued one step ahead so it overlaps the previous step's "
                        "kernels; the first step of a region copies its own inputs serially), CUDA-graph replay, loss device -> pinned "
                        "host, read by the host one step later") if use_graph else
                       "every step: inputs pinned host -> device on the compute stream, eager step, loss.item()"},
        "gpu_launches": int(lt.item()),
        "clocks": clocks,
    }
    if world == 1 and not args.no_cpu_baseline:
        # bounded sample of the same workload on the host cores: the full 64-graph step, fixed thread count
        threads = min(32, os.cpu_count() or 1)
        gps, ms = cpu_oracle_run(args, args.batch if args.cpu_sample_graphs <= 0 else args.cpu_sample_graphs, 2, 1, threads)
        line["cpu_baseline"] = {"value": gps, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"2 steps x {args.batch if args.cpu_sample_graphs <= 0 else args.cpu_sample_graphs} graphs "
                                          f"(fwd+bwd+AdamW) after 1 warm-up, torch-CPU restatement of the reference DGL path, "
                                          f"{threads} threads of the box's {os.cpu_count()} cores"}
    print(json.dumps(line), flush=True)
    if world > 1:
        _finish(nccl_in_graph)


def _finish(hard_exit):
    """Tear the process group down; after replayed in-graph collectives the NCCL teardown hangs on this stack, so that
    mode leaves through os._exit once everything is printed."""
    sys.stdout.flush()
    if hard_exit:
        os._exit(0)
    dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
