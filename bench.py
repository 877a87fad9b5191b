#!/usr/bin/env python
"""Headline benchmark: sampled-subgraph train steps/sec for 2-layer GraphSAGE
(fan-out 25,10) on an ogbn-products-shaped synthetic graph (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W          # our engine
    python bench.py --impl reference --gpus N ...          # unmodified reference (baseline/_ref)

One JSON line is printed by rank 0.  `value` is the whole-job steps/sec summed
over all N GPUs (each rank trains its own 1024-seed batch per step: weak
scaling), device-timed with CUDA events, max over ranks.
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

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

PRODUCTS = dict(num_nodes=2_449_029, num_edges=123_718_280, feat_dim=100, num_classes=47)
FANOUTS = [25, 10]
HIDDEN = 256
BATCH = 1024
# BASELINE.json configs.  `products_sage2` is the headline the driver runs; the others are selected with --config.
CONFIGS = {
    "products_sage2": dict(shape=PRODUCTS, fanouts=[25, 10], hidden=256,
                           metric="sampled-subgraph train steps/sec (2-layer GraphSAGE fanout 25,10, ogbn-products-shaped synthetic)",
                           model="GraphSAGE-2layer-mean hidden256",
                           data="synthetic (random graph of ogbn-products shape, random-init weights)"),
    # ogbn-papers100M is 111M nodes / 1.6B edges / 128-d / 172 classes; the reference arm has to write and parse the
    # graph as TSV text, so both arms use the same 1/32-scale graph of that shape (same degree, dims, fan-outs)
    "sage3": dict(shape=dict(num_nodes=3_468_000, num_edges=50_500_000, feat_dim=128, num_classes=172), fanouts=[15, 10, 5],
                  hidden=256,
                  metric="sampled-subgraph train steps/sec (3-layer GraphSAGE fanout 15,10,5, ogbn-papers100M-shaped synthetic at 1/32 scale)",
                  model="GraphSAGE-3layer-mean hidden256",
                  data="synthetic (random graph of ogbn-papers100M shape at 1/32 scale: 3.47M nodes / 50.5M edges / 128-d, random-init weights)"),
    "deepwalk": dict(shape=dict(num_nodes=3_468_000, num_edges=50_500_000, feat_dim=0, num_classes=2), walk_len=40, neg=5,
                     metric="DeepWalk random walks/sec (random_walk length 40 + 5 random negatives per walk, ogbn-papers100M-shaped synthetic at 1/32 scale)",
                     model="DeepWalk walk engine (sampling only)",
                     data="synthetic (random graph of ogbn-papers100M shape at 1/32 scale: 3.47M nodes / 50.5M edges)"),
    # Taobao-shaped user-item graph (BASELINE config 4: 50M users / 100M items / 1B edges) at 1/32 scale for the same
    # reason as above; 2-layer 4-head GAT towers, weighted (edge_weight) neighbour sampling, in-batch + in-degree-weighted
    # sampled negatives
    "taobao_gat": dict(shape=dict(num_users=1_562_500, num_items=3_125_000, num_edges=31_250_000, feat_dim=64), fanouts=[10, 5],
                       hidden=128, heads=4, neg=5,
                       metric="train steps/sec (2-layer 4-head bipartite GAT, weighted + in-batch negative sampling, Taobao-shaped synthetic at 1/32 scale)",
                       model="EgoBipartite GAT 2-layer 4-head hidden128 (user / item towers)",
                       data="synthetic (random bipartite graph of Taobao shape at 1/32 scale: 1.56M users / 3.1M items / 31M weighted edges, random-init weights)"),
}


class ClockSampler:
    """Samples SM clocks / throttle reasons DURING the timed region (NVML in a thread, 20 ms period;
    falls back to polling nvidia-smi)."""

    def __init__(self, index=0, period=0.02):
        self.index, self.period = index, period
        self.sm, self.mx, self.reasons = [], [], set()
        self._stop = threading.Event()
        self._th = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self._nvml = None

    def _run_nvml(self):
        n = self._nvml
        bits = {"hw_slowdown": getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self._stop.is_set():
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)))
                self.mx.append(float(n.nvmlDeviceGetMaxClockInfo(self._h, n.NVML_CLOCK_SM)))
                r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for name, b in bits.items():
                    if r & b:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.sm.append(float(parts[0])); self.mx.append(float(parts[1]))
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[3:7]):
                        if v.lower().startswith("active"):
                            self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._th = threading.Thread(target=self._run_nvml if self._nvml else self._run_smi, daemon=True)
        self._th.start()

    def stop(self):
        self._stop.set()
        if self._th:
            self._th.join(timeout=6)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "source": "nvml" if self._nvml else "nvidia-smi"}


DUMP_BYTES = 64 << 20


def dump_outputs(d, arrays):
    """Write each array as ``d/<name>.npy`` (floats as float32 / float64, integer ids as float64, exact below 2**53) so that
    two builds can be compared output for output.  An array larger than its share of DUMP_BYTES is replaced by a fixed,
    seeded sample of its elements (same indices for the same shape)."""
    import numpy as np
    import torch
    os.makedirs(d, exist_ok=True)
    share = DUMP_BYTES // max(len(arrays), 1)
    for name, t in arrays.items():
        t = torch.as_tensor(t).detach()
        a = t.double() if (not t.is_floating_point() or t.dtype == torch.float64) else t.float()
        a = a.cpu().numpy()
        if a.nbytes > share:
            idx = np.sort(np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(d, name + ".npy"), a)


def count_own_launches(trainer):
    """Kernel launches of one step, split into ours (namespace glb::) and library kernels."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    trainer_graph, trainer.graph = trainer.graph, None         # eager step so every launch is visible
    try:
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            trainer._step_body()
            torch.cuda.synchronize()
        if trainer.rt.world > 1:
            trainer.rt.barrier()                                # outside the profile: NCCL's barrier kernels are not the step's
        own, lib = 0, 0
        names = {}
        times = {}
        for ev in prof.events():
            if ev.device_type is not None and str(ev.device_type).endswith("CUDA") and ev.name and \
                    not ev.name.startswith("Memcpy") and not ev.name.startswith("Memset"):
                key = ev.name.split("(")[0][:60]
                t = getattr(ev, "device_time", None)
                if t is None:
                    t = getattr(ev, "cuda_time", 0.0)
                times[key] = round(times.get(key, 0.0) + float(t), 1)
                if "glb::" in ev.name:
                    own += 1
                    names[key] = names.get(key, 0) + 1
                else:
                    lib += 1
        trainer._kernel_us = times
        return own, lib, names
    finally:
        trainer.graph = trainer_graph


def build_trainer(args, rt, shape, feature_dtype, cache_rows_arg):
    FANOUTS, HIDDEN = args.cfg["fanouts"], args.cfg["hidden"]
    """Public-API path: in-memory sources -> gl.Graph -> GSL query -> compiled plan -> fused engine.
    (--api raw keeps the round-1 path that hands raw shards to the trainer, for A/B.)"""
    import torch
    import torch.distributed as dist

    import graphlearn_b200 as gl
    from graphlearn_b200.engine.fast_sage import FastSageTrainer
    from graphlearn_b200.engine.trainer import SageTrainer
    from graphlearn_b200.models.graphsage import EgoGraphSAGE
    from graphlearn_b200.store.synthetic import make_partitioned_sources, make_sharded_graph

    W = rt.world
    t0 = time.time()
    gl.set_feature_dtype(feature_dtype)
    g = q = None
    if args.api == "gsl":
        node_src, edge_src = make_partitioned_sources(rt, seed=0, **shape)
        g = gl.Graph()
        g.node(node_src, "n", decoder=gl.Decoder(labeled=True, attr_types=["float"] * shape["feat_dim"]))
        g.edge(edge_src, ("n", "n", "e"), decoder=gl.Decoder())
        g.init()
        del node_src, edge_src
        nodes, csr = g.store.nodes["n"], g.store.edges["e"]
        q = g.V("n").batch(args.batch).shuffle(traverse=True).alias("src")
        for i, k in enumerate(FANOUTS):
            q = q.outV("e").sample(k).by("random").alias("h%d" % (i + 1))
        q = q.values()
    else:
        fdt = {"bf16": torch.bfloat16, "fp8": torch.float8_e4m3fn}.get(feature_dtype, torch.float32)
        nodes, csr = make_sharded_graph(rt, feature_dtype=fdt, seed=0, **shape)
    # N17 replica cache of remote feature rows in local HBM (the reference's set_local_node_cache_capacity, default 0 =
    # off there and here): -1 = as many remote rows as fit in 25% of the free HBM
    cache_rows = 0
    if W > 1 and cache_rows_arg != 0:
        cap = cache_rows_arg
        if cap < 0:
            free_b, _ = torch.cuda.mem_get_info()
            cap = int(0.25 * free_b) // (nodes.feats.local.size(1) * nodes.feats.local.element_size())
        scores = None
        if cap < shape["num_nodes"]:
            max_vid = max(int(n) for n in nodes.nrows) * W
            scores = torch.bincount(csr.indices.local.clamp(min=0), minlength=max_vid).float()[:max_vid]
            dist.all_reduce(scores)
        cache_rows = nodes.build_feature_cache(cap, scores=scores)
    torch.cuda.synchronize()
    build_s = time.time() - t0
    torch.manual_seed(0)
    model = EgoGraphSAGE(shape["feat_dim"], HIDDEN, shape["num_classes"], len(FANOUTS)).to(rt.device)
    if args.engine == "autograd":
        tr = SageTrainer(rt, nodes, csr, model, FANOUTS, args.batch, lr=3e-3, allreduce=args.allreduce,
                         use_cuda_graph=not args.no_graph)
    elif q is not None:
        tr = FastSageTrainer.from_query(g, q, model, lr=3e-3, allreduce=args.allreduce, use_cuda_graph=not args.no_graph)
    else:
        tr = FastSageTrainer(rt, nodes, csr, model, FANOUTS, args.batch, lr=3e-3, allreduce=args.allreduce,
                             use_cuda_graph=not args.no_graph)
    return tr, nodes, csr, cache_rows, build_s, g


def time_trainer(args, rt, tr, nodes, steps, clocks=None, dump_dir=None):
    """(device-timed ms, e2e ms, last loss).  Device region: K graph replays, every one samples a FRESH seed batch
    (already resident on the device).  End-to-end region: the public step - host seeds (GSL traversal when built
    from a query) -> pinned staging -> H2D inside the step graph, loss -> pinned host every step."""
    import torch
    import torch.distributed as dist
    W = rt.world
    gen = torch.Generator().manual_seed(1234 + rt.rank)
    n_local = nodes.n_local
    warm = max(args.warmup, 3)
    total = warm + 2 * steps + 8
    seed_ids = (torch.randint(0, n_local, (total, args.batch), generator=gen) * W + rt.rank)
    dev_seeds = seed_ids.to(rt.device)
    seed_ids = seed_ids.pin_memory()
    use_query = hasattr(tr, "step_query")
    tr.seeds.copy_(seed_ids[0])
    tr.capture()
    it = 0
    for _ in range(warm):
        tr.step(seed_ids[it]); it += 1
    for _ in range(2):
        tr.step_device(dev_seeds[it]); it += 1
    torch.cuda.synchronize()
    rt.barrier()
    if clocks:
        clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rt.barrier(); torch.cuda.synchronize()
    ev0.record()
    for _ in range(steps):
        tr.step_device(dev_seeds[it]); it += 1
    ev1.record()
    torch.cuda.synchronize(); rt.barrier()
    ms_dev = ev0.elapsed_time(ev1)
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    import graphlearn_b200 as gl
    rt.barrier(); torch.cuda.synchronize()
    ev2.record()
    last = None
    done = 0
    while done < steps:
        if use_query:
            try:
                last = tr.step_query()
            except gl.OutOfRangeError:      # epoch boundary of the GSL traversal: the next call starts a new pass
                continue
        else:
            last = tr.step(seed_ids[it]); it += 1
        done += 1
    ev3.record()
    torch.cuda.synchronize(); rt.barrier()
    ms_e2e = ev2.elapsed_time(ev3)
    final_loss = float(last)
    if hasattr(tr, "ar"):
        tr.ar.check()
    if dump_dir and rt.rank == 0:
        # the last step's loss as the caller received it, the logits of that step's seed batch, the updated weights
        outs = {"loss": last}
        if hasattr(tr, "H"):
            outs["logits"] = tr.H[-1]
        outs.update(("param." + n, p) for n, p in tr.model.named_parameters())
        dump_outputs(dump_dir, outs)
    t = torch.tensor([ms_dev, ms_e2e], device=rt.device, dtype=torch.float64)
    if W > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0]), float(t[1]), final_loss


def run_ours(args):
    import torch

    from graphlearn_b200.parallel.runtime import init

    rt = init()
    assert rt.is_cuda, "bench.py needs a CUDA device"
    W = rt.world
    if "walk_len" in args.cfg:
        return run_walks(args, rt)
    if "heads" in args.cfg:
        return run_bipartite_gat(args, rt)
    FANOUTS = args.cfg["fanouts"]
    shape = dict(args.cfg["shape"])
    if args.small:
        shape = dict(num_nodes=200_000, num_edges=5_000_000, feat_dim=100, num_classes=47)
    # ---- headline: hash-partitioned graph, NO replica cache: every remote row crosses NVLink inside the fused kernel
    tr, nodes, csr, cache_rows, build_s, g = build_trainer(args, rt, shape, args.feature_dtype, args.feature_cache_rows)
    clocks = ClockSampler(rt.local_rank) if rt.rank == 0 else None
    ms_dev, ms_e2e, final_loss = time_trainer(args, rt, tr, nodes, args.steps, clocks, args.dump_outputs)
    clk = clocks.stop() if clocks else None
    own, lib, names = count_own_launches(tr)
    # payload bytes of a feature row (the 128-byte aligned stride adds padding that is never read)
    row_bytes = (nodes.float_dim + 2 * ((nodes.float_dim + 31) // 32)) if nodes.feats.local.dtype == torch.uint8 \
        else nodes.float_dim * nodes.feats.local.element_size()
    rows_per_step, m_ = 0, args.batch
    for k_ in FANOUTS:                      # layer 1 gathers (1 + k_i) rows per destination of every hop pair
        rows_per_step += m_ * (1 + k_)
        m_ *= k_
    n_total = sum(int(x) for x in nodes.nrows)
    remote_frac = 0.0 if W == 1 else (W - 1) / W * max(0.0, 1.0 - cache_rows / max(n_total - nodes.n_local, 1))
    remote_bytes = rows_per_step * row_bytes * remote_frac
    kernel_us = getattr(tr, "_kernel_us", {})
    extra = {}
    # ---- secondary measurements (clearly labelled; never the headline)
    sec_steps = min(args.steps, 300)
    if W > 1 and args.feature_cache_rows == 0 and not args.no_secondary:
        del tr
        torch.cuda.empty_cache()
        tr2, nodes2, _, cr2, _, _ = build_trainer(args, rt, shape, args.feature_dtype, -1)
        d2, e2, _ = time_trainer(args, rt, tr2, nodes2, sec_steps)
        extra["replica_cache_run"] = {"what": "same job with the N17 replica cache of remote feature rows filled (reference: "
                                      "set_local_node_cache_capacity); remote feature traffic = 0", "feature_cache_rows_per_gpu": cr2,
                                      "value": W * sec_steps / (d2 / 1e3), "e2e_value": W * sec_steps / (e2 / 1e3), "unit": "steps/s",
                                      "steps": sec_steps}
        del tr2, nodes2
    elif W == 1 and not args.no_secondary:
        del tr
        torch.cuda.empty_cache()
        for other in [o for o in ("fp32", "bf16", "fp8") if o != args.feature_dtype]:
            what = ("same job with %s feature rows in HBM (compute stays bf16)" % other) if other != "fp8" else \
                "same job with fp8 (e4m3, one bf16 scale per 32 elements) feature rows - storage precision BELOW the reference's: " \
                "capacity / bandwidth data point, never the headline"
            tr2, nodes2, _, _, _, _ = build_trainer(args, rt, shape, other, 0)
            d2, e2, _ = time_trainer(args, rt, tr2, nodes2, sec_steps)
            extra["%s_feature_rows_run" % other] = {"what": what, "value": sec_steps / (d2 / 1e3), "e2e_value": sec_steps / (e2 / 1e3),
                                                    "unit": "steps/s", "steps": sec_steps}
            del tr2, nodes2
            torch.cuda.empty_cache()
    if rt.rank == 0:
        steps_per_s = W * args.steps / (ms_dev / 1e3)
        e2e_steps_per_s = W * args.steps / (ms_e2e / 1e3)
        fbytes = {"bf16": 2, "fp8": 1}.get(args.feature_dtype, 4)
        out = {
            "metric": args.cfg["metric"],
            "value": steps_per_s, "unit": "steps/s", "n_gpus": W, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": args.cfg["data"],
            "impl": "graphlearn_b200",
            "config": {"name": args.config, "model": args.cfg["model"], "global_batch": args.batch * W, "seq_len": None,
                       "fanout": FANOUTS, "parallelism": "dp%d+graph-partition%d" % (W, W),
                       "api": "gsl (in-memory sources -> gl.Graph -> GSL query -> compiled plan -> fused engine)" if args.api == "gsl"
                              else "raw shards",
                       "num_nodes": shape["num_nodes"], "num_edges": shape["num_edges"],
                       "feat_dim": shape["feat_dim"], "feature_storage": args.feature_dtype,
                       "feature_cache_rows_per_gpu": cache_rows,
                       "feature_cache": ("n/a (single GPU)" if W == 1 else
                                         "none: the graph is hash-partitioned, every remote row is read from its owner's HBM over NVLink "
                                         "inside the fused kernel" if cache_rows == 0 else
                                         "replica cache of remote feature rows in local HBM (reference: set_local_node_cache_capacity)"),
                       "remote_feature_bytes_per_step_per_gpu": int(remote_bytes),
                       "remote_feature_GBps_per_gpu": round(remote_bytes / (ms_dev / args.steps * 1e-3) / 1e9, 1),
                       "nvlink_peer_copy_GBps_measured": 770,
                       "seeds": "fresh seed batch every step in both timed regions (device region: resident on the device; "
                                "e2e region: GSL shuffle(traverse=True) epochs on the host)",
                       "l2_policy": "inputs larger than L2: every step gathers ~%d random feature rows from a %.1f GB table"
                                    % (rows_per_step, shape["num_nodes"] * shape["feat_dim"] * fbytes / 1e9),
                       "allreduce": tr_backend(W, args), "cuda_graph": not args.no_graph, "engine": args.engine,
                       "graph_build_s": round(build_s, 2)},
            "e2e": {"value": e2e_steps_per_s, "unit": "steps/s", "h2d_bytes_per_step": args.batch * 8,
                    "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": own * args.steps, "own_kernels_per_step": own, "library_kernels_per_step": lib,
            "own_kernel_names": names, "kernel_us_eager_step": kernel_us, "clocks": clk, "final_loss": final_loss,
        }
        out.update(extra)
        print(json.dumps(out))
    rt.barrier()
    rt.shutdown()


def run_walks(args, rt):
    """BASELINE config 5: DeepWalk random_walk(length 40) + random negatives.  Device region: the resident-walker kernel
    (K3) + the negative sampler kernel (K2) per step on fresh seeds; e2e region: the same through gl.Graph + GSL +
    gl.Dataset (``V().batch().shuffle().random_walk().outNeg()``) including the D2H read of the walks."""
    import torch
    import torch.distributed as dist

    import graphlearn_b200 as gl
    from graphlearn_b200.ops import negative as NEG
    from graphlearn_b200.ops import rng as rng_ops
    from graphlearn_b200.ops import walk as WALK
    from graphlearn_b200.store.synthetic import make_partitioned_sources
    W, cfg = rt.world, args.cfg
    shape = dict(cfg["shape"])
    if args.small:
        shape.update(num_nodes=200_000, num_edges=5_000_000)
    L, NEGS, B = cfg["walk_len"], cfg["neg"], args.batch
    t0 = time.time()
    node_src, edge_src = make_partitioned_sources(rt, seed=0, feat_dim=1, num_classes=2,
                                                  num_nodes=shape["num_nodes"], num_edges=shape["num_edges"])
    node_src.pop("float_attrs"); node_src.pop("labels")
    g = gl.Graph()
    g.node(node_src, "n", decoder=gl.Decoder())
    g.edge(edge_src, ("n", "n", "e"), decoder=gl.Decoder())
    g.init()
    del node_src, edge_src
    torch.cuda.synchronize()
    build_s = time.time() - t0
    store = g.store
    csr, nodes = store.edges["e"], store.nodes["n"]
    rng = rng_ops.DeviceRng(rt, 0)
    gen = torch.Generator().manual_seed(99 + rt.rank)
    warm = max(args.warmup, 3)
    seeds = (torch.randint(0, nodes.n_local, (warm + args.steps + 4, B), generator=gen) * W + rt.rank).to(rt.device)

    def one(i):
        walks = WALK.random_walk(csr, seeds[i], L, 1.0, 1.0, rng=rng, salt=i)
        neg = NEG.edge_negative(store, "e", walks.reshape(-1), NEGS, "random", None, rng=rng, salt=1000 + i)
        rng.advance()
        return walks, neg
    for i in range(warm):
        one(i)
    torch.cuda.synchronize(); rt.barrier()
    clocks = ClockSampler(rt.local_rank) if rt.rank == 0 else None
    if clocks:
        clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(args.steps):
        walks, neg = one(warm + i)
    ev1.record()
    torch.cuda.synchronize(); rt.barrier()
    ms_dev = ev0.elapsed_time(ev1)
    if args.dump_outputs and rt.rank == 0:
        dump_outputs(args.dump_outputs, {"walks": walks, "neg": neg})
    # e2e through the public API
    q = g.V("n").batch(B).shuffle(traverse=True).alias("src").random_walk("e", L).alias("walk") \
         .outNeg("e").sample(NEGS).by("random").alias("neg").values()
    ds = gl.Dataset(q, window=4)
    for _ in range(warm):
        ds.next()["walk"].ids
    torch.cuda.synchronize(); rt.barrier()
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev2.record()
    done, d2h = 0, 0
    while done < args.steps:
        try:
            v = ds.next()
        except gl.OutOfRangeError:
            continue
        w_ids, n_ids = v["walk"].ids, v["neg"].ids          # numpy: device -> host read of the step's result
        d2h = w_ids.nbytes + n_ids.nbytes
        done += 1
    ev3.record()
    torch.cuda.synchronize(); rt.barrier()
    ms_e2e = ev2.elapsed_time(ev3)
    clk = clocks.stop() if clocks else None
    t = torch.tensor([ms_dev, ms_e2e], device=rt.device, dtype=torch.float64)
    if W > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = float(t[0]), float(t[1])
    if rt.rank == 0:
        walks_s = W * B * args.steps / (ms_dev / 1e3)
        hops_s = walks_s * L
        print(json.dumps({
            "metric": cfg["metric"], "value": walks_s, "unit": "walks/s", "n_gpus": W, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64 ids",
            "data": cfg["data"], "impl": "graphlearn_b200",
            "config": {"name": args.config, "model": cfg["model"], "global_batch": B * W, "walk_len": L, "negatives_per_position": NEGS,
                       "num_nodes": shape["num_nodes"], "num_edges": shape["num_edges"], "parallelism": "graph-partition%d" % W,
                       "walk_hops_per_s": hops_s,
                       "remote_adjacency_reads_per_s_per_gpu": round(hops_s / W * (W - 1) / W * 3) if W > 1 else 0,
                       "l2_policy": "inputs larger than L2: random rows of a %.1f GB CSR" % (shape["num_edges"] * 8 / 1e9),
                       "graph_build_s": round(build_s, 2)},
            "e2e": {"value": W * B * args.steps / (ms_e2e / 1e3), "unit": "walks/s", "h2d_bytes_per_step": B * 8,
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": 3 * args.steps, "own_kernel_names": {"glb::random_walk_kernel": 1, "glb::negative_sample_kernel": 1,
                                                                 "glb::step_advance_kernel": 1}, "clocks": clk}))
    rt.barrier()
    rt.shutdown()


def run_bipartite_gat(args, rt):
    """BASELINE config 4 through the public API: gl.Graph (in-memory sources) -> GSL edge-rooted query with weighted
    neighbour sampling and in-degree-weighted negatives -> EgoBipartiteSAGE(conv="gat") whose first layer gathers inside
    the fused attention kernel (csrc/gat.cu) -> in-batch softmax + sampled-negative loss -> Adam.  Every step reads the
    loss back to the host; the timed region is the whole loop (sampling + training), device timed."""
    import torch
    import torch.distributed as dist

    import graphlearn_b200 as gl
    from graphlearn_b200 import models
    W, cfg = rt.world, args.cfg
    sh = dict(cfg["shape"])
    if args.small:
        sh.update(num_users=50_000, num_items=100_000, num_edges=1_000_000)
    NU, NI, NE, D = sh["num_users"], sh["num_items"], sh["num_edges"], sh["feat_dim"]
    K1, K2 = cfg["fanouts"]
    B, NEG = args.batch, cfg["neg"]
    dev = rt.device
    t0 = time.time()
    gen = torch.Generator(device=dev).manual_seed(7)                # same data on every rank: init() keeps what it owns
    src = torch.randint(0, NU, (NE,), device=dev, generator=gen)
    pop = torch.exp(torch.randn(NI, device=dev, generator=gen))       # skewed item popularity
    dst = torch.multinomial(pop, NE, replacement=True, generator=gen)
    wts = torch.rand(NE, device=dev, generator=gen) + 0.05
    gl.set_feature_dtype(args.feature_dtype)
    g = gl.Graph()
    g.node({"ids": torch.arange(NU, device=dev), "float_attrs": torch.randn(NU, D, device=dev, generator=gen)}, "u",
           decoder=gl.Decoder(attr_types=["float"] * D))
    g.node({"ids": torch.arange(NI, device=dev), "float_attrs": torch.randn(NI, D, device=dev, generator=gen)}, "i",
           decoder=gl.Decoder(attr_types=["float"] * D))
    g.edge({"src_ids": src, "dst_ids": dst, "weights": wts}, ("u", "i", "u2i"), decoder=gl.Decoder(weighted=True), directed=False)
    g.init()
    del src, dst, wts, pop
    torch.cuda.synchronize()
    build_s = time.time() - t0
    q = g.E("u2i").batch(B).shuffle(traverse=True).alias("e").each(lambda e: (
        e.outV().alias("u").each(lambda u: (
            u.outV("u2i").sample(K1).by("edge_weight").alias("u1").outV("u2i_reverse").sample(K2).by("random").alias("u2"),
            u.outNeg("u2i").sample(NEG).by("in_degree").alias("neg").outV("u2i_reverse").sample(K1).by("random").alias("n1")
             .outV("u2i").sample(K2).by("edge_weight").alias("n2"))),
        e.inV().alias("i").outV("u2i_reverse").sample(K1).by("random").alias("i1")
         .outV("u2i").sample(K2).by("edge_weight").alias("i2"))).values()
    ds = gl.Dataset(q, window=4)
    torch.manual_seed(0)
    model = models.EgoBipartiteSAGE(D, D, cfg["hidden"], cfg["hidden"], hops=2, conv="gat", num_head=cfg["heads"]).to(dev)
    if W > 1:
        for p_ in model.parameters():
            dist.broadcast(p_.data, src=0)
    use_graph = not args.no_graph and W == 1
    opt = torch.optim.Adam(model.parameters(), lr=3e-3, fused=True, capturable=use_graph)
    tu, ti = g.store.nodes["u"], g.store.nodes["i"]
    h_loss = torch.zeros(1).pin_memory()
    names = ("u", "u1", "u2", "i", "i1", "i2", "neg", "n1", "n2")

    def next_batch():
        while True:
            try:
                r = ds.next()
                return {a: r[a].vids_t for a in names}
            except gl.OutOfRangeError:
                continue

    def loss_fn(v):
        ue, ie = model.forward_store([tu, ti, tu], [v["u"], v["u1"], v["u2"]], [ti, tu, ti], [v["i"], v["i1"], v["i2"]], [K1, K2], [K1, K2])
        ne = model.item_tower.forward_store([ti, tu, ti], [v["neg"], v["n1"], v["n2"]], [K1, K2])
        return model.in_batch_negative_loss(ue, ie) + model.loss(ue, ie, ne, kind="sigmoid")

    def allreduce_grads():
        flat = torch.cat([p_.grad.reshape(-1) for p_ in model.parameters()])
        dist.all_reduce(flat)
        flat /= W
        o = 0
        for p_ in model.parameters():
            p_.grad.copy_(flat[o:o + p_.numel()].view_as(p_)); o += p_.numel()

    graphed = None
    if use_graph:
        # forward + loss + backward + Adam of the two towers as ONE CUDA graph over static id buffers (engine/graphed.py)
        from graphlearn_b200.engine.graphed import GraphedTrainStep
        try:
            graphed = GraphedTrainStep(loss_fn, opt, next_batch())
        except Exception as e:      # a non-capturable op in the model path: keep the eager step, say so in the JSON line
            print("graph capture of the GAT step failed, running eagerly: %r" % (e,), file=sys.stderr)
            graphed = None
            opt = torch.optim.Adam(model.parameters(), lr=3e-3, fused=True)

    def step():
        v = next_batch()
        if graphed is not None:
            loss = graphed(v)
        else:
            loss = loss_fn(v)
            opt.zero_grad(set_to_none=True)
            loss.backward()
            if W > 1:
                allreduce_grads()
            opt.step()
            loss = loss.detach()
        h_loss.copy_(loss, non_blocking=True)
        return h_loss
    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    torch.cuda.synchronize(); rt.barrier()
    clocks = ClockSampler(rt.local_rank) if rt.rank == 0 else None
    if clocks:
        clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        last = step()
    ev1.record()
    torch.cuda.synchronize(); rt.barrier()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rt.rank == 0:
        outs = {"loss": last}
        outs.update(("param." + n, p) for n, p in model.named_parameters())
        dump_outputs(args.dump_outputs, outs)
    clk = clocks.stop() if clocks else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if W > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    if rt.rank == 0:
        v_ = W * args.steps / (ms / 1e3)
        print(json.dumps({
            "metric": cfg["metric"], "value": v_, "unit": "steps/s", "n_gpus": W, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16 rows / fp32 math",
            "data": cfg["data"], "impl": "graphlearn_b200",
            "config": {"name": args.config, "model": cfg["model"], "global_batch": B * W, "fanout": cfg["fanouts"], "heads": cfg["heads"],
                       "negatives": "in-batch softmax + %d in-degree-weighted sampled negatives per user (item tower applied to them)" % NEG,
                       "api": "gsl (in-memory sources -> gl.Graph -> GSL E() query -> interpreter -> fused GAT kernels + autograd)",
                       "cuda_graph": ("model step (forward + loss + backward + Adam) captured as one CUDA graph, %d replays / %d eager"
                                      % (graphed.replays, graphed.eager_steps)) if graphed is not None else "no (eager autograd)",
                       "num_users": NU, "num_items": NI, "num_edges": NE, "feat_dim": D, "parallelism": "dp%d+graph-partition%d" % (W, W),
                       "graph_build_s": round(build_s, 2)},
            "e2e": {"value": v_, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 4,
                    "note": "the timed loop IS the public path (Dataset.next() + model + optimiser + loss read-back); the edge-rooted "
                            "traversal draws its seeds on the device"},
            "clocks": clk, "final_loss": float(last)}))
    rt.barrier()
    rt.shutdown()


def tr_backend(W, args):
    return "none" if W == 1 else ("peer" if args.allreduce == "peer" else "nccl")


def run_reference(args):
    try:
        from baseline import run_reference as rr
    except Exception as e:  # pragma: no cover
        print(json.dumps({"impl": "reference", "unavailable": "baseline runner import failed: %r" % (e,)}))
        return
    rr.main(args)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="products_sage2", choices=sorted(CONFIGS),
                    help="BASELINE.json config: products_sage2 (headline, default) | sage3 | deepwalk | taobao_gat")
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--feature-dtype", default="bf16", choices=["fp32", "bf16", "fp8"],
                    help="HBM storage dtype of the float attribute table (compute is bf16 either way; bf16 halves NVLink bytes)")
    ap.add_argument("--allreduce", default="peer", choices=["peer", "nccl"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--engine", default="fast", choices=["fast", "autograd"],
                    help="fast = hand-scheduled fwd/bwd kernel chain; autograd = torch.autograd over the same kernels")
    ap.add_argument("--feature-cache-rows", type=int, default=0,
                    help="remote feature rows replicated per GPU (N17 cache): 0 off (default, = the reference's default), "
                         "-1 auto (25%% of free HBM)")
    ap.add_argument("--api", default="gsl", choices=["gsl", "raw"],
                    help="gsl = in-memory sources -> gl.Graph -> GSL query -> compiled plan -> engine; raw = shards handed to the trainer")
    ap.add_argument("--no-secondary", action="store_true", help="skip the labelled secondary run (replica cache / other row dtype)")
    ap.add_argument("--small", action="store_true", help="small graph for quick functional runs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step returned (loss, logits, updated weights; walks and "
                         "negatives for deepwalk) as DIR/<name>.npy; the inputs are seeded, so two builds compare file for file. "
                         "Float atomics (loss, bias gradients) round in a run-dependent order and Adam amplifies that over the "
                         "steps: compare trained outputs with a tolerance, or with few --steps")
    args = ap.parse_args()
    args.cfg = CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
