"""Headline benchmark: epochs/s of full-graph partitioned GraphSAGE training (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the CPU path (oracle port of the reference) on the host cores

Default workload (BASELINE.json configs[1]): synthetic RMAT 1 M nodes / 20 M edges, one partition per GPU
(random partition), 3-layer GraphSAGE, hidden 256, bf16 activations, --enable-pipeline.  A step is one
epoch: forward, loss, backward (with the gradient halo exchange), gradient all-reduce, Adam step.

Order of a run: set-up -> (N > 1) parity of the real multi-GPU path against the CPU oracle -> warm-up -> a short
Python-launched region instrumented with CUDA events (roofline of the aggregate kernel) -> the timed region: K epochs
replayed from CUDA graphs (`--no-graph`: launched from Python), exposed communication accumulated ON THE DEVICE by the
flag-wait kernel inside that region -> (--dump-outputs) the last timed epoch's outputs -> the end-to-end region (host
buffers, H2D + D2H per step) -> (N = 1) the CPU baseline -> ONE JSON line from rank 0.  The process returns normally
(no os._exit).
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[1]
    "rmat-1m": dict(shape="rmat-1m", n_layers=3, n_hidden=256, dtype="bf16", enable_pipeline=True,
                    feat_corr=False, grad_corr=False,
                    desc="RMAT 1M nodes / 20M edges, F=256, C=64, 3-layer GraphSAGE hidden 256, bf16, --enable-pipeline"),
    # configs[2] (layers as scripts/reddit.sh:8)
    "reddit-shaped": dict(shape="reddit-shaped", n_layers=4, n_hidden=256, dtype="fp32", enable_pipeline=True,
                          feat_corr=True, grad_corr=True,
                          desc="Reddit-shaped RMAT 233K nodes / 115M edges, F=602, C=41, 4-layer GraphSAGE hidden 256, "
                               "fp32, --enable-pipeline --feat-corr --grad-corr"),
    # configs[3]: no pipeline -> the exchange is waited for in the epoch that needs it
    "products-shaped": dict(shape="products-shaped", n_layers=3, n_hidden=128, dtype="fp32", enable_pipeline=False,
                            feat_corr=False, grad_corr=False,
                            desc="ogbn-products-shaped RMAT 2.4M nodes / 62M edges, F=100, C=47, 3-layer GraphSAGE "
                                 "hidden 128, fp32, no pipeline"),
    # configs[4]: per-rank graph construction (no rank holds the global edge list), see pipegcn_b200/distgraph.py
    "papers100m-shaped": dict(shape="papers100m-shaped", n_layers=3, n_hidden=128, dtype="bf16", enable_pipeline=True,
                              feat_corr=False, grad_corr=False, distributed_build=True,
                              desc="ogbn-papers100M-shaped RMAT 111M nodes / 1.6B edges, F=128, C=172, 3-layer GraphSAGE "
                                   "hidden 128, bf16, --enable-pipeline, per-rank graph construction"),
    "small": dict(shape="small", n_layers=3, n_hidden=64, dtype="bf16", enable_pipeline=True,
                  feat_corr=False, grad_corr=False, desc="20K-node RMAT (debug)"),
}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", choices=["ours", "reference"], default="ours")
    p.add_argument("--workload", default="rmat-1m", choices=list(WORKLOADS))
    p.add_argument("--dropout", type=float, default=0.5, help="reference default (helper/parser.py:14)")
    p.add_argument("--partition-method", default="random", choices=["random", "metis"])
    p.add_argument("--partition-obj", default="vol", choices=["vol", "cut"])
    p.add_argument("--graph-device", default="cuda", choices=["cuda", "cpu"],
                   help="where the synthetic graph is generated (the CPU and CUDA generators give different graphs; a METIS "
                        "partition cached under partitions/ belongs to the graph of one of them)")
    p.add_argument("--scale-down", type=int, default=1, help="1/k nodes and edges of the named shape (debug, stated in config)")
    p.add_argument("--cpu-full", action="store_true", help="cpu_baseline leg: time the full graph instead of the bounded sample")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-parity", action="store_true", help="skip the multi-GPU parity check before timing (N > 1)")
    p.add_argument("--use-pp", action="store_true", help="--use-pp of the reference scripts: layer-0 aggregate precomputed once")
    p.add_argument("--ncu-region", action="store_true", help="cudaProfilerStart/Stop around the instrumented steps")
    p.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying CUDA graphs")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32): its loss, "
                        "a seeded sample of its logits rows and every parameter and reduced gradient (rank 0)")
    args = p.parse_args()
    if args.steps < 1 or args.warmup < 0:
        p.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        p.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    return args


def engine_args(w, n_feat, n_class, n_train, n_parts, dropout, cuda_graph=False, use_pp=False):
    return argparse.Namespace(
        model="graphsage", backend="nccl", dtype=w["dtype"], n_layers=w["n_layers"], n_hidden=w["n_hidden"],
        n_linear=0, n_feat=n_feat, n_class=n_class, n_train=n_train, dropout=dropout,
        norm="layer", lr=1e-2, weight_decay=0.0, use_pp=use_pp, enable_pipeline=w["enable_pipeline"],
        feat_corr=w["feat_corr"], grad_corr=w["grad_corr"], corr_momentum=0.95, seed=0, n_epochs=0,
        log_every=10, n_partitions=n_parts, cuda_graph=cuda_graph)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=5)
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": float(self.rows[0][1]) if self.rows else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def shape_spec(w, scale_down=1):
    from pipegcn_b200.synthetic import SHAPES
    spec = dict(SHAPES[w["shape"]])
    if scale_down > 1:
        spec["n_nodes"] //= scale_down
        spec["n_edges"] //= scale_down
    return spec


# ----------------------------------------------------------------------------------------------- CPU arm
def cpu_reference_run(w, args, steps, warmup, full=True):
    """The reference's algorithm on the host cores: the oracle port (torch CPU + C/OpenMP SpMM), ONE partition, on
    the FULL graph of the workload (`full`) or on a stated 1/16 sample (the in-run `cpu_baseline` leg, bounded to
    ~30 s).  Nothing is extrapolated: `value` is epochs/s of exactly the graph named in `sample`."""
    from oracle import dglpart
    from oracle import setup as osetup
    from oracle.cbuild import set_threads
    from oracle.fabric import ThreadFabric
    from oracle.train import OracleArgs, run_rank
    from pipegcn_b200.synthetic import make_graph
    n_cpu = os.cpu_count() or 1
    base_scale = max(1, args.scale_down)

    def world(scale):
        g = make_graph(shape_spec(w, scale), device="cpu")
        part = torch.zeros(g.n_nodes, dtype=torch.int64)
        parts = dglpart.partition_graph(g.n_nodes, g.src, g.dst, part, 1, g.feat, g.label, g.train_mask)
        oargs = OracleArgs(n_layers=w["n_layers"], n_hidden=w["n_hidden"], n_feat=g.n_feat,
                           n_class=shape_spec(w)["n_class"], n_train=int(g.train_mask.sum()), dropout=args.dropout,
                           n_epochs=2, enable_pipeline=w["enable_pipeline"], feat_corr=w["feat_corr"],
                           grad_corr=w["grad_corr"])
        return g, osetup.setup_world(parts), oargs

    # thread count: on many-core hosts the fastest setting is below the core count; probe on a 1/16 sample
    probe_scale = base_scale * 16
    g_s, setups_s, oargs_s = world(probe_scale)
    cand = sorted({t for t in (8, 16, 32, 64, n_cpu) if t <= n_cpu})
    best = None
    for t in cand:
        set_threads(t)
        w1 = run_rank(setups_s[0], oargs_s, ThreadFabric(1), keep_trace=False).wall[-1]
        if best is None or w1 < best[0]:
            best = (w1, t)
    cores = best[1]
    set_threads(cores)
    if full:
        del g_s, setups_s
        gc.collect()
        g, setups, oargs = world(base_scale)
        scale_txt = "the FULL graph of the workload" if base_scale == 1 else f"the 1/{base_scale}-scale graph this run uses"
    else:
        g, setups, oargs = g_s, setups_s, oargs_s
        scale_txt = f"a 1/{probe_scale}-scale sample of the workload's graph (bounded leg; NOT extrapolated)"
    oargs = OracleArgs(**{**oargs.__dict__, "n_epochs": warmup + steps})
    tr = run_rank(setups[0], oargs, ThreadFabric(1), keep_trace=False)
    per_epoch = sum(tr.wall[warmup:]) / max(len(tr.wall[warmup:]), 1)
    return {
        "value": 1.0 / max(per_epoch, 1e-9), "unit": "epochs/s", "cores": cores, "kind": "port",
        "sample": (f"oracle (CPU port of the reference: torch {torch.__version__} CPU kernels + C/OpenMP SpMM, fp32), "
                   f"{cores} of {n_cpu} host threads (fastest of {cand} on a 1/{probe_scale} sample), 1 partition, on "
                   f"{scale_txt}: {g.n_nodes} nodes, {g.n_edges} edges, {steps} timed epochs after {warmup} warm-up"),
        "n_nodes": g.n_nodes, "n_edges": g.n_edges, "steps": steps, "warmup": warmup,
    }


LOGITS_SAMPLE_VALUES = 1 << 22      # 16 MB of float32: the dump stays far below 64 MB on every workload


def dump_outputs(out_dir, engine, loss):
    """The last timed step's results as float32 .npy files, so that two builds can be compared output for output: the
    summed loss, a fixed sample of logits rows (seed 0, sorted row ids, at most LOGITS_SAMPLE_VALUES values), and every
    parameter after the optimiser step with the reduced gradient that step applied."""
    import numpy as np
    out_dir.mkdir(parents=True, exist_ok=True)
    logits = engine.last_logits
    n_rows, n_class = logits.shape
    k = min(n_rows, LOGITS_SAMPLE_VALUES // n_class)
    rows = torch.randperm(n_rows, generator=torch.Generator().manual_seed(0))[:k].sort().values
    arrays = {"loss": loss.reshape(1), "logits_sample": logits[rows.to(logits.device)]}
    for name, p in engine.model.named_parameters():
        arrays[f"param.{name}"] = p.detach()
        arrays[f"grad.{name}"] = p.grad
    for name, t in arrays.items():
        np.save(out_dir / f"{name}.npy", t.float().cpu().numpy())


def teardown(world_size, engine_holder):
    """Leave like a library user would: drop the captured graphs (they hold NCCL kernels), free the engine, destroy
    the process group, return.  A watchdog only fires if communicator teardown hangs."""
    import torch.distributed as dist
    dog = threading.Timer(90.0, lambda: (sys.stderr.write("[bench] teardown watchdog fired\n"), os._exit(0)))
    dog.daemon = True
    dog.start()
    eng = engine_holder.pop("engine", None)
    if eng is not None:
        eng.graphs = None
        del eng
    gc.collect()
    torch.cuda.synchronize()
    if world_size > 1 and dist.is_initialized():
        dist.barrier()
        torch.cuda.synchronize()
        dist.destroy_process_group()
    dog.cancel()


def main():
    args = parse()
    w = WORKLOADS[args.workload]
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return
        steps, warmup = args.steps, args.warmup
        cb = cpu_reference_run(w, args, steps, warmup, full=True)
        line = {"impl": "reference", "metric": "epochs_per_sec", "value": cb["value"], "unit": "epochs/s",
                "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": 1e3 / cb["value"],
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": f"{args.workload}: {w['desc']}", "n_nodes": cb["n_nodes"], "n_edges": cb["n_edges"],
                           "partitions": 1, "partitions_note": "the CPU arm runs ONE partition at every --gpus N "
                           "(all host threads in one process; splitting it over gloo processes shares the same cores)",
                           "dropout": args.dropout},
                "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "epochs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (or --impl reference)"
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    import torch.distributed as dist
    from pipegcn_b200 import _C, ops
    from pipegcn_b200.partition import PartitionPlan
    from pipegcn_b200.synthetic import make_graph, random_partition
    from pipegcn_b200.train import RankEngine
    from pipegcn_b200.world import DistWorld, LocalWorld

    if world_size > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world_size, device_id=dev)
        world = DistWorld(device=dev)
    else:
        world = LocalWorld(1, dev).view(0)
    assert args.gpus == world_size, f"--gpus {args.gpus} but WORLD_SIZE={world_size}"

    # ---- real multi-GPU parity (CUDA IPC + NVLink pushes + NCCL + graph replay) against the CPU oracle, before timing
    parity = None
    if world_size > 1 and not args.no_parity:
        from tools.dist_parity import check_world
        parity = check_world(world, dev, shapes=("tiny", "small"), modes=("pipeline_corr",), graph_modes=(False, True))
        if rank == 0 and not parity["ok"]:
            print(f"[bench] multi-GPU parity FAILED: {parity}", file=sys.stderr)

    t_setup = time.time()
    spec = shape_spec(w, args.scale_down)
    n_class = spec["n_class"]
    if w.get("distributed_build"):
        from pipegcn_b200.distgraph import build_rank_layout
        layout, ginfo = build_rank_layout(spec, rank, world_size, dev, world)
        n_nodes, n_edges, n_feat, n_train = ginfo["n_nodes"], ginfo["n_edges"], spec["n_feat"], ginfo["n_train"]
        part_method = "random (hash of the node id; per-rank construction)"
    else:
        g = make_graph(spec, device=dev if args.graph_device == "cuda" else "cpu")
        if args.graph_device == "cpu":
            g = type(g)(g.n_nodes, g.src.to(dev), g.dst.to(dev), g.feat.to(dev), g.label.to(dev), g.train_mask.to(dev))
        if args.partition_method == "random" or world_size == 1:
            part = random_partition(g.n_nodes, world_size, seed=1, device=dev)
        else:
            from pipegcn_b200.helper.utils import graph_partition
            pargs = argparse.Namespace(partition_method="metis", partition_obj=args.partition_obj, n_partitions=world_size,
                                       dataset=f"synthetic:{w['shape']}" + (f"-div{args.scale_down}" if args.scale_down > 1 else "")
                                       + ("-cpugen" if args.graph_device == "cpu" else ""),
                                       graph_name="", inductive=False, partition_cache=True, skip_partition=False)
            part = graph_partition(g, pargs, rank)
        if world_size > 1:   # every rank built the graph itself; make sure they agree
            chk = torch.stack([g.src.sum(), g.dst.sum(), part.sum(), g.train_mask.sum()]).to(torch.float64)
            lo, hi = chk.clone(), chk.clone()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            assert torch.equal(lo, hi), "ranks generated different synthetic graphs"
        layout = PartitionPlan(g, part, world_size).build(rank)
        n_nodes, n_edges, n_feat, n_train = g.n_nodes, g.n_edges, g.n_feat, int(g.train_mask.sum().item())
        part_method = args.partition_method if world_size > 1 else "none (1 partition)"
        del g, part
    eargs = engine_args(w, n_feat, n_class, n_train, world_size, args.dropout, cuda_graph=not args.no_graph,
                        use_pp=args.use_pp)
    engine = RankEngine(layout, eargs, world)
    engine.keep_logits = bool(args.dump_outputs)      # a reference to the logits each step writes anyway; no extra work
    holder = {"engine": engine}
    feat_host = layout.feat.to(engine.dtype).cpu().pin_memory()
    label_host = engine.labels.cpu().pin_memory()
    layout_info = dict(n_in=layout.num_in, halo=layout.num_all - layout.num_in, nnz=layout.nnz)
    del layout
    gc.collect()
    torch.cuda.empty_cache()
    setup_s = time.time() - t_setup

    def barrier():
        torch.cuda.synchronize()
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world_size > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(n_steps, fn):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_steps):
            fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    last = {}

    def step():
        last["loss"] = engine.run_epoch()

    def step_e2e():
        engine.set_features(feat_host)
        engine.labels.copy_(label_host, non_blocking=True)
        loss = engine.run_epoch()
        return float(loss.item())      # device -> host read of the step's result

    for _ in range(max(args.warmup, 3)):
        step()
    engine.buffer.check_status()

    # ---- instrumented eager epochs: every aggregate launch bracketed by CUDA events (roofline)
    ops.PROFILE = []
    _C.LAUNCHES = 0
    n_eager = args.steps if args.no_graph else min(args.steps, 5)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    engine.buffer.take_wait_ns()
    if args.ncu_region:
        torch.cuda.cudart().cudaProfilerStart()
    ms_eager_total = timed(n_eager, step)
    if args.ncu_region:
        torch.cuda.cudart().cudaProfilerStop()
    launches_per_step = _C.LAUNCHES / max(n_eager, 1)
    prof, ops.PROFILE = ops.PROFILE, None
    engine.buffer.check_status()
    eager_wait_s = engine.buffer.take_wait_ns() / 1e9 / max(n_eager, 1)
    ms_eager = ms_eager_total / n_eager

    # ---- timed region proper: K epochs replayed from CUDA graphs (one graph per epoch parity)
    graph_info = {"enabled": False}
    if not args.no_graph:
        try:
            engine.capture()
            for _ in range(2):
                step()
            graph_info = {"enabled": True, "graphs": len(engine.graphs)}
        except Exception as e:   # noqa: BLE001  -- same kernels either way; only the launch mechanism differs
            engine.graphs = None
            engine.buffer.graph_mode = False
            ops.STEP_DEV = None
            graph_info = {"enabled": False, "error": f"{type(e).__name__}: {str(e)[:200]}"}
            print(f"[bench] CUDA graph capture failed, timing eager launches: {e}", file=sys.stderr)
    engine.buffer.take_wait_ns()
    if graph_info["enabled"] or not args.no_graph:
        ms_total = timed(args.steps, step)
        wait_s = engine.buffer.take_wait_ns() / 1e9 / args.steps
    else:
        ms_total = ms_eager_total * args.steps / n_eager
        wait_s = eager_wait_s
    engine.buffer.check_status()
    if args.dump_outputs and rank == 0:
        dump_outputs(Path(args.dump_outputs), engine, last["loss"])
    exposed_s = max_over_ranks(wait_s)
    launches = int(round(launches_per_step * args.steps))
    ms_step = ms_total / args.steps
    value = 1e3 / ms_step

    # ---- roofline of the dominant kernel (the forward+backward neighbour aggregate, HBM bound)
    hbm_peak, peak_src = peaks()
    agg_ms = sum(a.elapsed_time(b) for a, b, _ in prof)
    agg_bytes = sum(nb for _, _, nb in prof)
    n_agg = len(prof)
    achieved = (agg_bytes / 1e9) / (agg_ms / 1e3) if agg_ms > 0 else 0.0
    traffic, traffic_src = None, None
    tf = ROOT / "profiles" / "agg_traffic.json"
    if tf.exists():       # per-launch DRAM bytes of the aggregate kernel from the committed `ncu --set full` captures
        ent = json.loads(tf.read_text()).get(f"{args.workload}:{world_size}")
        if isinstance(ent, dict):
            traffic, traffic_src = ent.get("bytes"), ent.get("source")
        else:
            traffic = ent
    roofline = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "traffic": traffic, "traffic_source": traffic_src,
                "kernel": "pg::agg2_kernel (+fix-up), forward and backward aggregate",
                "launches": n_agg, "avg_launch_ms": agg_ms / max(n_agg, 1),
                "algorithmic_bytes_per_launch": agg_bytes / max(n_agg, 1),
                "share_of_step": agg_ms / ms_eager_total if ms_eager_total else None, "peak_source": peak_src,
                "measured_in": f"{n_eager} eager (Python-launched) epochs before the graph-replayed timed region (rank 0)"}

    # ---- end to end: host buffers, H2D of the step's inputs and D2H of its loss inside the timed region.  The inputs
    #      of step i + 1 travel (pinned host -> staging buffer, copy stream) while step i computes; every one of the K
    #      copies, the first included, is issued and completed inside the timed region
    e2e = None
    if not args.no_e2e:
        step_e2e()

        def e2e_region(n_steps):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            slot = engine.prefetch_features(feat_host, label_host)
            for i in range(n_steps):
                nxt = engine.prefetch_features(feat_host, label_host) if i + 1 < n_steps else None
                engine.commit_features(slot)
                loss = engine.run_epoch()
                float(loss.item())                       # device -> host read of the step's result
                slot = nxt
            e1.record()
            barrier()
            return max_over_ranks(e0.elapsed_time(e1))

        e2e_region(2)
        ms_e2e = e2e_region(args.steps) / args.steps
        e2e = {"value": 1e3 / ms_e2e, "unit": "epochs/s",
               "h2d_bytes_per_step": int(feat_host.numel() * feat_host.element_size() + label_host.numel() * 8),
               "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e,
               "how": "public API (RankEngine.prefetch_features / commit_features / run_epoch): per step one H2D copy of "
                      "the features (double-buffered: step i+1's copy overlaps step i's compute) + labels, one D2H read "
                      "of the loss; all K copies inside the timed region"}

    clocks = sampler.stop() if sampler else None      # sampled across the eager, replayed and end-to-end regions
    cb = None
    if rank == 0 and world_size == 1 and not args.no_cpu_baseline:
        # same graph as the GPU arm when one CPU epoch takes ~20 s (<= 25 M edges), else the stated 1/16 sample
        cpu_full = args.cpu_full or n_edges <= 25_000_000
        cb = cpu_reference_run(w, args, steps=1 if cpu_full else 2, warmup=1, full=cpu_full)

    if rank == 0:
        secondary = None
        sf = ROOT / "profiles" / "r2_secondary.json"
        if sf.exists() and args.workload == "rmat-1m":
            try:
                secondary = json.loads(sf.read_text())
            except Exception:   # noqa: BLE001
                secondary = None
        line = {
            "metric": "epochs_per_sec", "value": value, "unit": "epochs/s", "n_gpus": world_size,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": w["dtype"], "data": "synthetic",
            "config": {"workload": f"{args.workload}: {w['desc']}", "n_nodes": n_nodes, "n_edges": n_edges,
                       "partitions": world_size, "partition_method": part_method, "graph_generated_on": args.graph_device,
                       "dropout": args.dropout,
                       "use_pp": args.use_pp, "scale_down": args.scale_down,
                       "n_in_rank0": layout_info["n_in"], "halo_rank0": layout_info["halo"],
                       "nnz_rank0": layout_info["nnz"], "linear": ops.LINEAR_IMPL,
                       "l2": "per-epoch working set (features, activations, indices) exceeds the 126 MB L2; no flush",
                       "setup_s": round(setup_s, 1)},
            "exposed_comm_s_per_epoch": exposed_s,
            "exposed_comm_frac": exposed_s / (ms_step / 1e3) if ms_step else None,
            "exposed_comm_how": "ns spent in pg::halo_wait_kernel, accumulated on the device (%globaltimer) inside the "
                                "timed region (graph replays), max over ranks",
            "eager_ms_per_step": ms_eager, "eager_exposed_comm_s_per_epoch": eager_wait_s, "cuda_graph": graph_info,
            "parity": parity, "roofline": roofline, "e2e": e2e, "cpu_baseline": cb, "gpu_launches": launches,
            "clocks": clocks, "secondary": secondary,
        }
        print(json.dumps(line), flush=True)
    sys.stdout.flush()
    del engine
    teardown(world_size, holder)


if __name__ == "__main__":
    main()
