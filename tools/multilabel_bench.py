"""Measurements of the multi-label task (scripts/yelp.sh) on the GPU; one JSON line per measurement.

    python tools/multilabel_bench.py [--out profiles/multilabel_bench.jsonl] [--steps 50]
    torchrun --nproc-per-node 3 tools/multilabel_bench.py --e2e-only     # the 3-GPU end-to-end row

* loss kernels: pg_bce_fwd + pg_bce_bwd (with the bias column sums) against torch's BCEWithLogitsLoss(reduction='sum')
  forward + backward on [538 K, 100] logits (yelp-shaped's train rows), bf16 and fp32, CUDA events over --iters
  launches after warm-up.  Algorithmic bytes: logits read twice, gradient written once, packed labels read twice
  (torch reads float32 labels: 400 B a row instead of 16 B).  The logits and the gradient together are larger than
  the 126 MB L2 in both dtypes.
* end to end: yelp.sh's flags (--n-layers 4 --n-linear 2 --n-hidden 512 --dropout 0.1 --lr 0.001 --inductive
  --enable-pipeline --use-pp) on synthetic:yelp-shaped, epochs replayed from CUDA graphs, device-timed epochs/s;
  one partition per GPU.
Every line records the card's name and power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True)
    name, limit = (q.stdout.strip().split(", ") + ["?", "?"])[:2] if q.returncode == 0 else ("?", "?")
    return dict(gpu=name or torch.cuda.get_device_name(), power_limit=limit)


def _time(fn, iters, warmup=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def loss_kernels(rows, c, dtype, iters):
    from pipegcn_b200 import _C, ops
    from pipegcn_b200.graph import alloc_rows
    gen = torch.Generator(device="cuda").manual_seed(0)
    z = alloc_rows(rows, c, dtype, "cuda")
    z.copy_(torch.randn(rows, c, generator=gen, device="cuda") * 3)
    y = (torch.rand(rows, c, generator=gen, device="cuda") < 0.15).float()
    yb = ops.pack_multilabel(y)
    g = alloc_rows(rows, c, dtype, "cuda")
    grid = _C.lib.pg_row_grid(rows)
    partial = torch.empty(grid * c, dtype=torch.float32, device="cuda")
    loss = torch.zeros(1, dtype=torch.float32, device="cuda")
    colsum = torch.empty(c, dtype=torch.float32, device="cuda")
    up = torch.ones(1, dtype=torch.float32, device="cuda")
    code, st = _C.dtype_code(dtype), _C.stream_ptr()

    def ours():
        _C.lib.pg_bce_fwd(z.data_ptr(), z.stride(0), yb.data_ptr(), yb.shape[1], rows, c, code, partial.data_ptr(),
                          loss.data_ptr(), st)
        _C.lib.pg_bce_bwd(z.data_ptr(), z.stride(0), yb.data_ptr(), yb.shape[1], up.data_ptr(), rows, rows, c, code,
                          g.data_ptr(), g.stride(0), colsum.data_ptr(), partial.data_ptr(), st)

    zt = z.detach().contiguous().requires_grad_()
    yt = y.to(dtype)
    fcn = torch.nn.BCEWithLogitsLoss(reduction="sum")

    def theirs():
        zt.grad = None
        fcn(zt, yt).backward()

    t_ours, t_torch = _time(ours, iters), _time(theirs, iters)
    es = z.element_size()
    nbytes = 3 * rows * c * es + 2 * rows * yb.shape[1] * 4
    nbytes_torch = 3 * rows * c * es + 2 * rows * c * yt.element_size()
    return dict(what="bce_loss_fwd_bwd", rows=rows, c=c, dtype=str(dtype).split(".")[1], iters=iters,
                pg_ms=round(t_ours, 4), torch_ms=round(t_torch, 4), speedup=round(t_torch / t_ours, 2),
                pg_alg_bytes=nbytes, pg_GBps=round(nbytes / t_ours / 1e6, 1),
                torch_alg_bytes=nbytes_torch, torch_GBps=round(nbytes_torch / t_torch / 1e6, 1))


def end_to_end(dtype, steps, world, rank, size, dev):
    from pipegcn_b200.partition import PartitionPlan
    from pipegcn_b200.synthetic import SHAPES, make_graph, random_partition, train_subgraph
    from pipegcn_b200.train import RankEngine
    g = train_subgraph(make_graph("yelp-shaped", device=dev))                     # --inductive
    part = random_partition(g.n_nodes, size, seed=1, device=dev)
    layout = PartitionPlan(g, part, size).build(rank)
    n_train = int(g.train_mask.sum().item())
    del g
    args = argparse.Namespace(model="graphsage", backend="nccl", dtype=dtype, n_layers=4, n_hidden=512, n_linear=2,
                              n_feat=300, n_class=SHAPES["yelp-shaped"]["n_class"], n_train=n_train, dropout=0.1,
                              norm="layer", lr=1e-3, weight_decay=0.0, use_pp=True, enable_pipeline=True,
                              feat_corr=False, grad_corr=False, corr_momentum=0.95, seed=0, cuda_graph=True)
    eng = RankEngine(layout, args, world)
    for _ in range(3):
        eng.run_epoch()
    eng.capture()
    for _ in range(3):
        eng.run_epoch()
    torch.cuda.synchronize()
    world.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = eng.run_epoch()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return dict(what="yelp_sh_end_to_end", shape="yelp-shaped", gpus=size, dtype=dtype, steps=steps,
                epoch_ms=round(ms, 3), epochs_per_s=round(1000.0 / ms, 1), final_loss=float(loss.item()) / max(eng.part_train, 1),
                flags="--n-layers 4 --n-linear 2 --n-hidden 512 --dropout 0.1 --lr 0.001 --inductive --enable-pipeline "
                      "--use-pp, CUDA-graph replay")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "multilabel_bench.jsonl"))
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--e2e-only", action="store_true")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "tools/multilabel_bench.py measures on a CUDA device"
    rank, size = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
    dev = torch.device("cuda", torch.cuda.current_device())
    from pipegcn_b200.world import DistWorld, LocalWorld
    if size > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", rank=rank, world_size=size, device_id=dev)
        world = DistWorld(device=dev)
    else:
        world = LocalWorld(1, dev).view(0)
    info = dict(card(), stamp=time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()))
    lines = []
    if not a.e2e_only and rank == 0:
        for dtype in (torch.bfloat16, torch.float32):
            lines.append(dict(loss_kernels(538_000, 100, dtype, a.iters), **info))
            print(json.dumps(lines[-1]), flush=True)
    for dtype in ("bf16", "fp32"):
        r = end_to_end(dtype, a.steps, world, rank, size, dev)
        if rank == 0:
            lines.append(dict(r, **info))
            print(json.dumps(lines[-1]), flush=True)
    if rank == 0:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        with open(a.out, "a") as f:
            for l in lines:
                f.write(json.dumps(l) + "\n")
    if size > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
