"""Multi-GPU parity: one process per GPU (torchrun), DistWorld + CUDA IPC + NVLink pushes, against the CPU oracle.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 \
        tools/dist_parity.py [tiny|small]
Every rank builds the same seeded graph, runs the oracle world on the host (threads) and its own rank of the
CUDA engine, and compares logits / losses / reduced gradients per epoch in the four exchange modes.
`check_world` is the same check as a function: `bench.py --gpus N` calls it before timing and reports the result in
its JSON line (`"parity"`), `tests/test_dist_gpu.py` launches this file under torchrun when >= 2 GPUs are visible.
"""
import os
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import torch
import torch.distributed as dist

MODES = {
    "sync": dict(),
    "sync_corr": dict(feat_corr=True, grad_corr=True, corr_momentum=0.9),
    "pipeline": dict(enable_pipeline=True),
    "pipeline_corr": dict(enable_pipeline=True, feat_corr=True, grad_corr=True, corr_momentum=0.95),
}
TOL = 2e-3      # worst relative error (logits, loss, reduced gradients; fp32, 3xTF32 GEMMs): measured ~5e-6


def check_mode(world, dev, shape, mode, use_graph, verbose=False):
    """Worst relative error (max over ranks) of this rank's engine against the oracle trace, teacher-forced weights."""
    from oracle.train import initial_state, run_world
    from pipegcn_b200.train import RankEngine
    from pipegcn_b200.synthetic import SHAPES
    from tests.helpers import make_args, small_world
    from tests.ml_oracle import multilabel_loss
    rank, size = world.rank, world.size
    n_class = SHAPES[shape]["n_class"]
    g, _, layouts, setups = small_world(shape, size)
    n_epochs = 6 if use_graph else 4
    oargs, eargs = make_args(g, n_class, n_epochs=n_epochs, **MODES[mode])
    eargs.cuda_graph = use_graph
    init = initial_state(oargs)
    if g.label.dim() == 2:                                  # multi-label shape: the reference's yelp loss
        with multilabel_loss():
            traces = run_world(setups, oargs, init_state=init)
    else:
        traces = run_world(setups, oargs, init_state=init)
    eng = RankEngine(layouts[rank], eargs, world, init_state=init, seg_len=32)
    eng.keep_logits = True
    worst = 0.0
    for e in range(n_epochs):
        if use_graph and e == 3:
            eng.capture()
        eng.model.load_state_dict(traces[0].states[e])      # teacher forcing, see tests/test_engine_gpu.py
        loss = eng.run_epoch()
        eng.buffer.check_status()
        ref = traces[rank]
        d = (eng.last_logits.float().cpu() - ref.logits[e]).abs().max().item()
        worst = max(worst, d / max(ref.logits[e].abs().max().item(), 1e-6))
        dl = abs(float(loss.item()) - ref.losses[e]) / abs(ref.losses[e])
        for n, p in eng.model.named_parameters():
            gd = (p.grad.float().cpu() - ref.grads[e][n]).abs().max().item()
            worst = max(worst, gd / max(ref.grads[e][n].abs().max().item(), 1e-6))
        worst = max(worst, dl)
        if verbose and rank == 0:
            print(f"[dist_parity]   mode={mode} epoch {e} graph={int(eng.graphs is not None)} logits err {d:.3e} "
                  f"loss rel {dl:.3e} worst {worst:.3e}", flush=True)
    eng.buffer.synchronize()
    torch.cuda.synchronize()
    flag = torch.tensor([worst], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MAX)
    eng.graphs = None
    eng.buffer.release()            # collective: unmap the peers' heaps, barrier, free
    del eng
    torch.cuda.synchronize()
    dist.barrier()
    return float(flag.item())


def check_world(world, dev, shapes=("tiny",), modes=tuple(MODES), graph_modes=(False,), verbose=False):
    from pipegcn_b200 import ops
    cases, worst = [], 0.0
    for shape in shapes:
        for use_graph in graph_modes:
            for mode in modes:
                err = check_mode(world, dev, shape, mode, use_graph, verbose)
                ops.STEP_DEV = None
                cases.append({"shape": shape, "mode": mode, "graph": bool(use_graph), "worst_rel": err})
                worst = max(worst, err)
    return {"ok": worst < TOL, "worst_rel": worst, "tol": TOL, "ranks": world.size,
            "what": "DistWorld (CUDA IPC + in-kernel NVLink stores + NCCL all-reduce) vs the CPU oracle: logits, loss, "
                    "reduced gradients per epoch, teacher-forced weights", "cases": cases}


def main():
    rank, size, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    dist.init_process_group("nccl", rank=rank, world_size=size, device_id=dev)
    from pipegcn_b200.world import DistWorld
    shape = sys.argv[1] if len(sys.argv) > 1 else "tiny"
    use_graph = os.environ.get("PG_PARITY_GRAPH", "0") == "1"       # epochs >= 3 replayed from CUDA graphs
    only = os.environ.get("PG_PARITY_MODES")
    modes = tuple(m for m in MODES if not only or m in only.split(","))
    res = check_world(DistWorld(device=dev), dev, shapes=(shape,), modes=modes, graph_modes=(use_graph,),
                      verbose=bool(os.environ.get("PG_PARITY_VERBOSE")))
    if rank == 0:
        for c in res["cases"]:
            print(f"[dist_parity] {c['shape']} P={size} graph={int(c['graph'])} mode={c['mode']:14s} worst relative error "
                  f"{c['worst_rel']:.3e} {'OK' if c['worst_rel'] < TOL else 'FAIL'}", flush=True)
        print("[dist_parity] " + ("ALL OK" if res["ok"] else "FAILED"), flush=True)
    sys.stdout.flush()
    torch.cuda.synchronize()
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0 and not res["ok"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
