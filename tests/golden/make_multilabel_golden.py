"""Generate tests/golden/multilabel/ref_multilabel_pp_p3.pt by running the UNMODIFIED reference (/root/reference) on
the host.

    python tests/golden/make_multilabel_golden.py     # build container only

The run is scripts/yelp.sh scaled down: a multi-label graph (`tiny-ml`: [N, 12] 0/1 labels), `dataset = 'yelp'`,
3 partitions, 4 layers of which 2 linear, --use-pp, --enable-pipeline, hidden 16, dropout 0, 3 epochs.  Each rank is
make_golden.py's worker, unchanged, with the settings it takes from module level replaced for this run: the graph,
the layer and class counts, `n_linear` and `dataset` in its argument namespace, and the loss of its epoch loop, which
follows /root/reference/train.py:317-320 (dataset 'yelp' -> BCEWithLogitsLoss(reduction='sum')).

The fixture lives in its own directory (the single-label golden tests take every tests/golden/ref_*.pt).  To keep
it small it holds the graph's labels, train mask and partition but only a fingerprint of its edges and features
(`make_graph('tiny-ml')` rebuilds them), of each rank's set-up the sizes, labels and train mask (the index spaces are
pinned by the single-label fixtures), per-layer records of the graph layers only (the linear tail is checked
through the logits), and tensors that are equal (the weights and reduced gradients every rank holds, the static
layer-0 input of every epoch) are stored once.
"""
import sys
import types
from pathlib import Path

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
OUT = HERE / "multilabel"

NAME, N_PARTS, SHAPE, DATASET = "multilabel_pp_p3", 3, "tiny-ml", "yelp"
N_LAYERS, N_LINEAR, N_CLASS = 4, 2, 12
CFG = dict(n_parts=N_PARTS, use_pp=True, enable_pipeline=True)


def worker(rank, size, name, cfg, port, q):
    sys.path.insert(0, str(ROOT))
    import argparse

    import torch

    import pipegcn_b200.synthetic as syn
    from tests.golden import make_golden as mg

    make_graph = syn.make_graph
    syn.make_graph = lambda shape, *a, **kw: make_graph(SHAPE if shape == "tiny" else shape, *a, **kw)
    mg.N_LAYERS, mg.N_CLASS = N_LAYERS, N_CLASS

    class Args(argparse.Namespace):
        def __init__(self, **kw):
            kw.update(n_linear=N_LINEAR, dataset=DATASET)
            super().__init__(**kw)
    mg.argparse = types.SimpleNamespace(Namespace=Args)

    ce = torch.nn.CrossEntropyLoss

    def loss(reduction="mean"):                                  # train.py:317-320
        return torch.nn.BCEWithLogitsLoss(reduction=reduction) if DATASET == "yelp" else ce(reduction=reduction)
    torch.nn.CrossEntropyLoss = loss
    mg.worker(rank, size, name, cfg, port, q)


def share_equal_tensors(obj, seen=None):
    """Replace every tensor equal to one met earlier by that earlier object (torch.save then stores it once)."""
    import torch
    seen = [] if seen is None else seen
    if isinstance(obj, torch.Tensor):
        for t in seen:
            if t.dtype == obj.dtype and t.shape == obj.shape and torch.equal(t, obj):
                return t
        seen.append(obj)
        return obj
    if isinstance(obj, dict):
        return {k: share_equal_tensors(v, seen) for k, v in obj.items()}
    if isinstance(obj, list):
        return [share_equal_tensors(v, seen) for v in obj]
    return obj


def main():
    import tempfile

    import torch
    import torch.multiprocessing as mp
    mp.set_start_method("spawn", force=True)
    sys.path.insert(0, str(ROOT))
    from pipegcn_b200.synthetic import make_graph, random_partition
    from tests.golden import make_golden as mg
    tmp = tempfile.mkdtemp(prefix="pg_golden_")
    procs = [mp.Process(target=worker, args=(r, N_PARTS, NAME, CFG, 29750, tmp)) for r in range(N_PARTS)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=600)
        assert p.exitcode == 0, f"reference worker failed ({NAME})"
    got = [torch.load(f"{tmp}/{NAME}_{r}.pt") for r in range(N_PARTS)]
    for e in range(mg.N_EPOCHS):                                 # the reducer's result is the same on every rank
        for n, t in got[0]["epochs"][e]["grads"].items():
            for r in range(1, N_PARTS):
                assert torch.equal(t, got[r]["epochs"][e]["grads"][n]), (e, n)
    for r in got:                # of the set-up, what multi-label labels pass through (index spaces: make_golden.py)
        r["layout"] = {k: r["layout"][k] for k in ("num_in", "num_all", "recv_shape", "label", "train_mask")}
        for ep in r["epochs"]:   # the linear tail: its input is the layer before's activation, its output the logits
            for i in range(N_LAYERS - N_LINEAR, N_LAYERS):
                del ep["layers"][i]
    g = make_graph(SHAPE)
    fixture = {
        "about": "outputs of the unmodified reference (GATECH-EIC/PipeGCN @ 73ab949) run by "
                 "tests/golden/make_multilabel_golden.py",
        "config": dict(CFG, n_epochs=mg.N_EPOCHS, n_layers=N_LAYERS, n_linear=N_LINEAR, n_hidden=mg.N_HIDDEN,
                       n_class=N_CLASS, seed=mg.SEED, shape=SHAPE, dataset=DATASET, dropout=0.0, lr=1e-2),
        # the graph is make_graph(SHAPE): its labels and mask are kept, the edges and features as a fingerprint
        "graph": dict(n_nodes=g.n_nodes, n_edges=g.n_edges, src_sum=int(g.src.sum()), dst_sum=int(g.dst.sum()),
                      feat_sum=float(g.feat.double().sum()), label=g.label, train_mask=g.train_mask,
                      part=random_partition(g.n_nodes, N_PARTS)),
        "ranks": got,
    }
    OUT.mkdir(exist_ok=True)
    path = OUT / f"ref_{NAME}.pt"
    torch.save(share_equal_tensors(fixture), path)
    print(f"wrote {path} ({path.stat().st_size / 1024:.0f} KiB); losses rank0 "
          f"{[round(ep['loss'], 4) for ep in got[0]['epochs']]}")


if __name__ == "__main__":
    main()
