"""Accuracy evaluation and checkpointing around the hot path.

Counterparts of /root/reference/train.py: `calc_acc` (:11-17), `evaluate_induc`
(:20-39), `evaluate_trans` (:42-61) and the best-model bookkeeping of `run`
(:377-400).  The reference deep-copies the model, moves it to the CPU and evaluates on
the whole DGL graph from a worker thread; here the SAME sm_100a kernels evaluate the
homogeneous full graph on the GPU (the eval branch of GraphSAGELayer, layer.py:52-62),
on the training stream, from the live weights.
"""
from __future__ import annotations

import os
from typing import Dict, Optional

import torch

from .graph import PartGraph
from .synthetic import GlobalGraph, induced_subgraph


def full_graph(g: GlobalGraph, device) -> PartGraph:
    """Homogeneous graph of all N nodes as a `PartGraph` (num_in == num_all): CSR by destination."""
    from .partition import _csr_from_pairs
    dev = torch.device(device)
    src, dst = g.src.to(dev), g.dst.to(dev)
    indptr, indices = _csr_from_pairs(dst, src, g.n_nodes, g.n_nodes)
    t_indptr, t_indices = _csr_from_pairs(src, dst, g.n_nodes, g.n_nodes)
    return PartGraph(g.n_nodes, g.n_nodes, indptr, indices, t_indptr, t_indices, g.in_degrees().to(dev), device=dev)


def calc_acc(logits: torch.Tensor, labels: torch.Tensor) -> float:
    """train.py:11-17: argmax accuracy for [N] labels; for [N, C] 0/1 labels the micro-F1 of `logits > 0`
    (f1_score(..., average='micro')), counted on the GPU by ops.multilabel_f1."""
    if labels.dim() == 2:
        from .ops import multilabel_f1, pack_multilabel
        return multilabel_f1(logits, pack_multilabel(labels))
    if labels.numel() == 0:
        return float('nan')
    return float((logits.argmax(dim=1) == labels).sum().item()) / labels.shape[0]


class EvalSet:
    """What rank 0 keeps for evaluation: graph(s), features, labels and masks on the device.  Multi-label targets are
    packed once (`ybits`, ops.pack_multilabel) together with the int32 row ids of every mask (`<mask>_rows`)."""

    def __init__(self, g: GlobalGraph, device, inductive: bool = False, dtype=torch.float32):
        self.inductive = bool(inductive)
        dev = torch.device(device)
        val_mask, test_mask = g.val_mask, g.test_mask

        def pack(sub: GlobalGraph, masks: Dict[str, torch.Tensor]):
            out = dict(graph=full_graph(sub, dev), feat=sub.feat.to(dev).to(dtype), label=sub.label.to(dev),
                       **{k: v.to(dev) for k, v in masks.items()})
            if sub.label.dim() == 2:
                from .ops import pack_multilabel
                out["ybits"] = pack_multilabel(out.pop("label"))
                for k in masks:
                    out[k[:-len("_mask")] + "_rows"] = torch.nonzero(out[k]).flatten().to(torch.int32)
            return out

        if inductive:
            # inductive_split (utils.py): the validation graph holds train+val nodes, the test graph everything
            keep = g.train_mask | val_mask
            sub, ids = induced_subgraph(g, keep)
            self.val = pack(sub, dict(val_mask=val_mask[ids]))
            self.test = pack(g, dict(test_mask=test_mask))
        else:
            self.val = self.test = pack(g, dict(val_mask=val_mask, test_mask=test_mask))


@torch.no_grad()
def _logits(model, part) -> torch.Tensor:
    was_training = model.training
    model.eval()
    try:
        return model(part["graph"], part["feat"]).float()
    finally:
        model.train(was_training)


def _score(logits: torch.Tensor, part, mode: str) -> float:
    """calc_acc over the rows of `<mode>_mask`: accuracy, or micro-F1 against the packed multi-label targets."""
    if "ybits" in part:
        from .ops import multilabel_f1
        return multilabel_f1(logits, part["ybits"], part[mode + "_rows"])
    mask = part[mode + "_mask"]
    return calc_acc(logits[mask], part["label"][mask])


def _emit(buf: str, result_file_name: Optional[str]):
    if result_file_name is not None:
        os.makedirs(os.path.dirname(result_file_name) or ".", exist_ok=True)
        with open(result_file_name, 'a+') as f:
            f.write(buf + '\n')
    print(buf)


def evaluate_trans(name, model, part, result_file_name=None) -> float:
    """train.py:42-61: validation and test accuracy (micro-F1 for a multi-label task, printed as "Accuracy" like the
    reference) on the full graph; returns the validation score."""
    logits = _logits(model, part)
    val_acc = _score(logits, part, "val")
    test_acc = _score(logits, part, "test")
    _emit("{:s} | Validation Accuracy {:.2%} | Test Accuracy {:.2%}".format(name, val_acc, test_acc), result_file_name)
    return val_acc


def evaluate_induc(name, model, part, mode, result_file_name=None) -> float:
    """train.py:20-39; mode: 'val' or 'test'."""
    logits = _logits(model, part)
    acc = _score(logits, part, mode)
    _emit("{:s} | Accuracy {:.2%}".format(name, acc), result_file_name)
    return acc


def result_file(args) -> str:
    """train.py:309-316."""
    tag = ('_grad_feat' if args.grad_corr and args.feat_corr else '_grad' if args.grad_corr
           else '_feat' if args.feat_corr else '')
    return 'results/%s_n%d_p%d%s.txt' % (str(args.dataset).replace(':', '_'), args.n_partitions,
                                         int(args.enable_pipeline), tag)


class BestModel:
    """Best-validation bookkeeping of train.py:377-400: keep the state_dict with the highest validation accuracy
    (micro-F1 for a multi-label task),
    save it under the reference's key names as `model/<graph_name>_final.pth.tar`."""

    def __init__(self):
        self.acc, self.state = 0.0, None

    def offer(self, acc: float, model):
        if self.state is None or acc > self.acc:
            self.acc = acc
            self.state = {k: v.detach().to('cpu', copy=True) for k, v in model.state_dict().items()}

    def save(self, args) -> Optional[str]:
        if self.state is None:
            return None
        os.makedirs('model', exist_ok=True)
        path = 'model/' + str(args.graph_name).replace(':', '_') + '_final.pth.tar'
        torch.save(self.state, path)
        return path
