"""Synthetic graphs of the shapes BASELINE.json names (SURVEY.md §8d).

The reference loads Reddit / ogbn-* through DGL + network downloads
(/root/reference/helper/utils.py:74-96); neither is available, so the engine is
fed seeded RMAT graphs with the same global preprocessing the reference applies
after loading: drop self loops, then add exactly one self loop per node
(utils.py:94-95).  Everything is plain torch so the same code runs on the host
(tests) and on the GPU (bench; a 115 M-edge build takes seconds there).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch


@dataclass
class GlobalGraph:
    """Edge list of the whole (un-partitioned) graph; ids are int64 in [0, n_nodes)."""
    n_nodes: int
    src: torch.Tensor          # [E] int64, message source u
    dst: torch.Tensor          # [E] int64, message destination v (edge u -> v)
    feat: torch.Tensor         # [N, F] float32
    label: torch.Tensor        # [N] int64, or [N, C] float32 0/1 for a multi-label shape
    train_mask: torch.Tensor   # [N] bool

    @property
    def n_edges(self) -> int:
        return int(self.src.numel())

    @property
    def n_feat(self) -> int:
        return int(self.feat.shape[1])

    def in_degrees(self) -> torch.Tensor:
        """Global in-degree including the self loop (utils.py:142)."""
        return torch.bincount(self.dst, minlength=self.n_nodes)

    # the reference's datasets carry val/test masks (utils.py:24-29); the synthetic graphs split the
    # non-training nodes in two by id parity
    @property
    def val_mask(self) -> torch.Tensor:
        ids = torch.arange(self.n_nodes, device=self.train_mask.device)
        return ~self.train_mask & (ids % 2 == 0)

    @property
    def test_mask(self) -> torch.Tensor:
        ids = torch.arange(self.n_nodes, device=self.train_mask.device)
        return ~self.train_mask & (ids % 2 == 1)


# named shapes: nodes, directed edges (incl. self loops), features, classes, train fraction; `multilabel`: every node
# has a 0/1 vector of n_class labels (BCEWithLogitsLoss + micro-F1, the reference's yelp mode, train.py:11-17,317-318)
SHAPES = {
    # BASELINE.json configs[1]
    "rmat-1m": dict(n_nodes=1_000_000, n_edges=20_000_000, n_feat=256, n_class=64, train_frac=0.66),
    # configs[0]/[2]: Reddit-shaped
    "reddit-shaped": dict(n_nodes=233_000, n_edges=115_000_000, n_feat=602, n_class=41, train_frac=0.66),
    # configs[3]
    "products-shaped": dict(n_nodes=2_400_000, n_edges=62_000_000, n_feat=100, n_class=47, train_frac=0.08),
    # configs[4]: built per rank (pipegcn_b200/distgraph.py), never as one global edge list
    "papers100m-shaped": dict(n_nodes=111_000_000, n_edges=1_600_000_000, n_feat=128, n_class=172, train_frac=0.011),
    # scripts/yelp.sh: Yelp as GraphSAINT ships it -- 716 847 nodes; 13 954 819 directed edges plus one self loop per
    # node (how the other shapes count edges) = 14 671 666; 300 features; 100 labels per node; 75 % train nodes
    "yelp-shaped": dict(n_nodes=716_847, n_edges=14_671_666, n_feat=300, n_class=100, train_frac=0.75, multilabel=True),
    # small shapes for tests / smoke
    "tiny": dict(n_nodes=300, n_edges=3_000, n_feat=20, n_class=5, train_frac=0.66),
    "small": dict(n_nodes=20_000, n_edges=400_000, n_feat=64, n_class=16, train_frac=0.66),
    # multi-label tests: 12 labels (not a multiple of 8 or 32: padded logit rows, a partial label word)
    "tiny-ml": dict(n_nodes=300, n_edges=3_000, n_feat=20, n_class=12, train_frac=0.66, multilabel=True),
}


def label_rates(n_class: int, seed: int = 5) -> torch.Tensor:
    """Positive rate p_c of every class of a multi-label shape: log-uniform in [0.01, 0.5], seeded (CPU fp32 [C]).
    A synthetic choice that gives frequent and rare labels, not Yelp's statistics."""
    gen = torch.Generator().manual_seed(seed)
    return torch.exp(torch.empty(n_class).uniform_(math.log(0.01), math.log(0.5), generator=gen))


def _rmat_pairs(n_pairs: int, scale: int, gen: torch.Generator, device, abcd=(0.57, 0.19, 0.19, 0.05)):
    a, b, c, _ = abcd
    u = torch.zeros(n_pairs, dtype=torch.int64, device=device)
    v = torch.zeros(n_pairs, dtype=torch.int64, device=device)
    for _level in range(scale):
        r = torch.rand(n_pairs, generator=gen, device=device)
        ubit = (r >= a + b)
        vbit = ((r >= a) & (r < a + b)) | (r >= a + b + c)
        u = (u << 1) | ubit.to(torch.int64)
        v = (v << 1) | vbit.to(torch.int64)
    return u, v


def rmat_edges(n_nodes: int, n_edges: int, seed: int = 0, device="cpu", max_rounds: int = 64):
    """Undirected RMAT edge set with one self loop per node.

    Returns (src, dst) with about `n_edges` directed entries: both directions of
    every unique unordered pair plus N self loops.  Vertex ids are scrambled by a
    seeded permutation so that the power-law hubs are spread over the id range.
    """
    device = torch.device(device)
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    scale = max(1, math.ceil(math.log2(max(n_nodes, 2))))
    space = 1 << scale
    perm = torch.randperm(space, generator=gen, device=device)
    want_pairs = max(0, (n_edges - n_nodes) // 2)
    keys = torch.empty(0, dtype=torch.int64, device=device)
    rounds = 0
    while keys.numel() < want_pairs and rounds < max_rounds:
        need = want_pairs - keys.numel()
        batch = int(min(max(need * 1.3, 1024), 64_000_000))
        u, v = _rmat_pairs(batch, scale, gen, device)
        u, v = perm[u], perm[v]
        ok = (u < n_nodes) & (v < n_nodes) & (u != v)
        u, v = u[ok], v[ok]
        lo, hi = torch.minimum(u, v), torch.maximum(u, v)
        new = torch.unique(lo * n_nodes + hi)
        keys = torch.unique(torch.cat([keys, new]))
        rounds += 1
    if keys.numel() > want_pairs:
        # drop a seeded random subset so that the count is exact and unbiased
        sel = torch.randperm(keys.numel(), generator=gen, device=device)[:want_pairs]
        keys = keys[sel.sort().values]
    lo, hi = keys // n_nodes, keys % n_nodes
    loops = torch.arange(n_nodes, dtype=torch.int64, device=device)
    src = torch.cat([lo, hi, loops])
    dst = torch.cat([hi, lo, loops])
    return src, dst


def make_graph(shape: str | dict, seed_graph: int = 0, seed_feat: int = 2, seed_mask: int = 3,
               device="cpu", feat_dtype=torch.float32, planted_labels: bool = False) -> GlobalGraph:
    """Build a named synthetic graph (SURVEY.md §8d seeds: graph 0, features 2, masks 3).
    `planted_labels`: labels = argmax of a fixed random linear map of (own + neighbour-mean) features instead of
    uniform noise, so that training has something to learn (accuracy tests).  Multi-label shapes: label [N, C] float32
    0/1, class c positive with rate p_c (`label_rates`); planted, where class c's score under the same kind of map
    exceeds its (1 - p_c) quantile."""
    spec = SHAPES[shape] if isinstance(shape, str) else dict(shape)
    n = spec["n_nodes"]
    src, dst = rmat_edges(n, spec["n_edges"], seed=seed_graph, device=device)
    dev = src.device
    g = torch.Generator(device=dev)
    g.manual_seed(seed_feat)
    feat = torch.randn(n, spec["n_feat"], generator=g, device=dev, dtype=torch.float32).to(feat_dtype)

    def planted_score():
        proj = torch.randn(spec["n_feat"], spec["n_class"], generator=g, device=dev)
        agg = torch.zeros(n, spec["n_feat"], device=dev).index_add_(0, dst, feat.float()[src])
        agg = agg / torch.bincount(dst, minlength=n).clamp(min=1).unsqueeze(1)
        return (feat.float() + 2.0 * agg) @ proj

    if spec.get("multilabel"):
        rate = label_rates(spec["n_class"]).to(dev)
        if planted_labels:
            score = planted_score()
            thr = torch.stack([torch.quantile(score[:, j], 1.0 - rate[j]) for j in range(spec["n_class"])])
            label = (score > thr).to(torch.float32)
        else:
            label = (torch.rand(n, spec["n_class"], generator=g, device=dev) < rate).to(torch.float32)
    else:
        label = torch.randint(0, spec["n_class"], (n,), generator=g, device=dev)
        if planted_labels:
            label = planted_score().argmax(dim=1)
    g.manual_seed(seed_mask)
    train_mask = torch.rand(n, generator=g, device=dev) < spec["train_frac"]
    if not bool(train_mask.any()):
        train_mask[0] = True
    return GlobalGraph(n, src, dst, feat, label, train_mask)


def random_partition(n_nodes: int, n_parts: int, seed: int = 1, device="cpu") -> torch.Tensor:
    """`--partition-method random` (/root/reference/helper/parser.py:41): uniform assignment."""
    gen = torch.Generator(device=torch.device(device))
    gen.manual_seed(seed)
    part = torch.randint(0, n_parts, (n_nodes,), generator=gen, device=device)
    # make sure that no part is empty on tiny graphs
    if n_nodes >= n_parts:
        part[:n_parts] = torch.arange(n_parts, device=device)
    return part


def induced_subgraph(g: GlobalGraph, keep: torch.Tensor):
    """(`g.subgraph(keep)`, original ids of its nodes): node ids compacted in ascending order (DGL `subgraph`)."""
    new_id = torch.full((g.n_nodes,), -1, dtype=torch.int64, device=g.src.device)
    ids = torch.nonzero(keep, as_tuple=True)[0]
    n = int(ids.numel())
    new_id[ids] = torch.arange(n, dtype=torch.int64, device=g.src.device)
    em = keep[g.src] & keep[g.dst]
    return GlobalGraph(n, new_id[g.src[em]], new_id[g.dst[em]], g.feat[keep], g.label[keep], g.train_mask[keep]), ids


def train_subgraph(g: GlobalGraph) -> GlobalGraph:
    """`--inductive`: the graph induced by the training nodes (`g.subgraph(g.ndata['train_mask'])`,
    /root/reference/main.py:34-35, helper/utils.py:226-230)."""
    return induced_subgraph(g, g.train_mask)[0]
