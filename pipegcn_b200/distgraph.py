"""Per-rank construction of a large synthetic graph and of this rank's `PartitionLayout`.

`PartitionPlan` (pipegcn_b200/partition.py) starts from the GLOBAL edge list, like the reference, whose every process
loads the whole DGL graph before `partition_graph` (/root/reference/helper/utils.py:132-144).  At the
ogbn-papers100M shape (111 M nodes, 1.6 B edges) no rank can hold that.  Here every rank streams the SAME seeded RMAT
pair stream in chunks and keeps only the edges whose destination it owns, so the largest array a rank ever holds is its
own ~1/P of the edges:

* node -> partition: the reference's `--partition-method random` (a seeded uniform draw, identical on all ranks);
* an undirected pair {a, b} contributes a -> b to owner(b) and b -> a to owner(a): duplicates of an edge always land
  on the same rank, so de-duplication is local;
* the graph is symmetric, hence "my rows that peer j holds as halo" (`boundary[j]`, utils.py:154-188) equals "the
  destinations of my edges whose source is owned by j" -- no communication is needed to build the send lists;
* index spaces follow partition.py exactly (reshuffled contiguous ids, halo of peer 0 | peer 1 | ..., train rows first).

Only per-node vectors of the whole graph (partition id, owner-local id, masks: a few hundred MB) are replicated.
"""
from __future__ import annotations

import math
from typing import List, Optional

import torch

from .partition import PartitionLayout, _csr_from_pairs
from .synthetic import _rmat_pairs


def _chunked_node_data(n_nodes, n_feat, n_class, mine: torch.Tensor, seed: int, dtype, device, chunk=2_000_000):
    """Features / labels of the nodes in `mine` (ascending global ids): a pure function of the global node id
    (seeded per chunk of ids), whichever rank generates them."""
    feat = torch.empty(mine.numel(), n_feat, dtype=dtype, device=device)
    label = torch.empty(mine.numel(), dtype=torch.int64, device=device)
    gen = torch.Generator(device=device)
    bounds = torch.searchsorted(mine, torch.arange(0, n_nodes + chunk, chunk, device=device))
    for c in range(bounds.numel() - 1):
        lo, hi = int(bounds[c].item()), int(bounds[c + 1].item())
        if hi == lo:
            continue
        base = c * chunk
        n = min(chunk, n_nodes - base)
        gen.manual_seed(seed * 1_000_003 + c)
        f = torch.randn(n, n_feat, generator=gen, device=device, dtype=torch.float32)
        lab = torch.randint(0, n_class, (n,), generator=gen, device=device)
        idx = mine[lo:hi] - base
        feat[lo:hi] = f[idx].to(dtype)
        label[lo:hi] = lab[idx]
    return feat, label


def build_rank_layout(spec: dict, rank: int, n_parts: int, device, world=None, seed_graph=0, seed_part=1, seed_feat=2,
                      seed_mask=3, feat_dtype=torch.float32, pair_chunk=32_000_000):
    if spec.get("multilabel"):
        raise NotImplementedError("the per-rank graph builder makes single-label graphs only; build multi-label shapes "
                                  "with synthetic.make_graph")
    dev = torch.device(device)
    n, P, r = int(spec["n_nodes"]), int(n_parts), int(rank)
    i64 = dict(dtype=torch.int64, device=dev)
    gen = torch.Generator(device=dev)

    # ---- replicated per-node vectors
    gen.manual_seed(seed_part)
    part = torch.randint(0, P, (n,), generator=gen, device=dev)
    if n >= P:
        part[:P] = torch.arange(P, device=dev)
    counts = torch.bincount(part, minlength=P)
    n_max = int(counts.max().item())
    local_id = torch.empty(n, dtype=torch.int32, device=dev)           # owner-local id (ascending global id)
    for p in range(P):
        m = part == p
        local_id[m] = torch.arange(int(counts[p].item()), dtype=torch.int32, device=dev)
    part8 = part.to(torch.int8)
    gen.manual_seed(seed_mask)
    train_mask = torch.rand(n, generator=gen, device=dev) < spec["train_frac"]
    if not bool(train_mask.any()):
        train_mask[0] = True
    n_train_global = int(train_mask.sum().item())
    inner_orig = torch.nonzero(part == r, as_tuple=True)[0]             # ascending global id
    n_in = int(inner_orig.numel())
    del part

    # ---- the seeded pair stream, filtered to edges into my nodes
    gen.manual_seed(seed_graph)
    scale = max(1, math.ceil(math.log2(max(n, 2))))
    perm = torch.randperm(1 << scale, generator=gen, device=dev)
    want_pairs = max(0, (int(spec["n_edges"]) - n) // 2)
    keys: List[torch.Tensor] = []
    done = 0
    # the stream is drawn once (no "until the exact count" loop, which would need a global count): a fraction
    # (n / 2^scale)^2 of the pairs survives the id rejection, a few percent more are duplicates
    oversample = float(spec.get("pair_oversample", 1.08))
    accept = (n / float(1 << scale)) ** 2
    to_draw = int(want_pairs * oversample / max(accept, 1e-6))
    while done < to_draw:
        batch = min(pair_chunk, to_draw - done)
        u, v = _rmat_pairs(batch, scale, gen, dev)
        u, v = perm[u], perm[v]
        ok = (u < n) & (v < n) & (u != v)
        u, v = u[ok], v[ok]
        for s, d in ((u, v), (v, u)):                                   # both directions of every pair
            mine = part8[d] == r
            keys.append(d[mine] * n + s[mine])
        done += batch
        if len(keys) >= 16:                                             # compact now and then
            keys = [torch.unique(torch.cat(keys))]
    del perm
    key = torch.unique(torch.cat(keys)) if keys else torch.empty(0, **i64)
    del keys
    ed, es = key // n, key % n
    del key
    ed = torch.cat([ed, inner_orig])                                    # one self loop per node (utils.py:94-95)
    es = torch.cat([es, inner_orig])

    # ---- move_train_first relabelling of the inner ids (train.py:139-141)
    tm = train_mask[inner_orig]
    n_tr = int(tm.sum().item())
    new_id = torch.empty(n_in, **i64)
    new_id[tm] = torch.arange(n_tr, **i64)
    new_id[~tm] = torch.arange(n_tr, n_in, **i64)

    v = new_id[local_id[ed].to(torch.int64)]
    owner = part8[es].to(torch.int64)
    is_inner = owner == r
    u = torch.empty_like(es)
    u[is_inner] = new_id[local_id[es[is_inner]].to(torch.int64)]
    hkey = owner[~is_inner] * n_max + local_id[es[~is_inner]].to(torch.int64)
    hsorted, hinv = torch.unique(hkey, return_inverse=True)
    u[~is_inner] = n_in + hinv
    n_halo = int(hsorted.numel())
    howner = hsorted // n_max
    order = torch.argsort(part8.to(torch.int16), stable=True)          # order[part_start[p] + l] = global id
    part_start = torch.zeros(P + 1, **i64)
    part_start[1:] = torch.cumsum(counts, 0)
    halo_gid = order[part_start[howner] + hsorted % n_max]
    del order
    recv_cnt = torch.bincount(howner, minlength=P)
    recv_shape: List[Optional[int]] = [None if j == r else int(recv_cnt[j].item()) for j in range(P)]
    num_all = n_in + n_halo

    # boundary[j]: my rows that j holds as halo == destinations of my edges whose source j owns (symmetric graph),
    # ascending owner-local id, then relabelled (utils.py:181, train.py:151-153)
    boundary: List[Optional[torch.Tensor]] = []
    dloc = local_id[ed].to(torch.int64)
    for j in range(P):
        boundary.append(None if j == r else new_id[torch.unique(dloc[owner == j])])
    del dloc, hkey, hinv

    indptr, indices = _csr_from_pairs(v, u, n_in, num_all)
    t_indptr, t_indices = _csr_from_pairs(u, v, num_all, n_in)
    in_deg = (indptr[1:] - indptr[:-1]).to(torch.int64)                 # every in-edge of my nodes is local
    del u, v, es, ed, owner, is_inner

    feat_o, label_o = _chunked_node_data(n, int(spec["n_feat"]), int(spec["n_class"]), inner_orig, seed_feat,
                                         feat_dtype, dev)

    def permute_rows(x):
        out = torch.empty_like(x)
        out[new_id] = x
        return out

    inner_gid = permute_rows(inner_orig)
    layout = PartitionLayout(
        rank=r, size=P, num_in=n_in, num_all=num_all, indptr=indptr, indices=indices, t_indptr=t_indptr,
        t_indices=t_indices, in_deg=in_deg, boundary=boundary, recv_shape=recv_shape, feat=permute_rows(feat_o),
        label=permute_rows(label_o), train_mask=permute_rows(tm), inner_gid=inner_gid,
        halo_gid=halo_gid, n_train_global=n_train_global)
    nnz = torch.tensor([float(layout.nnz)], dtype=torch.float64, device=dev)
    if world is not None and getattr(world, "size", 1) > 1 and not getattr(world, "is_local", False):
        world.all_reduce_sum_(nnz)
    info = dict(n_nodes=n, n_edges=int(nnz.item()), n_train=n_train_global)
    return layout, info
