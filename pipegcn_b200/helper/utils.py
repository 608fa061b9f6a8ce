"""Data / partition helpers on the path into the hot loop.

Counterparts of /root/reference/helper/utils.py: `load_data` (:74-96),
`graph_partition` (:132-144), `load_partition` (:99-129), `get_layer_size` (:147-151).
The reference's datasets need DGL, ogb and a network; this engine accepts
`synthetic:<shape>` datasets (pipegcn_b200/synthetic.py).  The reference's own dataset
names (`reddit`, `ogbn-products`, `yelp`) are refused unless `PG_ALLOW_SYNTHETIC_FALLBACK=1`
is set, in which case the synthetic graph of the same shape (random labels!) is used.
`get_boundary` (:154-188) has no per-process counterpart: boundary lists come out of
the one-pass layout builder (pipegcn_b200/partition.py).

Partition cache: like the reference's `partitions/<graph_name>/` directory written by
`graph_partition` and read back by `load_partition` (:99-144), the node -> partition
assignment is stored on disk (`partitions/<graph_name>/part.pt`) and reused by later runs
and by the other ranks of the same run (`--skip-partition` requires it to exist).  METIS at
20 M edges takes minutes, the cached read milliseconds.
"""
import os
import time
import warnings

import torch

from ..partition import PartitionPlan, get_layer_size  # noqa: F401  (re-export)
from ..synthetic import SHAPES, make_graph, random_partition, train_subgraph

_ALIAS = {'reddit': 'reddit-shaped', 'ogbn-products': 'products-shaped', 'yelp': 'yelp-shaped'}


def _shape_of(dataset: str) -> str:
    if dataset.startswith('synthetic:'):
        return dataset.split(':', 1)[1]
    if dataset in _ALIAS:
        if os.environ.get('PG_ALLOW_SYNTHETIC_FALLBACK') != '1':
            raise ValueError(f"dataset '{dataset}' needs DGL/ogb and a download, neither of which exists here; pass "
                             f"--dataset synthetic:{_ALIAS[dataset]} (same shape, synthetic features and labels) or set "
                             f"PG_ALLOW_SYNTHETIC_FALLBACK=1 to substitute it silently")
        warnings.warn(f"dataset '{dataset}': using the synthetic graph '{_ALIAS[dataset]}' of the same shape")
        return _ALIAS[dataset]
    if dataset in SHAPES:
        return dataset
    raise ValueError('Unknown dataset: {}'.format(dataset))


def load_data(dataset, device='cpu'):
    """-> (GlobalGraph with one self loop per node, n_feat, n_class)  (utils.py:74-96); for a multi-label shape n_class
    is the width of the [N, C] label matrix (utils.py:88-91).  Not cached: the caller
    drops the global graph once its partition layout is built."""
    shape = _shape_of(dataset)
    g = make_graph(shape, device=device, planted_labels=os.environ.get('PG_PLANTED_LABELS') == '1')
    return g, g.n_feat, SHAPES[shape]['n_class']


def partition_dir(args) -> str:
    name = getattr(args, 'graph_name', '') or '%s-%d-%s-%s-%s' % (
        args.dataset, args.n_partitions, args.partition_method, getattr(args, 'partition_obj', 'vol'),
        'induc' if getattr(args, 'inductive', False) else 'trans')
    return os.path.join(os.environ.get('PG_PARTITION_ROOT', 'partitions'), str(name).replace(':', '_').replace('/', '_'))


def _compute_partition(g, args):
    if args.partition_method == 'random':
        return random_partition(g.n_nodes, args.n_partitions, seed=1, device=g.src.device)
    from ..metis import metis_partition
    return metis_partition(g, args.n_partitions, objtype=args.partition_obj)


def graph_partition(g, args, rank=0):
    """Node -> partition assignment (utils.py:132-144), through the on-disk cache: rank 0 computes and writes
    `partitions/<graph_name>/part.pt` atomically, every other rank waits for the file."""
    path = os.path.join(partition_dir(args), 'part.pt')
    use_cache = getattr(args, 'partition_cache', True) and args.partition_method != 'random'
    if not use_cache:
        if getattr(args, 'skip_partition', False) and not os.path.exists(path):
            pass                                        # random is recomputed from its seed: nothing to skip
        return _compute_partition(g, args)
    if not os.path.exists(path):
        if getattr(args, 'skip_partition', False):
            raise FileNotFoundError(f"--skip-partition: {path} does not exist (run once without it)")
        if rank == 0:
            part = _compute_partition(g, args).cpu()
            os.makedirs(os.path.dirname(path), exist_ok=True)
            tmp = path + f'.tmp{os.getpid()}'
            torch.save({'part': part.to(torch.int32), 'n_nodes': g.n_nodes, 'n_edges': g.n_edges,
                        'n_partitions': args.n_partitions, 'method': args.partition_method,
                        'obj': getattr(args, 'partition_obj', 'vol')}, tmp)
            os.replace(tmp, path)
        else:
            t0 = time.time()
            while not os.path.exists(path):
                if time.time() - t0 > float(os.environ.get('PG_PARTITION_WAIT_S', 3600)):
                    raise TimeoutError(f"rank {rank}: {path} was not written by rank 0")
                time.sleep(0.2)
    blob = torch.load(path)
    if blob['n_nodes'] != g.n_nodes or blob['n_edges'] != g.n_edges or blob['n_partitions'] != args.n_partitions:
        raise ValueError(f"{path} was written for another graph / partition count; delete it or change --graph-name")
    return blob['part'].to(torch.int64).to(g.src.device)


def load_partition(args, rank, device=None, return_graph=False):
    """This rank's `PartitionLayout` (utils.py:99-129 + the set-up half of train.run).  With `return_graph` the
    (transductive) global graph is returned too -- rank 0 evaluates on it (train.py:250-256)."""
    device = device if device is not None else (f'cuda:{torch.cuda.current_device()}' if torch.cuda.is_available() else 'cpu')
    g_full, n_feat, n_class = load_data(args.dataset, device=device)
    args.n_feat, args.n_class = n_feat, n_class
    g = train_subgraph(g_full) if getattr(args, 'inductive', False) else g_full    # main.py:34-35
    args.n_train = int(g.train_mask.sum().item())
    part = graph_partition(g, args, rank)
    layout = PartitionPlan(g, part, args.n_partitions).build(rank)
    return (layout, g_full) if return_graph else layout
