"""Per-rank trainer: the epoch loop around the hot path.

Keeps the entry points of /root/reference/train.py -- `init_processes(rank, size, args)`
(:408-416) and `run(...)` (:242-400) -- and the order of an epoch (:341-362):
forward, summed cross-entropy on the local train rows (softmax, or sigmoid for a
multi-label task, :317-320), backward (which runs the
gradient halo exchange), `buffer.next_epoch()`, `reducer.synchronize()`, Adam step.
The DGL partition arguments of the reference's `run(graph, node_dict, gpb, args)` are
replaced by a `PartitionLayout` (pipegcn_b200/partition.py); evaluation and
checkpointing (train.py:20-61,377-400) run on the GPU with the same kernels (pipegcn_b200/evaluate.py).

`RankEngine` is one rank; `LocalTrainer` steps several simulated ranks of a
`LocalWorld` in lock-step on one GPU (each on its own stream).
"""
from __future__ import annotations

import os
import time
from typing import List, Optional

import numpy as np
import torch
import torch.nn.functional as F

from .graph import PartGraph
from .helper import context as ctx
from .helper.feature_buffer import Buffer
from .helper.reducer import Reducer
from .helper.timer.comm_timer import CommTimer
from .module.model import GraphSAGE
from .partition import PartitionLayout, get_layer_size


def create_model(layer_size, args, buffer=None, dtype=torch.float32):
    if args.model in ('graphsage', 'gcn'):
        return GraphSAGE(layer_size, F.relu, args.use_pp, norm=args.norm, dropout=args.dropout,
                         n_linear=args.n_linear, train_size=args.n_train, buffer=buffer, dtype=dtype)
    raise NotImplementedError(args.model)


def reduce_hook(reducer, param, name, n_train):
    def fn(grad):
        reducer.reduce(param, name, grad, n_train)
    return fn


def act_dtype(args):
    return torch.bfloat16 if getattr(args, 'dtype', 'fp32') in ('bf16', 'bfloat16') else torch.float32


class RankEngine:
    """Everything one rank owns: graph, exchange buffer, model replica, reducer, optimiser."""

    def __init__(self, layout: PartitionLayout, args, world, buffer: Optional[Buffer] = None,
                 reducer: Optional[Reducer] = None, init_state=None, seg_len=None):
        self.args, self.world, self.rank = args, world, world.rank
        dev = world.device
        self.device = dev
        self.dtype = act_dtype(args)
        self.graph = PartGraph.from_layout(layout, device=dev, seg_len=seg_len)
        self.in_deg = self.graph.in_deg
        self.layer_size = get_layer_size(args.n_feat, args.n_hidden, args.n_class, args.n_layers)
        self.buffer = buffer if buffer is not None else Buffer(world)
        if buffer is None:
            self.buffer.timer = CommTimer()
        self.buffer.init_buffer(layout.num_in, layout.num_all, layout.boundary, layout.recv_shape,
                                self.layer_size[:args.n_layers - args.n_linear], use_pp=args.use_pp,
                                backend=args.backend, pipeline=args.enable_pipeline, corr_feat=args.feat_corr,
                                corr_grad=args.grad_corr, corr_momentum=args.corr_momentum,
                                dtype=self.dtype, world=world,
                                static_layer0=bool(getattr(args, 'static_layer0', True)))
        self.feat = layout.feat.to(dev).to(self.dtype)
        self._pp = None
        if args.use_pp:
            self.pp_begin(layout)
            if not getattr(world, 'is_local', False) or world.size == 1:
                self.pp_end()
                self.release_pp()
        else:
            # the static input features live in the exchange buffer of layer 0 (all versions): update(0, .) copies nothing
            self.buffer.load_inner(0, self.feat)
            if not getattr(world, 'is_local', False) or world.size == 1:
                self.static0()          # LocalWorld ranks: `LocalTrainer` runs the two phases over all ranks
        tm = layout.train_mask.to(dev)
        self.part_train = int(tm.sum().item())
        prefix = bool(tm[:self.part_train].all().item()) if self.part_train else True
        self.train_sel = slice(0, self.part_train) if prefix else tm
        # multi-label task (the reference's yelp mode, train.py:317-318): [N, C] 0/1 labels, summed sigmoid
        # cross-entropy; the train rows' labels are kept bit-packed (ops.pack_multilabel)
        self.multilabel = layout.label.dim() == 2
        if self.multilabel:
            from . import ops
            if not prefix:
                from ._C import PgError
                raise PgError("multi-label training needs the train rows first (move_train_first layout)")
            self.labels = ops.pack_multilabel(layout.label[:self.part_train].to(dev))
        else:
            self.labels = layout.label.to(dev)[tm]
        torch.manual_seed(args.seed)                                      # train.py:298
        self.model = create_model(self.layer_size, args, buffer=self.buffer, dtype=self.dtype)
        if init_state is not None:
            self.model.load_state_dict(init_state)
        self.model.to(dev)
        self.reducer = reducer if reducer is not None else Reducer(world)
        self.reducer.init(self.model, world)
        for name, p in self.model.named_parameters():
            p.register_hook(reduce_hook(self.reducer, p, name, args.n_train))
        self.loss_fcn = torch.nn.CrossEntropyLoss(reduction='sum')        # train.py:320
        self.use_graph = bool(getattr(args, 'cuda_graph', False))
        # the reference's optimiser (train.py:321-323); `fused`: torch's single-kernel implementation of the same update
        # (one launch instead of seven foreach kernels per step -- 0.17 ms of a 3.3 ms step at 8 GPUs)
        self.optimizer = torch.optim.Adam(self.model.parameters(), lr=args.lr, weight_decay=args.weight_decay,
                                          capturable=self.use_graph, fused=bool(getattr(args, 'fused_adam', True)))
        self.graphs = None
        self.epoch = 0
        self.last_logits = None
        self.keep_logits = False

    # ------------------------------------------------------------------ --use-pp (train.py:169-189)
    def pp_begin(self, layout):
        """One-shot exchange of the raw boundary features through the push kernel (first half of `precompute`)."""
        from .graph import alloc_rows
        pp = Buffer(self.world)
        pp.timer = CommTimer()
        pp.init_buffer(layout.num_in, layout.num_all, layout.boundary, layout.recv_shape, [self.args.n_feat],
                       backend=self.args.backend, pipeline=False, dtype=self.dtype, world=self.world,
                       key='pipegcn.buffer.pp')
        self._pp = pp
        self._pp_started = False

    def _pp_push(self):
        pp = self._pp
        pp._connect()
        d = self.args.n_feat
        feat = self.feat if self.feat.stride(1) == 1 else self.feat.contiguous()
        pp._push(pp._self_msgs[(0, 0)], feat, d, 0)
        pp._push(pp._fwd_msgs[(0, 0)], feat, d, 1)
        self._pp_started = True

    def pp_end(self):
        """Wait for the peers' rows, neighbour mean, feat <- cat(feat, mean) (second half of `precompute`).  With
        several LocalWorld ranks in one process every rank must have pushed before any rank waits
        (`LocalTrainer` calls `_pp_push` on all engines first)."""
        from . import ops
        from .graph import alloc_rows
        pp = self._pp
        if not self._pp_started:
            self._pp_push()
        pp._wait_flags(0, 0, 1, 'forward_0')
        d = self.args.n_feat
        merged = pp._f_buf[(0, 0)][:, :d]
        mean = ops.aggregate(self.graph.fwd, merged, row_div=self.graph.in_deg_f)
        both = alloc_rows(self.graph.num_in, 2 * d, self.dtype, self.device)
        both[:, :d].copy_(self.feat)
        both[:, d:].copy_(mean)
        self.feat = both
        torch.cuda.synchronize()
        pp.check_status()
        self._pp_done = pp                 # peers may still be reading its heap: freed by `release_pp`
        self._pp = None

    def release_pp(self):
        """Free the one-shot --use-pp exchange heap (collective for a DistWorld: every rank calls it after its
        `pp_end`; for LocalWorld ranks call it once every rank has finished `pp_end`)."""
        pp = getattr(self, '_pp_done', None)
        if pp is not None:
            pp.release()
            self._pp_done = None

    def static0(self, phase=None):
        """One-shot exchange of the static layer-0 halo rows (SURVEY.md §8f-2); `phase` 'begin' / 'end' / both."""
        if self.args.use_pp:
            return
        if phase in (None, 'begin'):
            self.buffer.static0_begin(self.buffer._f_buf[(0, 0)][:self.buffer._num_in, :self.args.n_feat])
        if phase in (None, 'end'):
            self.buffer.static0_end()

    def forward_backward(self, keep_logits=False):
        """train.py:343-355; returns the summed loss (device tensor, no host sync)."""
        self.model.train()
        feat = self.buffer.inner_view(0)
        logits = self.model(self.graph, feat if feat is not None else self.feat, self.in_deg)
        if self.multilabel:
            from . import ops
            loss = ops.bce_with_logits_sum(logits, self.labels, self.part_train, self.args.n_class)
        elif isinstance(self.train_sel, slice) and logits.dtype in (torch.float32, torch.bfloat16):
            from . import ops
            loss = ops.cross_entropy_sum(logits, self.labels, self.part_train)      # fused softmax-CE (sum)
        else:
            loss = self.loss_fcn(logits[self.train_sel].float(), self.labels)
        if keep_logits or self.keep_logits:
            self.last_logits = logits.detach()
        self.optimizer.zero_grad(set_to_none=True)
        from . import ops as _ops
        _ops.reset_colsum()
        loss.backward()
        return loss.detach()

    def set_features(self, feat):
        """New input features for the coming epoch (host or device tensor, [N_in, n_feat])."""
        if self.buffer.inner_view(0) is not None:
            # layer 0 lives in the exchange buffer, one copy per version (epoch parity): refresh all of them
            self.buffer.load_inner(0, feat.to(self.device, non_blocking=True) if not feat.is_cuda else feat)
            self.static0()          # new features: their halo rows have to be exchanged again
            return
        # --use-pp: `self.feat` is cat(feat, neighbour mean) (train.py:169-189); the raw half is refreshed, the mean is
        # set-up work of the reference (precompute runs once, train.py:287-288) and is not recomputed per step
        dst = self.feat[:, :feat.shape[1]]
        if feat.is_cuda and feat.dtype == dst.dtype:
            torch.mul(feat, 1, out=dst)
        else:
            dst.copy_(feat, non_blocking=True)

    # ---- input pipeline: the next epoch's features travel host -> device while this epoch computes
    def prefetch_features(self, feat_host, label_host=None) -> int:
        """Start the asynchronous copy of a [N_in, n_feat] pinned host tensor (and optionally the train labels, in the
        format of `self.labels`: bit-packed words for a multi-label task) into one of two staging buffers on a copy
        stream; returns the slot to hand to `commit_features`."""
        if not hasattr(self, '_stage'):
            self._stage_lab = [torch.empty_like(self.labels) for _ in range(2)]
            n_feat = feat_host.shape[1]
            self._stage = [torch.empty(feat_host.shape[0], n_feat, dtype=self.dtype, device=self.device) for _ in range(2)]
            self._copy_stream = torch.cuda.Stream(device=self.device)
            self._staged = [torch.cuda.Event(), torch.cuda.Event()]
            self._consumed = [torch.cuda.Event(), torch.cuda.Event()]
            self._stage_n = 0
        slot = self._stage_n % 2
        self._stage_n += 1
        with torch.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(self._consumed[slot])        # the epoch that last read this slot has taken it
            self._stage[slot].copy_(feat_host, non_blocking=True)
            if label_host is not None:
                self._stage_lab[slot].copy_(label_host, non_blocking=True)
            self._stage_has_lab = label_host is not None
            self._staged[slot].record()
        return slot

    def commit_features(self, slot: int):
        """Make the staged features of `slot` the input of the coming epoch (device-to-device, on the compute stream)."""
        cur = torch.cuda.current_stream()
        cur.wait_event(self._staged[slot])
        self.set_features(self._stage[slot])
        if getattr(self, '_stage_has_lab', False):
            torch.add(self._stage_lab[slot], 0, out=self.labels)     # SM kernel (see Buffer.load_inner)
        self._consumed[slot].record(cur)

    def finish_epoch(self, reduce=True):
        """train.py:357-362."""
        self.buffer.next_epoch()
        if reduce:
            self.reducer.synchronize()
        self.optimizer.step()
        self.epoch += 1

    def run_epoch(self):
        if self.graphs is not None:
            return self.replay()
        self.buffer.timer.clear()            # sections are per epoch (comm_timer.py:14-15 raises on duplicates)
        loss = self.forward_backward()
        self.finish_epoch()
        return loss

    # ------------------------------------------------------------------ CUDA graphs
    def capture(self):
        """Capture one whole epoch (forward, loss, backward with both halo exchanges, gradient all-reduce, Adam
        step) into a CUDA graph -- two graphs with --enable-pipeline, one per epoch parity, because the exchange
        buffers alternate.  Everything that changes from epoch to epoch is read from the device: the epoch counter
        behind the flag values (`Buffer._epoch_dev`) and the dropout step.  Call after >= 3 eager epochs."""
        from . import ops
        assert self.epoch >= 3, "run a few eager epochs first (allocator, lazy handles, steady-state control flow)"
        assert self.use_graph, "create the engine with args.cuda_graph=True (capturable optimizer)"
        self.buffer.graph_mode = True
        self.buffer._push_done.clear()
        ops.STEP_DEV = self.buffer._epoch_dev
        torch.cuda.synchronize()
        graphs = []
        pool = None
        for _ in range(2 if self.args.enable_pipeline else 1):
            g = torch.cuda.CUDAGraph()
            self.optimizer.zero_grad(set_to_none=True)
            with torch.cuda.graph(g, pool=pool):
                loss = self.forward_backward()
                self.finish_epoch()
            pool = g.pool()
            graphs.append((g, loss, self.last_logits, [p.grad for p in self.model.parameters()]))
        torch.cuda.synchronize()
        self.graphs, self._replays = graphs, 0
        return self

    def replay(self):
        g, loss, logits, grads = self.graphs[self._replays % len(self.graphs)]
        g.replay()
        self._replays += 1
        self.last_logits = logits
        for p, gr in zip(self.model.parameters(), grads):     # each graph owns its gradient tensors
            p.grad = gr
        return loss


class LocalTrainer:
    """Lock-step driver of all ranks of a LocalWorld on one GPU (one stream per rank)."""

    def __init__(self, layouts: List[PartitionLayout], args, local_world, init_state=None, seg_len=None):
        self.streams = [torch.cuda.Stream(device=local_world.device) for _ in layouts]
        if len(layouts) > 1 and not args.enable_pipeline:
            self._dry_run(layouts, args, local_world, seg_len)
        self.world = local_world
        self.engines = [RankEngine(l, args, local_world.view(r), init_state=init_state, seg_len=seg_len)
                        for r, l in enumerate(layouts)]
        if args.use_pp and len(layouts) > 1:          # all ranks push before any rank waits (one host thread)
            for e, s in zip(self.engines, self.streams):
                with torch.cuda.stream(s):
                    e._pp_push()
            for e, s in zip(self.engines, self.streams):
                with torch.cuda.stream(s):
                    e.pp_end()
            for e in self.engines:
                e.release_pp()
        if not args.use_pp and len(layouts) > 1:      # static layer-0 halo: all ranks push before any rank waits
            for ph in ('begin', 'end'):
                for e, s in zip(self.engines, self.streams):
                    with torch.cuda.stream(s):
                        e.static0(ph)
            torch.cuda.synchronize()
        for e in self.engines:
            e.buffer.timeout_ms = 5000

    def _dry_run(self, layouts, args, local_world, seg_len):
        """One GPU, one process, non-pipelined exchange: a rank's flag-wait kernel spins until its peers'
        pushes are LAUNCHED by this same host thread, so nothing on the host may synchronise with the
        device in between (lazy module loading, first-use handle creation, allocator growth).  Two
        throw-away pipelined epochs (which never wait on unlaunched work) on the same streams trigger
        all of that first.  Real multi-GPU runs (one process per GPU) do not need this."""
        import copy
        from .world import LocalWorld
        dry_args = copy.copy(args)
        dry_args.enable_pipeline = True
        dry = LocalTrainer.__new__(LocalTrainer)
        dry.world = LocalWorld(local_world.size, local_world.device)
        dry.streams = self.streams
        dry.engines = [RankEngine(l, dry_args, dry.world.view(r), seg_len=seg_len) for r, l in enumerate(layouts)]
        rng = torch.cuda.get_rng_state(local_world.device)
        for _ in range(2):
            dry.run_epoch()
        torch.cuda.synchronize()
        for e in dry.engines:
            e.buffer._heap.free()
        torch.cuda.set_rng_state(rng, local_world.device)
        del dry

    def run_epoch(self, keep_logits=False):
        cur = torch.cuda.current_stream()
        losses = []
        for e in self.engines:
            e.buffer.timer.clear()
        for e, s in zip(self.engines, self.streams):
            s.wait_stream(cur)
            with torch.cuda.stream(s):
                losses.append(e.forward_backward(keep_logits))
        for e, s in zip(self.engines, self.streams):
            with torch.cuda.stream(s):
                e.buffer.next_epoch()
                e.reducer.pack()
        for s in self.streams:
            cur.wait_stream(s)
        total = self.engines[0].reducer._flat.clone()
        for e in self.engines[1:]:
            total += e.reducer._flat
        for e in self.engines:
            e.reducer._flat.copy_(total)
            e.reducer.unpack()
            e.optimizer.step()
            e.epoch += 1
        for e in self.engines:
            e.buffer.check_status()
        return losses


def run(layout: PartitionLayout, args, world=None, eval_graph=None):
    """One rank's training loop with the reference's log line, evaluation and checkpoint (train.py:341-400).
    `eval_graph`: the global graph rank 0 evaluates on every `log_every` epochs when `args.eval` is set."""
    if world is None:
        from .world import default_world
        world = default_world()
    rank = world.rank
    engine = RankEngine(layout, args, world, buffer=ctx.buffer, reducer=ctx.reducer)
    timer = engine.buffer.timer
    do_eval = bool(getattr(args, 'eval', False)) and rank == 0
    eval_set = best = result_file_name = None
    if do_eval:
        if eval_graph is None:
            raise ValueError("run(..., eval_graph=None) with args.eval set: rank 0 needs the global graph "
                             "(load_partition(..., return_graph=True)) or pass --no-eval")
        from .evaluate import BestModel, EvalSet, evaluate_induc, evaluate_trans, result_file
        eval_set = EvalSet(eval_graph, engine.device, inductive=getattr(args, 'inductive', False), dtype=engine.dtype)
        best = BestModel()
        os.makedirs('checkpoint/', exist_ok=True)                         # train.py:258-260
        os.makedirs('results/', exist_ok=True)
        result_file_name = result_file(args)
    del eval_graph
    train_dur, comm_dur, reduce_dur = [], [], []
    for epoch in range(args.n_epochs):
        torch.cuda.synchronize()
        t0 = time.time()
        loss = engine.forward_backward()
        engine.buffer.next_epoch()
        torch.cuda.synchronize()
        pre_reduce = time.time()
        engine.reducer.synchronize()
        torch.cuda.synchronize()
        reduce_time = time.time() - pre_reduce
        engine.optimizer.step()
        torch.cuda.synchronize()
        if epoch >= 5 and epoch % args.log_every != 0:                    # train.py:364-367
            train_dur.append(time.time() - t0)
            comm_dur.append(timer.tot_time())
            reduce_dur.append(reduce_time)
        if (epoch + 1) % 10 == 0:
            print("Process {:03d} | Epoch {:05d} | Time(s) {:.4f} | Comm(s) {:.4f} | Reduce(s) {:.4f} | Loss {:.4f}".format(
                rank, epoch, np.mean(train_dur) if train_dur else float('nan'),
                np.mean(comm_dur) if comm_dur else float('nan'),
                np.mean(reduce_dur) if reduce_dur else float('nan'), loss.item() / max(engine.part_train, 1)))
        timer.clear()
        engine.buffer.check_status()
        if do_eval and (epoch + 1) % args.log_every == 0:                 # train.py:377-390
            name = 'Epoch %05d' % epoch
            if not eval_set.inductive:
                val_acc = evaluate_trans(name, engine.model, eval_set.val, result_file_name)
            else:
                val_acc = evaluate_induc(name, engine.model, eval_set.val, 'val', result_file_name)
            best.offer(val_acc, engine.model)
    engine.buffer.synchronize()
    if do_eval and best.state is not None:                                # train.py:392-400
        path = best.save(args)
        print('model saved')
        print("Validation accuracy {:.2%}".format(best.acc))
        final = create_model(engine.layer_size, args, buffer=engine.buffer, dtype=engine.dtype).to(engine.device)
        final.load_state_dict(best.state)
        engine.test_acc = evaluate_induc('Test Result', final, eval_set.test, 'test')
        engine.best_val_acc, engine.checkpoint_path = best.acc, path
    return engine


def check_parser(args):
    if args.norm == 'none':
        args.norm = None


def init_processes(rank, size, args):
    """Initialise the distributed environment and train this rank (train.py:408-416)."""
    os.environ['MASTER_ADDR'] = args.master_addr
    os.environ['MASTER_PORT'] = '%d' % args.port
    import torch.distributed as dist
    if args.backend not in ('nccl', 'nvlink'):
        raise NotImplementedError("backend '%s': this engine implements the NVLink/NCCL path only" % args.backend)
    if size > torch.cuda.device_count() or getattr(args, 'node_rank', 0) > 0 \
            or size > getattr(args, 'parts_per_node', size):
        # peer heaps are mapped with CUDA IPC, which does not cross nodes
        raise NotImplementedError(f"single-node only: {size} partitions need {size} GPUs of ONE node "
                                  f"({torch.cuda.device_count()} visible, --parts-per-node "
                                  f"{getattr(args, 'parts_per_node', size)}, --node-rank {getattr(args, 'node_rank', 0)})")
    torch.cuda.set_device(rank)
    # 'nvlink' names the halo path; the process group (gradient all-reduce, handle exchange) is always NCCL
    dist.init_process_group('nccl', rank=rank, world_size=size, device_id=torch.device('cuda', rank))
    check_parser(args)
    from .helper.utils import load_partition
    want_graph = bool(getattr(args, 'eval', False)) and rank == 0
    out = load_partition(args, rank, return_graph=want_graph)
    layout, g_full = out if want_graph else (out, None)
    try:
        return run(layout, args, eval_graph=g_full)
    finally:
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
