"""GPU parity of the multi-label task (the reference's yelp configuration: BCEWithLogitsLoss(reduction='sum') and
micro-F1, train.py:11-17,317-318): the kernels against fp64 torch, the engine against the reference's own outputs
(tests/golden/multilabel) and against the oracle, scripts/yelp.sh's flags at 1/32 scale, CUDA-graph replay, and
train -> evaluate -> checkpoint."""
import argparse
import math
import os
import subprocess
import sys
import warnings
from pathlib import Path

import pytest
import torch

from tests.ml_oracle import multilabel_loss

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent

MODES = {
    "sync": dict(),
    "sync_corr": dict(feat_corr=True, grad_corr=True, corr_momentum=0.9),
    "pipeline": dict(enable_pipeline=True),
    "pipeline_corr": dict(enable_pipeline=True, feat_corr=True, grad_corr=True, corr_momentum=0.95),
}


# ---- kernels ----------------------------------------------------------------------------------------------------
def _logits(n_total, c, dtype, seed):
    """[n_total, c] logits (randn * 4 with +-30, +-100, +-1e4 planted) in rows padded with NaN columns: the padding
    must never be read into a result."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    ld = (c + 7) // 8 * 8 + 8
    full = torch.full((n_total, ld), float("nan"), dtype=dtype, device="cuda")
    z = full[:, :c]
    z.copy_(torch.randn(n_total, c, generator=gen, device="cuda") * 4)
    special = torch.tensor([30.0, -30.0, 100.0, -100.0, 1e4, -1e4], device="cuda")
    k = min(n_total * c, 6 * 64)
    idx = torch.randperm(n_total * c, generator=gen, device="cuda")[:k]
    r, col = idx // c, idx % c
    z[r, col] = special.repeat(k // 6 + 1)[:k].to(dtype)
    return z


def _labels(n_total, c, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed + 1)
    return (torch.rand(n_total, c, generator=gen, device="cuda") < 0.3).float()


def _bce_launch(z, ybits, n_rows, n_total, c, up):
    from pipegcn_b200 import _C
    code = _C.dtype_code(z.dtype)
    partial = torch.empty(_C.lib.pg_row_grid(max(n_rows, 1)) * c, dtype=torch.float32, device="cuda")
    loss = torch.full((1,), float("nan"), dtype=torch.float32, device="cuda")
    _C.check(_C.lib.pg_bce_fwd(z.data_ptr(), z.stride(0), ybits.data_ptr(), ybits.shape[1], n_rows, c, code,
                               partial.data_ptr(), loss.data_ptr(), _C.stream_ptr()), "pg_bce_fwd")
    ldg = (c + 7) // 8 * 8 + 8
    g = torch.full((n_total, ldg), float("nan"), dtype=z.dtype, device="cuda")[:, :c]
    colsum = torch.full((c,), float("nan"), dtype=torch.float32, device="cuda")
    partial2 = torch.empty(_C.lib.pg_row_grid(n_total) * c, dtype=torch.float32, device="cuda")
    upt = torch.tensor([up], dtype=torch.float32, device="cuda")
    _C.check(_C.lib.pg_bce_bwd(z.data_ptr(), z.stride(0), ybits.data_ptr(), ybits.shape[1], upt.data_ptr(), n_rows,
                               n_total, c, code, g.data_ptr(), g.stride(0), colsum.data_ptr(), partial2.data_ptr(),
                               _C.stream_ptr()), "pg_bce_bwd")
    torch.cuda.synchronize()
    return loss, g, colsum


# widest row one launch holds (fp32 512, bf16 1024) and a row cut into column chunks
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("c", [1, 12, 32, 33, 100, "widest", 1500])
@pytest.mark.parametrize("n", [0, 1, 37, 100_003])
def test_bce_kernels_match_fp64(dtype, c, n):
    from pipegcn_b200.ops import pack_multilabel
    if c == "widest":
        c = 512 if dtype == torch.float32 else 1024
    n_total, up = n + 5, -1.7
    z = _logits(n_total, c, dtype, seed=c * 7 + n)
    y = _labels(n_total, c, seed=c + n)
    ybits = pack_multilabel(y)
    loss, g, colsum = _bce_launch(z, ybits, n, n_total, c, up)
    z64, y64 = z[:n].double(), y[:n].double()                   # bf16: the reference sees the same bf16 values
    ref = (z64.clamp(min=0) - z64 * y64 + torch.log1p(torch.exp(-z64.abs()))).sum().item()
    assert abs(loss.item() - ref) <= 1e-5 * abs(ref), (loss.item(), ref)
    gref = (torch.sigmoid(z64) - y64) * up
    err = (g[:n].double() - gref).abs()
    if dtype == torch.float32:
        assert bool((err <= 2e-6 * abs(up)).all()), err.max().item()
    else:                                                        # one bf16 rounding of the fp32 value
        assert bool((err <= gref.abs() * 2.0 ** -8 + 2e-6 * abs(up)).all()), err.max().item()
    assert int(torch.count_nonzero(g[n:])) == 0 and not bool(torch.isnan(g[n:]).any())      # padding rows: exactly 0
    gs = g.double()
    cref = gs.sum(0)
    assert bool(((colsum.double() - cref).abs() <= 1e-5 * gs.abs().sum(0) + 1e-30).all())
    loss2, g2, colsum2 = _bce_launch(z, ybits, n, n_total, c, up)                             # deterministic
    assert torch.equal(loss, loss2) and torch.equal(g, g2) and torch.equal(colsum, colsum2)


def test_bce_kernels_reject_bad_arguments():
    from pipegcn_b200 import _C
    z = torch.zeros(4, 16, device="cuda")
    yb = torch.zeros(4, 1, dtype=torch.int32, device="cuda")
    out = torch.zeros(64, device="cuda")
    for c, lw in ((0, 1), (-3, 1), (40, 1)):                     # no classes; too few label words
        rc = _C.lib.pg_bce_fwd(z.data_ptr(), z.stride(0), yb.data_ptr(), lw, 4, c, _C.PG_F32, out.data_ptr(),
                               out.data_ptr(), _C.stream_ptr())
        assert rc == _C.PG_ERR_INVALID and b"pg_bce_fwd" in _C.lib.pg_last_error()
    zodd = torch.zeros(4, 5, device="cuda")                      # 20-byte rows: not 16-byte aligned
    rc = _C.lib.pg_f1_counts(zodd.data_ptr(), 5, yb.data_ptr(), 1, None, 4, 5, _C.PG_F32, out.data_ptr(),
                             _C.stream_ptr())
    assert rc == _C.PG_ERR_INVALID and b"16-byte" in _C.lib.pg_last_error()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("c", [1, 12, 100, 1500])
def test_f1_counts_match_host_and_sklearn(dtype, c):
    f1_score = pytest.importorskip("sklearn.metrics").f1_score
    from pipegcn_b200 import ops
    n_total = 5000
    z = _logits(n_total, c, dtype, seed=c)
    z[:3] = 0                                                    # z == 0 predicts negative
    y = _labels(n_total, c, seed=3 * c)
    ybits = ops.pack_multilabel(y)
    gen = torch.Generator().manual_seed(c)
    rows = torch.randperm(n_total, generator=gen)[:1234]
    for sel in (rows, None):
        counts = ops.f1_counts(z, ybits, sel).cpu()
        idx = torch.arange(n_total) if sel is None else sel
        pred, lab = (z.float().cpu()[idx] > 0), y.cpu()[idx].bool()
        host = [int((pred & lab).sum()), int((pred & ~lab).sum()), int((~pred & lab).sum())]
        assert counts.tolist() == host
        f1 = ops.multilabel_f1(z, ybits, sel)
        assert abs(f1 - f1_score(lab.numpy(), pred.numpy(), average="micro")) <= 1e-12


def test_f1_without_positives_or_predictions():
    f1_score = pytest.importorskip("sklearn.metrics").f1_score
    from pipegcn_b200 import ops
    z = -torch.ones(10, 12, device="cuda")
    y = torch.zeros(10, 12, device="cuda")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want = f1_score(y.cpu().numpy(), (z > 0).cpu().numpy(), average="micro")
    assert ops.multilabel_f1(z, ops.pack_multilabel(y)) == want == 0.0
    assert ops.f1_counts(z, ops.pack_multilabel(y), torch.zeros(0, dtype=torch.int64)).tolist() == [0, 0, 0]


# ---- engine ------------------------------------------------------------------------------------------------------
def _close(got, ref, rtol, atol_frac, what):
    scale = ref.abs().max().item()
    bad = (got - ref).abs() > atol_frac * scale + rtol * ref.abs()
    assert not bool(bad.any()), (f"{what}: {int(bad.sum())}/{bad.numel()} outside rtol {rtol} atol {atol_frac}*{scale:.3g}; "
                                 f"max err {(got - ref).abs().max().item():.3e}")


def _hooks(trainer):
    caps = [dict() for _ in trainer.engines]
    for r, eng in enumerate(trainer.engines):
        for i, layer in enumerate(eng.model.layers):
            def hook(mod, inp, out, r=r, i=i):
                caps[r][i] = ((inp[1] if len(inp) > 1 else inp[0]).detach().clone(), out.detach().clone())
            layer.register_forward_hook(hook)
    return caps


@pytest.mark.parametrize("static0", [True, False])
def test_engine_matches_multilabel_reference_golden(static0):
    """Against the unmodified reference's run of yelp.sh's structure (3 partitions, 4 layers of which 2 linear,
    --use-pp, --enable-pipeline; tests/golden/make_multilabel_golden.py), fp32, teacher-forced weights, at the
    tolerances of test_engine_matches_reference_golden."""
    from pipegcn_b200.partition import build_layouts
    from pipegcn_b200.train import LocalTrainer
    from pipegcn_b200.world import LocalWorld
    from tests.helpers import make_args
    from tests.test_multilabel_cpu import load_fixture
    fx, g, part = load_fixture()
    c = fx["config"]
    P = c["n_parts"]
    layouts = build_layouts(g, part, P)
    _, eargs = make_args(g, c["n_class"], n_epochs=c["n_epochs"], n_layers=c["n_layers"], n_hidden=c["n_hidden"],
                         n_linear=c["n_linear"], enable_pipeline=c["enable_pipeline"], use_pp=c["use_pp"])
    eargs.static_layer0 = static0
    trainer = LocalTrainer(layouts, eargs, LocalWorld(P, "cuda"), init_state=fx["ranks"][0]["init_state"], seg_len=32)
    assert all(e.multilabel for e in trainer.engines)
    caps = _hooks(trainer)
    for e in range(c["n_epochs"]):
        for eng in trainer.engines:
            eng.model.load_state_dict(fx["ranks"][0]["epochs"][e]["state"])
        losses = trainer.run_epoch(keep_logits=True)
        for r, eng in enumerate(trainer.engines):
            ep = fx["ranks"][r]["epochs"][e]
            for i, rec in ep["layers"].items():
                if i not in caps[r]:          # the linear tail runs as ops.linear, not through its module: logits below
                    continue
                if i == 0:
                    torch.testing.assert_close(caps[r][i][0].cpu(), rec["f_buf"], rtol=1e-5, atol=1e-6)
                torch.testing.assert_close(caps[r][i][0].cpu(), rec["f_buf"], rtol=2e-4, atol=2e-5)
                torch.testing.assert_close(caps[r][i][1].cpu(), rec["layer_out"], rtol=2e-4, atol=2e-4)
            torch.testing.assert_close(eng.last_logits.cpu(), ep["logits"], rtol=2e-4, atol=2e-4)
            assert abs(float(losses[r].item()) - ep["loss"]) <= 1e-4 * abs(ep["loss"])
            for n, p in eng.model.named_parameters():
                torch.testing.assert_close(p.grad.cpu(), ep["grads"][n], rtol=2e-3, atol=2e-5)


def _run(g, part, n_parts, n_epochs, dtype, free_running=False, n_class=None, **flags):
    from oracle import dglpart
    from oracle import setup as osetup
    from oracle.train import initial_state, run_world
    from pipegcn_b200.partition import build_layouts
    from pipegcn_b200.train import LocalTrainer
    from pipegcn_b200.world import LocalWorld
    from tests.helpers import make_args
    layouts = build_layouts(g, part, n_parts)
    setups = osetup.setup_world(dglpart.partition_graph(g.n_nodes, g.src, g.dst, part, n_parts, g.feat, g.label,
                                                        g.train_mask))
    oargs, eargs = make_args(g, n_class or g.label.shape[1], n_epochs=n_epochs, **flags)
    eargs.dtype = dtype
    init = initial_state(oargs)
    with multilabel_loss():
        traces = run_world(setups, oargs, init_state=init)
    trainer = LocalTrainer(layouts, eargs, LocalWorld(n_parts, "cuda"), init_state=init, seg_len=32)
    caps = _hooks(trainer)
    out = []
    for e in range(n_epochs):
        if not free_running:
            for eng in trainer.engines:
                eng.model.load_state_dict(traces[0].states[e])
        losses = trainer.run_epoch(keep_logits=True)
        out.append(dict(loss=[float(l.item()) for l in losses],
                        logits=[en.last_logits.float().cpu() for en in trainer.engines],
                        layers=[{i: (a.float().cpu(), b.float().cpu()) for i, (a, b) in cp.items()} for cp in caps],
                        grads=[{n: p.grad.detach().float().cpu().clone() for n, p in en.model.named_parameters()}
                               for en in trainer.engines]))
    return traces, out


def _tiny_ml(n_parts):
    from pipegcn_b200.synthetic import make_graph, random_partition
    g = make_graph("tiny-ml")
    return g, random_partition(g.n_nodes, n_parts)


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("n_parts", [1, 2, 4])
def test_engine_matches_oracle_fp32(n_parts, mode):
    g, part = _tiny_ml(n_parts)
    traces, out = _run(g, part, n_parts, 4, "fp32", **MODES[mode])
    for e, ep in enumerate(out):
        for r in range(n_parts):
            torch.testing.assert_close(ep["logits"][r], traces[r].logits[e], rtol=2e-4, atol=2e-4)
            assert abs(ep["loss"][r] - traces[r].losses[e]) <= 1e-4 * abs(traces[r].losses[e]) + 1e-4
            for n, gref in traces[r].grads[e].items():
                torch.testing.assert_close(ep["grads"][r][n], gref, rtol=2e-3, atol=2e-5)


@pytest.mark.parametrize("n_parts", [1, 4])
def test_engine_matches_oracle_bf16(n_parts):
    """bf16 at the tolerances of test_baseline_configs_gpu.py: rtol 2e-2, atol 1e-2 of the tensor's scale, loss 1e-2."""
    g, part = _tiny_ml(n_parts)
    traces, out = _run(g, part, n_parts, 3, "bf16", enable_pipeline=True)
    for e, ep in enumerate(out):
        for r in range(n_parts):
            _close(ep["logits"][r], traces[r].logits[e], 2e-2, 1e-2, f"epoch {e} rank {r} logits")
            assert abs(ep["loss"][r] - traces[r].losses[e]) <= 1e-2 * abs(traces[r].losses[e])


# scripts/yelp.sh at 1/32 scale: 22 401 nodes, ~458 K edges, F = 300, C = 100; --n-layers 4 --n-linear 2
# --n-hidden 512 --inductive --enable-pipeline --use-pp, 3 partitions, lr 1e-3
YELP_32 = None


def _yelp_32():
    global YELP_32
    if YELP_32 is None:
        from pipegcn_b200.synthetic import SHAPES, make_graph, random_partition, train_subgraph
        spec = dict(SHAPES["yelp-shaped"], n_nodes=716_847 // 32, n_edges=14_671_666 // 32)
        g = train_subgraph(make_graph(spec))                     # --inductive
        YELP_32 = (g, random_partition(g.n_nodes, 3))
    return YELP_32


YELP_FLAGS = dict(n_layers=4, n_linear=2, n_hidden=512, use_pp=True, enable_pipeline=True, lr=1e-3)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_yelp_sh_config_per_layer(dtype):
    g, part = _yelp_32()
    assert g.label.shape[1] == 100 and g.n_feat == 300
    traces, out = _run(g, part, 3, 3, dtype, **YELP_FLAGS)
    rt, at, lt = (2e-4, 2e-4, 1e-4) if dtype == "fp32" else (2e-2, 1e-2, 1e-2)
    for e, ep in enumerate(out):
        for r in range(3):
            for i, rec in traces[r].layers[e].items():
                if i not in ep["layers"][r]:  # linear tail: compared through the logits
                    continue
                if "f_buf" in rec:
                    _close(ep["layers"][r][i][0], rec["f_buf"], rt, at, f"epoch {e} rank {r} f_buf[{i}]")
                _close(ep["layers"][r][i][1], rec["layer_out"], rt, at, f"epoch {e} rank {r} layer_out[{i}]")
            _close(ep["logits"][r], traces[r].logits[e], rt, at, f"epoch {e} rank {r} logits")
            assert abs(ep["loss"][r] - traces[r].losses[e]) <= lt * abs(traces[r].losses[e])
            if dtype == "fp32":
                for n, gref in traces[r].grads[e].items():
                    _close(ep["grads"][r][n], gref, 2e-3, 3e-2, f"epoch {e} rank {r} grad {n}")


@pytest.mark.parametrize("dtype,tol", [("fp32", 1e-4), ("bf16", 1e-2)])
def test_yelp_sh_config_free_running(dtype, tol):
    g, part = _yelp_32()
    traces, out = _run(g, part, 3, 10, dtype, free_running=True, **YELP_FLAGS)
    for r in range(3):
        ref, got = traces[r].losses[-1], out[-1]["loss"][r]
        assert abs(got - ref) <= tol * abs(ref), f"rank {r}: final loss {got} vs oracle {ref} ({dtype})"


def test_yelp_sh_config_with_dropout():
    """yelp.sh's --dropout 0.1 (no oracle counterpart: the masks are the engine's own): finite, decreasing loss."""
    from pipegcn_b200.partition import build_layouts
    from pipegcn_b200.train import LocalTrainer
    from pipegcn_b200.world import LocalWorld
    from tests.helpers import make_args
    g, part = _yelp_32()
    _, eargs = make_args(g, 100, n_epochs=20, dropout=0.1, **YELP_FLAGS)
    eargs.dtype = "bf16"
    trainer = LocalTrainer(build_layouts(g, part, 3), eargs, LocalWorld(3, "cuda"))
    losses = [sum(float(l.item()) for l in trainer.run_epoch()) for _ in range(20)]
    assert all(math.isfinite(l) for l in losses)
    assert losses[-1] < 0.9 * losses[0], losses


@pytest.mark.parametrize("mode", ["sync", "pipeline_corr"])
def test_cuda_graph_replay_equals_eager(mode):
    """Replayed multi-label epochs (BCE forward and backward inside the captured graph) produce the oracle's
    logits, loss and gradients, as eagerly launched ones do."""
    from oracle.train import initial_state, run_world
    from pipegcn_b200.train import RankEngine
    from pipegcn_b200.world import LocalWorld
    from tests.helpers import make_args, small_world
    g, _, layouts, setups = small_world("tiny-ml", 1)
    n_epochs = 7
    oargs, eargs = make_args(g, 12, n_epochs=n_epochs, **MODES[mode])
    init = initial_state(oargs)
    with multilabel_loss():
        traces = run_world(setups, oargs, init_state=init)
    eargs.cuda_graph = True
    eng = RankEngine(layouts[0], eargs, LocalWorld(1, "cuda").view(0), init_state=init, seg_len=32)
    eng.keep_logits = True
    for e in range(n_epochs):
        if e == 3:
            eng.capture()
        eng.model.load_state_dict(traces[0].states[e])
        loss = eng.run_epoch()
        torch.testing.assert_close(eng.last_logits.float().cpu(), traces[0].logits[e], rtol=2e-4, atol=2e-4)
        assert abs(float(loss.item()) - traces[0].losses[e]) <= 1e-4 * abs(traces[0].losses[e])
        for n, p in eng.model.named_parameters():
            torch.testing.assert_close(p.grad.cpu(), traces[0].grads[e][n], rtol=2e-3, atol=2e-5)


def test_prefetched_packed_labels_and_non_prefix_train_rows():
    """The host-buffer input path carries the packed train labels; a layout whose train rows do not come first is
    refused instead of being trained through a second loss path."""
    from pipegcn_b200 import ops
    from pipegcn_b200._C import PgError
    from pipegcn_b200.train import RankEngine
    from pipegcn_b200.world import LocalWorld
    from tests.helpers import make_args, small_world
    g, _, layouts, _ = small_world("tiny-ml", 1)
    _, eargs = make_args(g, 12, enable_pipeline=True)
    L = layouts[0]
    eng = RankEngine(L, eargs, LocalWorld(1, "cuda").view(0))
    want = ops.pack_multilabel(L.label[:eng.part_train].cuda())
    assert torch.equal(eng.labels, want)
    l0 = eng.run_epoch()
    flipped = ops.pack_multilabel(1.0 - L.label[:eng.part_train]).pin_memory()
    slot = eng.prefetch_features(L.feat.pin_memory(), label_host=flipped)
    eng.commit_features(slot)
    l1 = eng.run_epoch()
    torch.cuda.synchronize()
    assert torch.equal(eng.labels.cpu(), flipped) and math.isfinite(float(l1)) and float(l1) != float(l0)
    L.train_mask = L.train_mask.roll(1)
    with pytest.raises(PgError, match="train rows first"):
        RankEngine(L, eargs, LocalWorld(1, "cuda").view(0))


def test_train_eval_checkpoint_roundtrip(tmp_path, monkeypatch):
    """train.run with --eval on a planted multi-label graph: micro-F1 lines in the results file, validation F1 rises,
    the best state_dict loads strictly into the oracle's modules and the oracle's sklearn F1 of it agrees with the
    engine's."""
    f1_score = pytest.importorskip("sklearn.metrics").f1_score
    import torch.nn.functional as F
    from oracle.model import OracleGraphSAGE
    from oracle.train import run_world
    from pipegcn_b200 import train
    from pipegcn_b200.helper import context as ctx
    from pipegcn_b200.helper.feature_buffer import Buffer
    from pipegcn_b200.helper.reducer import Reducer
    from pipegcn_b200.partition import build_layouts, get_layer_size
    from pipegcn_b200.synthetic import make_graph
    from pipegcn_b200.world import LocalWorld
    from tests.helpers import make_args, small_world
    monkeypatch.chdir(tmp_path)
    spec = dict(n_nodes=3_000, n_edges=30_000, n_feat=24, n_class=12, train_frac=0.6, multilabel=True)
    g = make_graph(spec, planted_labels=True)
    layout = build_layouts(g, torch.zeros(g.n_nodes, dtype=torch.int64), 1)[0]
    args = argparse.Namespace(
        model="graphsage", backend="nccl", dtype="fp32", n_layers=2, n_hidden=32, n_linear=0, n_feat=24, n_class=12,
        n_train=int(g.train_mask.sum()), dropout=0.1, norm="layer", lr=1e-2, weight_decay=0.0, use_pp=False,
        enable_pipeline=False, feat_corr=False, grad_corr=False, corr_momentum=0.95, seed=0, n_epochs=30, log_every=1,
        n_partitions=1, eval=True, inductive=False, dataset="synthetic:test", graph_name="roundtrip_ml")
    world = LocalWorld(1, "cuda").view(0)
    ctx.buffer, ctx.reducer = Buffer(world), Reducer(world)
    eng = train.run(layout, args, world, eval_graph=g)
    text = next((tmp_path / "results").iterdir()).read_text().splitlines()
    assert len(text) == 30 and text[0].startswith("Epoch 00000 | Validation Accuracy")
    val = [float(t.split("Validation Accuracy ")[1].split("%")[0]) / 100 for t in text]
    assert val[-1] > val[0], val
    state = torch.load(tmp_path / eng.checkpoint_path)
    ref_model = OracleGraphSAGE(get_layer_size(24, 32, 12, 2), F.relu, False, norm="layer", dropout=0.1)
    ref_model.load_state_dict(state, strict=True)
    # the oracle's forward of the un-partitioned graph from the checkpoint (lr 0, dropout 0), scored by sklearn
    _, _, layouts, setups = small_world(spec, 1)
    oargs, _ = make_args(g, 12, n_epochs=1, n_layers=2, n_hidden=32, lr=0.0)
    with multilabel_loss():
        logits = run_world(setups, oargs, init_state=state)[0].logits[0]
    order = layouts[0].inner_gid
    vm = g.val_mask[order]
    ref_f1 = f1_score(g.label[order][vm].numpy(), (logits[vm] > 0).numpy(), average="micro")
    assert abs(ref_f1 - eng.best_val_acc) <= 1e-3, (ref_f1, eng.best_val_acc)


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_two_ranks_match_oracle_multilabel():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29541", str(ROOT / "tools" / "dist_parity.py"), "tiny-ml"]
    p = subprocess.run(cmd, cwd=ROOT, env=dict(os.environ), capture_output=True, text=True, timeout=900)
    assert p.returncode == 0 and "ALL OK" in p.stdout, p.stdout[-3000:] + p.stderr[-3000:]
