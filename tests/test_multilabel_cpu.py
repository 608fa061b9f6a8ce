"""Multi-label task (the reference's yelp configuration) on the host: the oracle against outputs of the unmodified
reference, the packed label format, the multi-label synthetic shapes and the data path they travel."""
import argparse
from pathlib import Path

import pytest
import torch

from oracle import dglpart
from oracle import setup as osetup
from oracle.train import run_world
from pipegcn_b200.synthetic import SHAPES, label_rates, make_graph, random_partition, train_subgraph
from tests.ml_oracle import fixture_oracle_args, multilabel_loss

GOLDEN = Path(__file__).resolve().parent / "golden" / "multilabel"


def load_fixture(name="ref_multilabel_pp_p3.pt"):
    """(fixture, graph, partition); the fixture keeps a fingerprint of the graph's edges and features, which
    make_graph rebuilds, and its labels, train mask and partition."""
    fx = torch.load(GOLDEN / name, weights_only=False)
    gr = fx["graph"]
    g = make_graph(fx["config"]["shape"])
    assert (g.n_nodes, g.n_edges, int(g.src.sum()), int(g.dst.sum())) == \
        (gr["n_nodes"], gr["n_edges"], gr["src_sum"], gr["dst_sum"]) and float(g.feat.double().sum()) == gr["feat_sum"]
    assert torch.equal(g.label, gr["label"]) and torch.equal(g.train_mask, gr["train_mask"])
    return fx, g, gr["part"]


def test_fixture_is_the_yelp_configuration():
    fx, g, _ = load_fixture()
    c = fx["config"]
    assert (c["n_parts"], c["n_layers"], c["n_linear"], c["use_pp"], c["enable_pipeline"], c["dataset"]) == \
        (3, 4, 2, True, True, "yelp")
    assert c["shape"] == "tiny-ml" and g.label.shape == (g.n_nodes, 12)


def test_labels_pass_the_reference_setup():
    """The reference's set-up helpers (move_train_first etc.) carry the [N, 12] labels; the layout builder puts the
    same label rows in the same order."""
    from pipegcn_b200.partition import build_layouts
    fx, g, part = load_fixture()
    P = fx["config"]["n_parts"]
    for ref, L in zip((r["layout"] for r in fx["ranks"]), build_layouts(g, part, P)):
        assert (ref["num_in"], ref["num_all"], ref["recv_shape"]) == (L.num_in, L.num_all, L.recv_shape)
        assert torch.equal(ref["label"], L.label) and torch.equal(ref["train_mask"], L.train_mask)


def test_oracle_reproduces_multilabel_reference_run():
    """Per-layer exchange buffers and outputs, logits, loss and reduced gradients of every epoch, as
    test_golden_cpu.py checks the single-label fixtures (fp32, rtol 1e-5)."""
    fx, g, part = load_fixture()
    P = fx["config"]["n_parts"]
    setups = osetup.setup_world(dglpart.partition_graph(g.n_nodes, g.src, g.dst, part, P, g.feat, g.label, g.train_mask))
    forced = [ep["state"] for ep in fx["ranks"][0]["epochs"]]
    with multilabel_loss():
        traces = run_world(setups, fixture_oracle_args(fx, g), init_state=fx["ranks"][0]["init_state"],
                           forced_states=forced)
    tol = dict(rtol=1e-5, atol=1e-6)
    for r in range(P):
        for e, ep in enumerate(fx["ranks"][r]["epochs"]):
            assert set(ep["layers"]) == {0, 1}                # the graph layers; the linear tail: through the logits
            for l, rec in ep["layers"].items():
                torch.testing.assert_close(traces[r].layers[e][l]["f_buf"], rec["f_buf"], **tol)
                torch.testing.assert_close(traces[r].layers[e][l]["layer_out"], rec["layer_out"], **tol)
            torch.testing.assert_close(traces[r].logits[e], ep["logits"], **tol)
            assert abs(traces[r].losses[e] - ep["loss"]) <= 1e-5 * abs(ep["loss"])
            for n, gref in ep["grads"].items():
                torch.testing.assert_close(traces[r].grads[e][n], gref, rtol=1e-4, atol=1e-7)


@pytest.mark.parametrize("c", [1, 31, 32, 33, 100])
def test_pack_unpack_round_trip(c):
    from pipegcn_b200.ops import pack_multilabel, unpack_multilabel
    gen = torch.Generator().manual_seed(c)
    y = (torch.rand(37, c, generator=gen) < 0.4).float()
    y[0] = 1.0
    y[1] = 0.0
    w = pack_multilabel(y)
    assert w.shape == (37, (c + 31) // 32) and w.dtype == torch.int32
    assert torch.equal(unpack_multilabel(w, c), y)
    everything = unpack_multilabel(w, w.shape[1] * 32)
    assert int(everything[:, c:].sum()) == 0                     # padding bits are zero
    j = c - 1                                                    # label j is bit j % 32 of word j // 32
    bit = (w[:, j // 32].to(torch.int64) >> (j % 32)) & 1
    assert torch.equal(bit.float(), y[:, j])


def test_yelp_shaped_spec():
    s = SHAPES["yelp-shaped"]
    assert s == dict(n_nodes=716_847, n_edges=13_954_819 + 716_847, n_feat=300, n_class=100, train_frac=0.75,
                     multilabel=True)
    t = SHAPES["tiny-ml"]
    assert t["multilabel"] and t["n_class"] % 8 and t["n_class"] % 32


@pytest.mark.parametrize("planted", [False, True])
def test_multilabel_graph_is_seeded_with_the_specified_rates(planted):
    a, b = make_graph("tiny-ml", planted_labels=planted), make_graph("tiny-ml", planted_labels=planted)
    assert torch.equal(a.label, b.label) and torch.equal(a.feat, b.feat) and torch.equal(a.src, b.src)
    assert a.label.shape == (300, 12) and a.label.dtype == torch.float32
    assert set(a.label.unique().tolist()) <= {0.0, 1.0}
    # the single-label shape of the same size draws exactly what it drew before (the goldens are built from it)
    tiny = make_graph("tiny")
    assert torch.equal(tiny.feat, a.feat) and tiny.label.dim() == 1
    # rates: a larger graph of the same kind, every class within 5 sigma of p_c
    spec = dict(SHAPES["tiny-ml"], n_nodes=20_000, n_edges=200_000)
    g = make_graph(spec, planted_labels=planted)
    p = label_rates(12)
    assert float(p.min()) >= 0.01 and float(p.max()) <= 0.5
    sigma = (p * (1 - p) / spec["n_nodes"]).sqrt()
    assert bool(((g.label.mean(0) - p).abs() <= 5 * sigma + 1.0 / spec["n_nodes"]).all()), (g.label.mean(0), p)


def test_yelp_shaped_labels():
    """The full-size shape: [716 847, 100] 0/1 labels at the class rates, deterministic."""
    g = make_graph("yelp-shaped")
    assert g.label.shape == (716_847, 100) and g.n_feat == 300
    assert abs(g.n_edges - SHAPES["yelp-shaped"]["n_edges"]) <= 2
    p = label_rates(100)
    sigma = (p * (1 - p) / g.n_nodes).sqrt()
    assert bool(((g.label.mean(0) - p).abs() <= 5 * sigma).all())
    gen = torch.Generator().manual_seed(7)
    rows = torch.randint(0, g.n_nodes, (1000,), generator=gen)
    again = make_graph("yelp-shaped")
    assert torch.equal(again.label[rows], g.label[rows]) and torch.equal(again.train_mask, g.train_mask)


def test_plan_cache_and_train_subgraph_keep_label_rows_aligned(tmp_path, monkeypatch):
    from pipegcn_b200.helper import utils
    from pipegcn_b200.partition import PartitionPlan
    g = make_graph("tiny-ml")
    # a row's label travels with its features: compare against the (feature row -> node) map
    key = {tuple(f.tolist()): i for i, f in enumerate(g.feat)}

    def aligned(feat, label):
        ids = torch.tensor([key[tuple(f.tolist())] for f in feat])
        return torch.equal(label, g.label[ids])

    part = random_partition(g.n_nodes, 3)
    for r in range(3):
        L = PartitionPlan(g, part, 3).build(r)
        assert L.label.shape == (L.num_in, 12) and aligned(L.feat, L.label)
        assert torch.equal(L.label, g.label[L.inner_gid])
    sub = train_subgraph(g)
    assert sub.label.shape == (int(g.train_mask.sum()), 12) and aligned(sub.feat, sub.label)
    # the on-disk partition cache, read back by a second run that skips partitioning
    monkeypatch.setenv("PG_PARTITION_ROOT", str(tmp_path))
    args = argparse.Namespace(dataset="synthetic:tiny-ml", n_partitions=3, partition_method="metis",
                              partition_obj="vol", inductive=True, graph_name="", partition_cache=True)
    first = [utils.load_partition(args, r, device="cpu") for r in range(3)]
    args.skip_partition = True
    for r in range(3):
        L = utils.load_partition(args, r, device="cpu")
        assert torch.equal(L.label, first[r].label) and torch.equal(L.feat, first[r].feat)
        assert aligned(L.feat, L.label) and int(L.train_mask.sum()) == L.num_in    # inductive: train nodes only
    assert args.n_class == 12


def test_yelp_dataset_name(monkeypatch):
    from pipegcn_b200.helper import utils
    monkeypatch.delenv("PG_ALLOW_SYNTHETIC_FALLBACK", raising=False)
    with pytest.raises(ValueError, match="synthetic:yelp-shaped"):
        utils.load_data("yelp")
    monkeypatch.setenv("PG_ALLOW_SYNTHETIC_FALLBACK", "1")
    built = []

    def fake_make_graph(shape, **kw):                 # the shape is what matters here, not 14.7 M edges
        built.append(shape)
        return make_graph("tiny-ml", **kw)
    monkeypatch.setattr(utils, "make_graph", fake_make_graph)
    with pytest.warns(UserWarning, match="yelp-shaped"):
        g, n_feat, n_class = utils.load_data("yelp")
    assert built == ["yelp-shaped"] and n_class == 100


def test_distgraph_refuses_multilabel_shapes():
    from pipegcn_b200.distgraph import build_rank_layout
    with pytest.raises(NotImplementedError, match="single-label"):
        build_rank_layout(SHAPES["tiny-ml"], 0, 2, "cpu")
