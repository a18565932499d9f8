"""CPU: host-side logic — the DGLGraph subset, the synthetic generator, the module's reference
API surface (ctor, hparams, state_dict names) and the no-fallback rule."""
import numpy as np
import pytest
import torch

import deepdfa_b200 as D
from deepdfa_b200 import batched_graph as G
from deepdfa_b200 import synth
from deepdfa_b200._lib import DdfaError
from oracle import ggnn_oracle as O

FEAT = "_ABS_DATAFLOW_api_all_limitall_1000_limitsubkeys_1000"


def test_graph_and_self_loop_like_dgl():
    g = D.graph(([1, 2, 2], [0, 0, 1]))          # dbize_graphs.py:24
    assert g.num_nodes() == 3 and g.num_edges() == 3 and g.batch_size == 1
    g2 = D.add_self_loop(g)                       # dbize_graphs.py:25
    src, dst = g2.edges()
    assert g2.num_edges() == 6
    assert torch.equal(src[-3:], torch.arange(3)) and torch.equal(dst[-3:], torch.arange(3))


def test_batch_unbatch_roundtrip():
    gs = [synth.make_batch(sizes=[n], input_dim=40, seed=i) for i, n in enumerate([3, 1, 8, 2])]
    b = D.batch(gs)
    assert b.batch_size == 4 and b.num_nodes() == 14
    assert b.batch_num_nodes().tolist() == [3, 1, 8, 2]
    assert b.batch_num_edges().tolist() == [x.num_edges() for x in gs]
    back = D.unbatch(b)
    for x, y in zip(gs, back):
        assert torch.equal(x.edges()[0], y.edges()[0]) and torch.equal(x.edges()[1], y.edges()[1])
        for k in x.ndata:
            assert torch.equal(x.ndata[k], y.ndata[k])


def test_collate_matches_graphdataloader_contract():
    gs = [(synth.make_batch(sizes=[n], input_dim=40, seed=i), {}) for i, n in enumerate([3, 5])]
    bg, extra = D.collate(gs)                     # consumer: base_module.py:172
    assert bg.batch_size == 2 and extra == {}


def test_ndata_row_check_and_errors():
    with pytest.raises(ValueError):
        G.BatchedCFG(torch.tensor([0]), torch.tensor([0]), torch.tensor([2]), {"x": torch.zeros(3)})
    with pytest.raises(ValueError):
        D.batch([])
    with pytest.raises(TypeError):
        D.as_batched_cfg(object())


def test_synth_is_bigvul_shaped_and_deterministic():
    g = synth.make_batch(256, 150, seed=0)
    assert (g.num_nodes(), g.num_edges(), g.batch_size) == (38400, 76800, 256)   # config C0 (SURVEY.md §8)
    src, dst = g.edges()
    assert int((src == dst).sum()) >= g.num_nodes()            # one self loop per node
    gid = torch.repeat_interleave(torch.arange(256), g.batch_num_nodes())
    assert torch.equal(gid[src], gid[dst])                      # block-diagonal adjacency
    idx = g.ndata["_ABS_DATAFLOW_api"]
    assert idx.dtype == torch.int64 and 0.70 < float((idx == 0).float().mean()) < 0.80
    assert int(idx.max()) < 1002
    zero_mask = [g.ndata[f"_ABS_DATAFLOW_{k}"] == 0 for k in D.allfeats]
    assert all(torch.equal(zero_mask[0], z) for z in zero_mask)  # subkeys share the not-a-definition mask
    assert g.ndata["_VULN"].dtype == torch.int32
    g2 = synth.make_batch(256, 150, seed=0)
    assert torch.equal(g2.edges()[0], src) and torch.equal(g2.ndata["_ABS_DATAFLOW_operator"], g.ndata["_ABS_DATAFLOW_operator"])
    gv = synth.make_batch(64, 150, seed=1, variable=True)
    assert gv.batch_num_nodes().min() >= 2 and gv.batch_num_nodes().max() <= 2000 and len(set(gv.batch_num_nodes().tolist())) > 10


def test_edge_case_batch_has_the_edge_cases():
    g = synth.make_edge_cases()
    src, dst = g.edges()
    deg = torch.bincount(dst, minlength=g.num_nodes())
    assert g.batch_num_nodes().tolist() == [1, 2, 300, 40, 5]
    assert int(deg.min()) == 0 and int(deg.max()) >= 80


def test_partition_and_split():
    g = synth.make_batch(40, 50, seed=2, variable=True)
    for world in (1, 2, 3, 8):
        offs = G.partition_graphs(g.batch_num_nodes(), world)
        assert offs[0] == 0 and offs[-1] == 40 and all(b > a for a, b in zip(offs, offs[1:]))
        parts = G.split_batch(g, world)
        assert sum(p.batch_size for p in parts) == 40
        assert sum(p.num_nodes() for p in parts) == g.num_nodes()
        assert sum(p.num_edges() for p in parts) == g.num_edges()
        if world > 1:
            sizes = [p.num_nodes() for p in parts]
            assert max(sizes) <= 2.0 * (g.num_nodes() / world) + int(g.batch_num_nodes().max())
    with pytest.raises(ValueError):
        G.partition_graphs(torch.tensor([3, 4]), 3)


def test_module_mirrors_reference_constructor_and_state_dict():
    torch.manual_seed(0)
    m = D.FlowGNNGGNNModule(FEAT, 1002, 32, 5, 3, "graph", True, False)   # positional order: linevul_main.py:589-602
    torch.manual_seed(0)
    o = O.OracleFlowGNNGGNN(FEAT, 1002, 32, 5, 3, "graph", True, False)
    sm, so = m.state_dict(), o.state_dict()
    assert list(sm.keys()) == list(so.keys())
    assert all(sm[k].shape == so[k].shape and torch.equal(sm[k], so[k]) for k in sm)   # same init stream as the reference modules
    assert m.out_dim == 256 and m.hparams.label_style == "graph" and m.hparams.encoder_mode is False
    assert m.feature_keys["feature"] == "_ABS_DATAFLOW"
    assert sum(p.numel() for p in m.parameters()) == 375938
    m.load_state_dict(so)                                       # a reference checkpoint's state_dict loads unchanged
    enc = D.FlowGNNGGNNModule(FEAT, 1002, 32, 5, 3, encoder_mode=True)
    assert not hasattr(enc, "output_layer") and enc.out_dim == 64   # single embedding: D = hidden_dim
    kw = D.FlowGNNGGNNModule(FEAT, 50, 8, 2, 1, positive_weight=3.0, time=True, profile=False, test_every=False, tune_nni=False,
                             undersample_node_on_loss_factor=None)   # BaseModule kwargs (base_module.py:27-29)
    assert kw.hparams.positive_weight == 3.0 and kw.hparams.time is True


def test_module_rejects_unsupported_and_has_no_cpu_fallback():
    with pytest.raises(NotImplementedError):
        D.FlowGNNGGNNModule(FEAT, 50, 8, 2, 1, label_style="dataflow_solution_out")
    node = D.FlowGNNGGNNModule(FEAT, 50, 8, 2, 2, label_style="node")      # ggnn.py:66-68: no pooling module in this style
    assert not hasattr(node, "pooling") and not any(k.startswith(("pooling", "_node")) for k in node.state_dict())
    with pytest.raises(TypeError):
        D.FlowGNNGGNNModule(FEAT, 50, 8, 2, 1, num_node_types=3)    # stale kwargs of other revisions (SURVEY App. E)
    with pytest.raises(ValueError):
        D.FlowGNNGGNNModule(FEAT, 50, 8, 2, 1, engine="triton")
    m = D.FlowGNNGGNNModule(FEAT, 50, 8, 2, 1, concat_all_absdf=True)
    g = synth.make_batch(sizes=[4, 5], input_dim=50, seed=0)
    with pytest.raises(DdfaError, match="no CPU fallback|CUDA"):
        m(g, {})
    with pytest.raises(DdfaError):
        m.ggnn(g, None)            # parameter containers never compute


def test_param_list_order_matches_parampack():
    from deepdfa_b200 import engine as E
    m = D.FlowGNNGGNNModule(FEAT, 50, 8, 2, 3, concat_all_absdf=True)
    pk = E.ParamPack.from_flat_list(m.param_list(), 4, 3)
    assert pk.w_msg is m.ggnn.linears[0].weight and pk.w_hh is m.ggnn.gru.weight_hh and pk.b_gate is m.pooling.gate_nn.bias
    assert pk.mlp_w[2] is m.output_layer[4].weight and pk.mlp_b[0] is m.output_layer[0].bias
    assert [t.shape for t in pk.flat_list()] == [p.shape for p in m.param_list()]


def test_analytic_counts_and_count_strings():
    """SURVEY.md §8 f4: the MAC model behind profiledata.jsonl and the '<number> <unit>' strings report_profiling.py parses."""
    m = D.FlowGNNGGNNModule(FEAT, 1002, 32, 8, 2, concat_all_absdf=True)
    flops, macs, params = m.analytic_counts(38400, 256)
    Dw = 128
    assert macs == 38400 * 8 * 7 * Dw * Dw + 38400 * 2 * Dw + 256 * (2 * Dw * 2 * Dw + 2 * Dw)
    assert flops == 2 * macs and params == sum(p.numel() for p in m.parameters()) == 375938 - (2 * Dw * 2 * Dw + 2 * Dw)  # L = 2 head
    for x, want in ((70.46e9, "70.46 G"), (3.5e6, "3.50 M"), (1234.0, "1.23 K")):
        s = m._count_str(x)
        assert s == want and len(s.split(" ")) == 2 and s.split(" ")[1] in ("G", "M", "K")
    enc = D.FlowGNNGGNNModule(FEAT, 1002, 32, 5, 3, concat_all_absdf=True, encoder_mode=True)
    assert enc.analytic_counts(100, 4)[1] == 100 * 5 * 7 * Dw * Dw + 100 * 2 * Dw


def test_module_state_dict_matches_the_reference_classes():
    """Key names and shapes of FlowGNNGGNNModule.state_dict() vs the state_dict the REAL reference classes produced
    (tests/golden/reference_ctrlflow_golden.pt.xz, written by make_reference_ctrlflow_golden.py), incl. loss_fn.pos_weight."""
    from golden_params import load
    data = load("reference_ctrlflow_golden.pt.xz")
    for case in data["cases"]:
        m = D.FlowGNNGGNNModule(**case["ctor"])
        ours, ref = m.state_dict(), case["state_dict"]
        assert sorted(ours.keys()) == sorted(ref.keys()), case["name"]
        for k in ref:
            assert ours[k].shape == ref[k].shape, (case["name"], k)
        m.load_state_dict(ref)                      # a reference checkpoint loads as is
