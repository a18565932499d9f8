"""CPU: pins the oracle (oracle/ggnn_oracle.py) — against the reference's own torch dependencies,
against independent dense restatements, against the committed golden vectors, and through the
size-independent properties of the path (SURVEY.md §4)."""
import torch
import pytest

from deepdfa_b200 import synth, batched_graph as G
from oracle import ggnn_oracle as O

FEAT = "_ABS_DATAFLOW_api_all_limitall_1000_limitsubkeys_1000"


def build(case, dtype=torch.float32):
    torch.manual_seed(case["seed"])
    m = O.OracleFlowGNNGGNN(**case["ctor"])
    return m.to(dtype)


def graph_of(case):
    b = case["graph"]
    return G.BatchedCFG(b["src"], b["dst"], b["batch_num_nodes"], b["ndata"])


def test_gru_formula_matches_torch_grucell():
    torch.manual_seed(0)
    cell = torch.nn.GRUCell(24, 24).double()
    a, h = torch.randn(50, 24, dtype=torch.float64), torch.randn(50, 24, dtype=torch.float64)
    ref = cell(a, h)
    got = O.gru_cell_formula(a, h, cell.weight_ih, cell.weight_hh, cell.bias_ih, cell.bias_hh)
    assert torch.allclose(ref, got, atol=1e-13)


def test_gated_graph_conv_matches_dense_adjacency():
    torch.manual_seed(1)
    g = synth.make_batch(sizes=[7, 11, 3], input_dim=30, seed=5)
    src, dst = g.edges()
    n = g.num_nodes()
    conv = O.GatedGraphConvRestated(16, 16, n_steps=3).double()
    feat = torch.randn(n, 16, dtype=torch.float64)
    A = torch.zeros(n, n, dtype=torch.float64)
    A.index_put_((dst, src), torch.ones(src.shape[0], dtype=torch.float64), accumulate=True)  # multi-edges count
    h = feat
    for _ in range(3):
        a = A @ conv.linears[0](h)
        h = conv.gru(a, h)
    assert torch.allclose(conv(g, feat), h, atol=1e-12)


def test_gated_graph_conv_zero_pads_input():
    torch.manual_seed(2)
    g = synth.make_batch(sizes=[5], input_dim=30, seed=6)
    conv = O.GatedGraphConvRestated(8, 12, n_steps=2)
    feat = torch.randn(5, 8)
    padded = torch.cat([feat, torch.zeros(5, 4)], 1)
    conv2 = O.GatedGraphConvRestated(12, 12, n_steps=2)
    conv2.load_state_dict(conv.state_dict())
    assert torch.allclose(conv(g, feat), conv2(g, padded))


def test_pooling_matches_per_graph_softmax():
    torch.manual_seed(3)
    g = synth.make_batch(sizes=[4, 1, 9], input_dim=30, seed=7)
    pool = O.GlobalAttentionPoolingRestated(torch.nn.Linear(10, 1)).double()
    feat = torch.randn(14, 10, dtype=torch.float64)
    got = pool(g, feat)
    outs, o = [], 0
    for nn_ in g.batch_num_nodes().tolist():
        f = feat[o:o + nn_]
        alpha = torch.softmax(pool.gate_nn(f), dim=0)
        outs.append((f * alpha).sum(0))
        o += nn_
    assert torch.allclose(got, torch.stack(outs), atol=1e-13)


def test_folded_step_equals_reference_step():
    torch.manual_seed(4)
    g = synth.make_edge_cases(input_dim=30)
    src, dst = g.edges()
    n, d = g.num_nodes(), 16
    conv = O.GatedGraphConvRestated(d, d, n_steps=1).double()
    conv.linears[0].bias.data.normal_()
    h = torch.randn(n, d, dtype=torch.float64)
    ref = conv(g, h)
    got = O.folded_step_formula(h, src, dst, conv.linears[0].weight, conv.linears[0].bias, conv.gru.weight_ih,
                                conv.gru.weight_hh, conv.gru.bias_ih, conv.gru.bias_hh)
    assert torch.allclose(ref, got, atol=1e-12)


def test_get_label_matches_reference_loop():
    g = synth.make_batch(num_graphs=40, nodes_per_graph=20, variable=True, seed=3, vuln_rate=0.5)
    m = O.OracleFlowGNNGGNN(FEAT, 30, 8, 1, 1, concat_all_absdf=True)
    graphs = G.unbatch(g)
    ref = torch.stack([x.ndata["_VULN"].max() for x in graphs]).float()   # base_module.py:87-88
    assert torch.equal(m.get_label(g), ref)
    assert ref.sum() > 0


def test_golden_vectors(golden):
    assert len(golden["cases"]) >= 10
    for case in golden["cases"]:
        m32 = build(case)
        sd = m32.state_dict()
        for k, (s, a) in case["checksums"].items():
            assert abs(float(sd[k].double().sum()) - s) <= 1e-9 * max(1.0, abs(a)), f"RNG drift in {case['name']}:{k}; regenerate goldens"
        g = graph_of(case)
        with torch.no_grad():
            out32 = m32(g)
        # fp32 on another CPU runs other kernels (vector width, summation order), so only the last bits are free: 64 ulps of
        # the output's scale (other instruction sets measured up to 14); the fp64 pin below stays at 1e-12
        ulp = torch.finfo(torch.float32).eps * float(case["out_fp32"].abs().max())
        assert (out32 - case["out_fp32"]).abs().max() <= 64 * ulp, case["name"]
        m64 = build(case, torch.float64)
        m64.load_state_dict({k: v.double() for k, v in sd.items()})
        with torch.no_grad():
            out64 = m64(g)
        assert torch.allclose(out64, case["out_fp64"], atol=1e-12)
        # fp32 oracle's own distance to fp64 = the noise floor of the 1e-3 parity bound
        assert (out32.double() - out64).abs().max() < 1e-4
        assert torch.equal(m32.get_label(g), case["labels"])
        if "state_dict" in case:
            for k, v in case["state_dict"].items():
                assert torch.equal(sd[k], v)


def test_golden_training_tiny(golden):
    case = next(c for c in golden["cases"] if c["name"] == "tiny_T3_L2")
    m = build(case)
    g = graph_of(case)
    opt = O.make_optimizer(m)
    losses = []
    for _ in range(3):
        opt.zero_grad()
        loss, _ = m.training_loss(g)
        loss.backward()
        opt.step()
        losses.append(float(loss))
    assert losses == pytest.approx(case["adam_losses"], rel=1e-6)
    for k, v in case["state_after_adam"].items():
        assert torch.allclose(m.state_dict()[k], v, atol=1e-6)


def test_state_dict_keys_are_the_reference_names():
    m = O.OracleFlowGNNGGNN(FEAT, 1002, 32, 5, 3, concat_all_absdf=True)
    keys = set(m.state_dict().keys())
    expect = {f"all_embeddings.{k}.weight" for k in O.allfeats} | {
        "ggnn.linears.0.weight", "ggnn.linears.0.bias", "ggnn.gru.weight_ih", "ggnn.gru.weight_hh",
        "ggnn.gru.bias_ih", "ggnn.gru.bias_hh", "pooling.gate_nn.weight", "pooling.gate_nn.bias",
        "output_layer.0.weight", "output_layer.0.bias", "output_layer.2.weight", "output_layer.2.bias",
        "output_layer.4.weight", "output_layer.4.bias"}
    assert expect <= keys
    assert sum(p.numel() for p in m.parameters()) == 375938  # SURVEY.md §6
    assert m.state_dict()["ggnn.gru.weight_ih"].shape == (384, 128)
    assert m.out_dim == 256


def test_batch_composition_invariance_and_squeeze():
    torch.manual_seed(0)
    m = O.OracleFlowGNNGGNN(FEAT, 50, 8, 3, 2, concat_all_absdf=True).double()
    gs = [synth.make_batch(sizes=[n], input_dim=50, seed=s) for s, n in enumerate([6, 1, 13])]
    with torch.no_grad():
        whole = m(G.batch(gs))
        singles = [m(x) for x in gs]
    assert singles[0].dim() == 0          # logits.squeeze() of a 1-graph batch (ggnn.py:107)
    assert torch.allclose(whole, torch.stack(singles), atol=1e-12)


def test_permutation_equivariance():
    torch.manual_seed(0)
    m = O.OracleFlowGNNGGNN(FEAT, 50, 8, 4, 2, concat_all_absdf=True).double()
    g = synth.make_batch(sizes=[9, 14], input_dim=50, seed=2)
    src, dst = g.edges()
    # relabel nodes inside each graph (keeps per-graph contiguity, as dgl.batch requires)
    perm = torch.cat([torch.randperm(9), 9 + torch.randperm(14)])
    inv = torch.empty_like(perm); inv[perm] = torch.arange(23)
    g2 = G.BatchedCFG(inv[src], inv[dst], g.batch_num_nodes(), {k: v[perm] for k, v in g.ndata.items()})
    with torch.no_grad():
        assert torch.allclose(m(g), m(g2), atol=1e-12)


def test_against_real_dgl_if_available():
    dgl = pytest.importorskip("dgl")
    from dgl.nn.pytorch import GatedGraphConv, GlobalAttentionPooling
    torch.manual_seed(0)
    g = synth.make_batch(sizes=[7, 11, 3], input_dim=30, seed=5)
    src, dst = g.edges()
    dg = dgl.batch([dgl.graph((x.edges()[0], x.edges()[1]), num_nodes=x.num_nodes()) for x in G.unbatch(g)])
    conv_ref = GatedGraphConv(16, 16, 3, 1)
    conv = O.GatedGraphConvRestated(16, 16, 3)
    conv.load_state_dict(conv_ref.state_dict())
    feat = torch.randn(g.num_nodes(), 16)
    assert torch.allclose(conv_ref(dg, feat), conv(g, feat), atol=1e-6)
    pool_ref = GlobalAttentionPooling(torch.nn.Linear(16, 1))
    pool = O.GlobalAttentionPoolingRestated(torch.nn.Linear(16, 1))
    pool.load_state_dict(pool_ref.state_dict())
    assert torch.allclose(pool_ref(dg, feat), pool(g, feat), atol=1e-6)


def test_oracle_matches_reference_control_flow():
    """The fixture was produced by the reference's OWN ggnn.py / base_module.py code (tests/golden/make_reference_ctrlflow_golden.py:
    real FlowGNNGGNNModule + BaseModule with stand-ins for the bookkeeping imports; the two DGL operators bound to the oracle's
    restatements).  It pins the oracle's — and therefore the module's — restatement of that code: parameter names and shapes,
    embedding order, concatenations, pooling / MLP placement, squeeze, encoder_mode, graph labels, BCE(pos_weight), gradients."""
    from deepdfa_b200.batched_graph import BatchedCFG
    from golden_params import load, sample_error
    data = load("reference_ctrlflow_golden.pt.xz")
    assert len(data["cases"]) == 8 and sum(c["ctor"].get("label_style") == "node" for c in data["cases"]) == 2 and any("grads" in c and c["ctor"]["hidden_dim"] == 32 for c in data["cases"])
    for case in data["cases"]:
        gd = case["graph"]
        g = BatchedCFG(gd["src"], gd["dst"], gd["batch_num_nodes"], gd["ndata"])
        o = O.OracleFlowGNNGGNN(**case["ctor"])
        # same parameter / buffer names (the reference lists loss_fn.pos_weight first: BaseModule.__init__ runs first; order is
        # irrelevant to load_state_dict)
        assert sorted(o.state_dict().keys()) == sorted(case["state_dict"].keys()), case["name"]
        for k, v in o.state_dict().items():
            assert v.shape == case["state_dict"][k].shape, (case["name"], k)
        o.load_state_dict(case["state_dict"])
        o.eval()
        with torch.no_grad():
            out = o(g)
        assert out.shape == case["out"].shape and torch.allclose(out, case["out"], atol=1e-6, rtol=1e-5), case["name"]
        assert torch.equal(o.get_label(g), case["label"]), case["name"]
        if "train_loss" in case:
            o.train()
            o.zero_grad()
            loss, _ = o.training_loss(g)
            loss.backward()
            assert torch.allclose(loss, case["train_loss"], atol=1e-6, rtol=1e-5), case["name"]
            grads = {k: p.grad for k, p in o.named_parameters() if p.grad is not None}
            assert set(grads) == set(case["grads"]), case["name"]
            for k, s in case["grads"].items():
                assert torch.allclose(grads[k].flatten()[s["idx"].long()], s["val"], atol=1e-6, rtol=1e-4), (case["name"], k)
                assert sample_error(grads[k], s) <= 1e-6 + 1e-4 * s["absmax"], (case["name"], k)
