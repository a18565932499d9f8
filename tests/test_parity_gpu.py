"""GPU: end-to-end parity of the reference-facing module (deepdfa_b200.FlowGNNGGNNModule, which
calls the C ABI) against the oracle — golden fixtures, live oracle on the same seeded inputs,
gradients, optimisation steps, and the size-independent properties at BASELINE's full sizes.

Bar (BASELINE.json north_star): logits within 1e-3 of the fp32 reference, identical labels
(sign of the logit == decision at the 0.5 sigmoid threshold, base_module.py:186,364)."""
import copy

import pytest
import torch

import deepdfa_b200 as D
from deepdfa_b200 import batched_graph as G
from deepdfa_b200 import synth
from oracle import ggnn_oracle as O
from parity_helpers import GRAD_TOL

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FEAT = "_ABS_DATAFLOW_api_all_limitall_1000_limitsubkeys_1000"
TOL = 1e-3


def graph_of(case):
    b = case["graph"]
    return G.BatchedCFG(b["src"], b["dst"], b["batch_num_nodes"], b["ndata"])


def module_of(case, engine):
    torch.manual_seed(case["seed"])
    m = D.FlowGNNGGNNModule(**case["ctor"], engine=engine)
    for k, (s, a) in case["checksums"].items():
        assert abs(float(m.state_dict()[k].double().sum()) - s) <= 1e-9 * max(1.0, abs(a)), "RNG drift: regenerate goldens"
    return m.to(DEV)


def tc_available():
    from deepdfa_b200._lib import ENGINE_TCGEN05, lib
    return lib().call("ddfa_engine_available", ENGINE_TCGEN05) == 1


def engines_of(case):
    d = case["ctor"]["hidden_dim"] * (4 if case["ctor"]["concat_all_absdf"] else 1)
    return ["simt", "tcgen05"] if (d == 128 and tc_available()) else ["simt"]


@pytest.fixture(autouse=True)
def _skip_unbuilt_engine(request):
    engine = request.node.callspec.params.get("engine") if hasattr(request.node, "callspec") else None
    if engine == "tcgen05" and not tc_available():
        pytest.skip("tcgen05 engine not compiled into libddfa_b200.so")


def assert_logits_close(got, ref64, tol=TOL):
    got = got.detach().cpu().double().reshape(ref64.shape)
    err = float((got - ref64).abs().max())
    assert err <= tol, f"max |dlogit| = {err:.3e} > {tol}"
    if ref64.dim() == 1:
        decisive = ref64.abs() > 10 * max(err, 1e-7)
        assert torch.equal((got > 0)[decisive], (ref64 > 0)[decisive])
    return err


def test_golden_forward_both_engines(golden):
    worst = {}
    for case in golden["cases"]:
        g = graph_of(case)
        for engine in engines_of(case):
            m = module_of(case, engine)
            with torch.no_grad():
                out = m(g.to(DEV), {})
            assert out.shape == case["out_fp64"].shape
            err = assert_logits_close(out, case["out_fp64"])
            worst[engine] = max(worst.get(engine, 0.0), err)
            labels = m.get_label(g.to(DEV))
            assert torch.equal(labels.cpu(), case["labels"])
    print("worst |dlogit| vs fp64 oracle per engine:", worst)
    assert worst["simt"] < 5e-5          # fp32 FFMA engine sits at the fp32 noise floor


def test_golden_gradients(golden):
    for case in golden["cases"]:
        if "grad_norm_fp64" not in case:
            continue
        g = graph_of(case).to(DEV)
        for engine in engines_of(case):
            m = module_of(case, engine)
            loss = m.training_step((g, {}), 0)
            assert abs(float(loss) - case["loss_fp64"]) < 1e-5
            loss.backward()
            for name, p in m.named_parameters():
                ref_norm = case["grad_norm_fp64"][name]
                got_norm = float(p.grad.double().norm())
                assert abs(got_norm - ref_norm) <= 2e-3 * max(ref_norm, 1e-4) + 1e-7, (case["name"], engine, name, got_norm, ref_norm)
                if case.get("grads_fp64"):
                    ref = case["grads_fp64"][name]
                    assert (p.grad.cpu().double() - ref).abs().max() <= 1e-4 * max(1.0, float(ref.abs().max())) + 1e-7, (case["name"], name)


def test_encoder_mode_backward_through_pooled(golden):
    case = next(c for c in golden["cases"] if c["name"] == "tiny_encoder_T2")
    g = graph_of(case)
    torch.manual_seed(case["seed"])
    o = O.OracleFlowGNNGGNN(**case["ctor"]).double()
    m = module_of(case, "simt")
    w = torch.randn(g.batch_size, m.out_dim, dtype=torch.float64)
    (o(g) * w).sum().backward()
    out = m(g.to(DEV), {})
    assert out.shape == (g.batch_size, m.out_dim)
    (out * w.float().to(DEV)).sum().backward()
    for (name, p), (_, q) in zip(m.named_parameters(), o.named_parameters()):
        assert (p.grad.cpu().double() - q.grad).abs().max() <= 1e-4 * max(1.0, float(q.grad.abs().max())) + 1e-7, name


@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
def test_adam_steps_width128_both_paths_against_oracle(engine):
    """Three Adam steps at hidden width 128 on both engines, through (a) the reference-style loop (module.training_step +
    loss.backward() + stock torch.optim.Adam) and (b) FusedTrainer (flat buffers + ddfa_adam_flat): losses and the parameters
    after the third step follow the fp32 oracle trained the same way."""
    g = synth.make_batch(12, 50, seed=21, variable=True, vuln_rate=0.4)
    torch.manual_seed(5)
    o = O.OracleFlowGNNGGNN(FEAT, 1002, 32, 6, 2, concat_all_absdf=True, positive_weight=2.5)
    state0 = copy.deepcopy(o.state_dict())
    opt = O.make_optimizer(o)
    ref_losses = []
    for _ in range(3):
        opt.zero_grad()
        loss_ref, _ = o.training_loss(g)
        loss_ref.backward()
        opt.step()
        ref_losses.append(float(loss_ref))
    for path in ("module_api", "fused_trainer"):
        m = D.FlowGNNGGNNModule(FEAT, 1002, 32, 6, 2, concat_all_absdf=True, positive_weight=2.5, engine=engine)
        m.load_state_dict(state0)
        m.to(DEV)
        gd = g.to(DEV)
        losses = []
        if path == "module_api":
            mopt = m.configure_optimizers()
            for _ in range(3):
                mopt.zero_grad()
                loss = m.training_step((gd, {}), 0)
                loss.backward()
                mopt.step()
                losses.append(float(loss))
        else:
            tr = D.FusedTrainer(m)
            losses = [float(tr.step(gd)) for _ in range(3)]
        assert losses == pytest.approx(ref_losses, abs=5e-5), (path, engine)
        worst = max(float((m.state_dict()[k].cpu() - v).abs().max()) for k, v in o.state_dict().items())
        print(f"adam x3 {path} {engine}: max |dparam| vs oracle {worst:.2e}")
        # Adam's first steps move every touched parameter by ~lr = 1e-3 whatever the gradient's size, so a sign flip of a
        # near-zero gradient component shows as 2e-3; bound well below that
        assert worst < (5e-5 if engine == "simt" else 5e-4), (path, engine, worst)      # measured r03c: 2.1e-5 / 1.7e-4


def test_tiny_adam_steps_autograd_path_and_fused_trainer(golden):
    case = next(c for c in golden["cases"] if c["name"] == "tiny_T3_L2")
    g = graph_of(case).to(DEV)
    # (a) reference-style loop: module.training_step + stock torch Adam (config_default.yaml:43-47)
    m = module_of(case, "simt")
    opt = m.configure_optimizers()
    losses = []
    for _ in range(3):
        opt.zero_grad()
        loss = m.training_step((g, {}), 0)
        loss.backward()
        opt.step()
        losses.append(float(loss))
    assert losses == pytest.approx(case["adam_losses"], abs=2e-5)
    for k, v in case["state_after_adam"].items():
        assert (m.state_dict()[k].cpu() - v).abs().max() < 2e-5, k
    # (b) fused trainer: flat buffers + ddfa_adam_flat
    m2 = module_of(case, "simt")
    tr = D.FusedTrainer(m2)
    losses2 = [float(tr.step(g)) for _ in range(3)]
    assert losses2 == pytest.approx(case["adam_losses"], abs=2e-5)
    for k, v in case["state_after_adam"].items():
        assert (m2.state_dict()[k].cpu() - v).abs().max() < 2e-5, k


@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
@pytest.mark.parametrize("T,L", [(8, 2), (5, 3)])
def test_full_size_c0_against_live_oracle(engine, T, L):
    """BASELINE config 1/2: 256 CFGs x 150 nodes / 300 edges, 128-d, T steps — logits vs the CPU oracle."""
    g = synth.make_batch(256, 150, seed=0)
    torch.manual_seed(0)
    o = O.OracleFlowGNNGGNN(FEAT, 1002, 32, T, L, concat_all_absdf=True)
    for p in o.parameters():           # trained-scale weights (SURVEY.md §7 hard part 1): x2
        p.data.mul_(2.0)
    with torch.no_grad():
        ref = o(g).double()
    m = D.FlowGNNGGNNModule(FEAT, 1002, 32, T, L, concat_all_absdf=True, engine=engine)
    m.load_state_dict(o.state_dict())
    m.to(DEV)
    with torch.no_grad():
        out = m(g, {})                  # CPU graph: moved to the module's device by the module
    err = assert_logits_close(out, ref)
    print(f"C0 T={T} L={L} engine={engine}: max|dlogit|={err:.2e}, |logit| range {float(ref.abs().max()):.2f}")
    assert torch.equal(m.get_label(g).cpu(), o.get_label(g))


@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
@pytest.mark.parametrize("variable", [False, True])
def test_c1_logits_against_live_fp64_oracle(engine, variable):
    """BASELINE configs[2] shape: 1024 CFGs (fixed 150 nodes, and lognormal sizes 2..2000) — logits of both engines against the
    fp64 CPU oracle at trained-scale weights, identical decisions."""
    g = synth.make_batch(1024, 150, seed=11, variable=variable)
    torch.manual_seed(0)
    o = O.OracleFlowGNNGGNN(FEAT, 1002, 32, 8, 2, concat_all_absdf=True)
    for p in o.parameters():
        p.data.mul_(2.0)
    m = D.FlowGNNGGNNModule(FEAT, 1002, 32, 8, 2, concat_all_absdf=True, engine=engine)
    m.load_state_dict(o.state_dict())
    m.to(DEV)
    o = o.double()
    with torch.no_grad():
        ref = o(g)
        out = m(g, {})
    err = assert_logits_close(out, ref)
    print(f"C1 variable={variable} engine={engine}: N={g.num_nodes()} max|dlogit| vs fp64 = {err:.2e}, |logit| max {float(ref.abs().max()):.2f}")
    assert torch.equal(m.get_label(g).cpu(), o.get_label(g).float())


@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
def test_full_size_gradients_against_live_oracle(engine):
    g = synth.make_batch(64, 150, seed=5, variable=True, vuln_rate=0.3)
    torch.manual_seed(1)
    o = O.OracleFlowGNNGGNN(FEAT, 1002, 32, 8, 3, concat_all_absdf=True, positive_weight=4.0).double()
    loss_ref, _ = o.training_loss(g)
    loss_ref.backward()
    m = D.FlowGNNGGNNModule(FEAT, 1002, 32, 8, 3, concat_all_absdf=True, positive_weight=4.0, engine=engine)
    m.load_state_dict({k: v.float() for k, v in o.state_dict().items()})
    m.to(DEV)
    loss = m.training_step((g.to(DEV), {}), 0)
    loss.backward()
    assert abs(float(loss) - float(loss_ref)) < 1e-4
    worst = {}
    for (name, p), (_, q) in zip(m.named_parameters(), o.named_parameters()):
        ref = q.grad
        # pooling.gate_nn.bias: the softmax is shift-invariant, its true gradient is 0 (|ref| ~ 1e-10) — absolute floor
        scale = max(float(ref.abs().max()), 1e-3)
        worst[name] = float((p.grad.cpu().double() - ref).abs().max()) / scale
    print(f"gradient worst case per parameter vs fp64 oracle, engine={engine}: " + ", ".join(f"{k}={v:.1e}" for k, v in worst.items()))
    bad = {k: v for k, v in worst.items() if v >= GRAD_TOL[engine]}
    assert not bad, bad


@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
def test_properties_at_c1_size(engine):
    """Batch 1024 (BASELINE config 3 shape): determinism, batch-composition invariance (graphs never
    exchange messages), and sharding over 2 'ranks' reproducing the unsharded logits."""
    g = synth.make_batch(1024, 150, seed=7, variable=True)
    torch.manual_seed(3)
    m = D.FlowGNNGGNNModule(FEAT, 1002, 32, 8, 3, concat_all_absdf=True, engine=engine).to(DEV)
    with torch.no_grad():
        a = m(g.to(DEV), {})
        b = m(g.to(DEV), {})
        assert torch.equal(a, b)
        parts = G.split_batch(g, 2)
        pa = torch.cat([m(p.to(DEV), {}) for p in parts])
    assert (a - pa).abs().max() < 1e-5
    assert a.shape == (1024,) and torch.isfinite(a).all()


def test_single_graph_squeeze_and_duck_typed_dgl_graph():
    m = D.FlowGNNGGNNModule(FEAT, 60, 8, 3, 2, concat_all_absdf=True).to(DEV)
    g = synth.make_batch(sizes=[9], input_dim=60, seed=1)
    out = m(g.to(DEV), {})
    assert out.dim() == 0                          # logits.squeeze() (ggnn.py:107)

    class FakeDGL:                                  # anything exposing the DGL subset is accepted
        def __init__(self, g):
            self._g, self.ndata = g, g.ndata
        def edges(self):
            return self._g.edges()
        def batch_num_nodes(self):
            return self._g.batch_num_nodes()
    g3 = synth.make_batch(sizes=[4, 9, 2], input_dim=60, seed=2)
    with torch.no_grad():
        assert torch.equal(m(FakeDGL(g3), {}), m(g3, {}))


def test_index_validation_raises():
    m = D.FlowGNNGGNNModule(FEAT, 60, 8, 2, 1, concat_all_absdf=True).to(DEV)
    g = synth.make_batch(sizes=[6, 3], input_dim=60, seed=1)
    good = synth.make_batch(sizes=[6, 3], input_dim=60, seed=2)
    g.ndata["_ABS_DATAFLOW_api"][2] = 60
    assert m.validate_inputs == "deferred"          # default: no host sync on the hot path, the error surfaces one call later
    m(g, {})
    with pytest.raises(IndexError):
        m.check_inputs()
    m(g, {})
    torch.cuda.synchronize()
    with pytest.raises(IndexError):
        m(good, {})
    m(good, {})
    m.check_inputs()                                # a clean batch raises nothing
    m.validate_inputs = "sync"                      # $DDFA_B200_VALIDATE=1: checked before forward returns
    with pytest.raises(IndexError):
        m(g, {})
    bad_edge = synth.make_batch(sizes=[6, 3], input_dim=60, seed=3)
    src, dst = bad_edge.edges()
    src[1] = 9                                      # endpoint outside [0, 9)
    with pytest.raises(IndexError):
        m(bad_edge, {})


@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
def test_fused_trainer_tracks_oracle_training(engine):
    """Config-3 style check at reduced size: 10 optimisation steps on a stream of batches; the loss
    curve and the final decisions follow the oracle trained on the identical stream (both engines, width 128)."""
    torch.manual_seed(0)
    o = O.OracleFlowGNNGGNN(FEAT, 1002, 32, 5, 3, concat_all_absdf=True, positive_weight=8.0)
    m = D.FlowGNNGGNNModule(FEAT, 1002, 32, 5, 3, concat_all_absdf=True, positive_weight=8.0, engine=engine)
    m.load_state_dict(copy.deepcopy(o.state_dict()))
    m.to(DEV)
    tr = D.FusedTrainer(m)
    opt = O.make_optimizer(o)
    batches = [synth.make_batch(32, 60, seed=50 + i, variable=True, vuln_rate=0.3) for i in range(5)]
    for step in range(10):
        b = batches[step % 5]
        opt.zero_grad()
        loss_ref, _ = o.training_loss(b)
        loss_ref.backward()
        opt.step()
        loss = float(tr.step(b))
        assert abs(loss - float(loss_ref)) < 2e-3 * max(1.0, abs(float(loss_ref))), (step, loss, float(loss_ref))
    with torch.no_grad():
        ref = o(batches[0]).double()
        out = m(batches[0], {})
    assert (out.cpu().double() - ref).abs().max() < 5e-3


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
def test_fused_trainer_cuda_graph_paths_match_eager(engine):
    """use_cuda_graph=True: (a) resident device batches -> one captured graph per batch object, (b) host batches -> static
    per-shape input buffers + one graph that includes the device CSR build.  Both must reproduce the eager loss curve."""
    batches = [synth.make_batch(16, 40, seed=70 + i, vuln_rate=0.3) for i in range(3)]        # same shape, different content
    losses = {}
    for mode in ("eager", "graph_host", "graph_host_prefetch", "graph_device"):
        torch.manual_seed(1)
        m = D.FlowGNNGGNNModule(FEAT, 1002, 32, 4, 2, concat_all_absdf=True, engine=engine).to(DEV)
        tr = D.FusedTrainer(m, use_cuda_graph=(mode != "eager"))
        bs = [b.to(DEV) for b in batches] if mode == "graph_device" else batches
        cur = []
        for step in range(9):                       # every batch is visited eagerly (warm-up), at capture, and on replay
            loss_t = tr.step(bs[step % 3])
            if mode == "graph_host_prefetch":       # H2D of the next batch overlaps this step
                tr.prefetch(bs[(step + 1) % 3])
            cur.append(float(loss_t))
        losses[mode] = cur
        if mode in ("graph_host", "graph_host_prefetch"):
            slot = next(iter(tr._stream_slots.values()))
            assert len(tr._stream_slots) == 1 and all(st["graph"] is not None for st in slot["sets"])
        if mode == "graph_device":
            assert len(tr._graphs) == 3
    for mode in ("graph_host", "graph_host_prefetch", "graph_device"):
        for a, b in zip(losses["eager"], losses[mode]):
            assert abs(a - b) < 1e-5 * max(1.0, abs(a)), (mode, losses["eager"], losses[mode])
    assert losses["eager"][0] != losses["eager"][3]      # the parameters did move


@pytest.mark.gpu
def test_batched_weight_gradient_matches_per_step(monkeypatch):
    """tcgen05 engine: the one-launch weight-gradient GEMM over all T steps (default) and the per-step deferred accumulation give
    the same parameter gradients; so do the backward with the transposed gather folded into gate_bwd and the unfused one."""
    torch.manual_seed(3)
    b = synth.make_batch(24, 60, seed=5, variable=True, vuln_rate=0.3)
    grads = {}
    from deepdfa_b200 import engine as E
    for key, opts in (("default", {}), ("per_step_wgrad", {"batched_wgrad": False}), ("unfused_gather", {"fuse_gather_bwd": False})):
        monkeypatch.setattr(E, "OPTIONS", dict(E.OPTIONS, **dict({"fuse_gather_bwd": True, "batched_wgrad": True}, **opts)))
        torch.manual_seed(11)
        m = D.FlowGNNGGNNModule(FEAT, 1002, 32, 6, 2, concat_all_absdf=True, engine="tcgen05").to(DEV)
        loss = m.training_step((b, {}), 0)
        loss.backward()
        grads[key] = {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}
    for key in ("per_step_wgrad", "unfused_gather"):
        for n, gref in grads["default"].items():
            scale = max(1e-6, float(gref.abs().max()))
            assert float((grads[key][n] - gref).abs().max()) < 2e-4 * scale, (key, n)


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
def test_linevul_style_combined_head(engine):
    """SURVEY.md §8 f3: the encoder_mode output feeding a LineVul-style head (LineVul/linevul/linevul_model.py:6-24:
    cat(<s> feature, flowgnn embedding) -> dense -> tanh -> out_proj(2), CrossEntropyLoss at :57-60) — loss and the
    gradients reaching the GGNN parameters match the oracle driving the same head; a tiny HF RoBERTa encoder (random
    weights, transformers is installed) provides the token features to show the two autograd graphs join."""
    from transformers import RobertaConfig, RobertaModel
    torch.manual_seed(0)
    hidden = 64
    cfg = RobertaConfig(vocab_size=120, hidden_size=hidden, num_hidden_layers=2, num_attention_heads=4, intermediate_size=128,
                        max_position_embeddings=40, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    roberta = RobertaModel(cfg, add_pooling_layer=False).to(DEV).eval()
    b = synth.make_batch(6, 30, seed=9, variable=True, vuln_rate=0.3)
    B = b.batch_size
    o = O.OracleFlowGNNGGNN(FEAT, 1002, 32, 5, 3, concat_all_absdf=True, encoder_mode=True).double()
    m = D.FlowGNNGGNNModule(FEAT, 1002, 32, 5, 3, concat_all_absdf=True, encoder_mode=True, engine=engine)
    m.load_state_dict({k: v.float() for k, v in o.state_dict().items()})
    m.to(DEV)
    assert m.out_dim == o.out_dim == 256
    dense = torch.nn.Linear(hidden + m.out_dim, hidden).double()
    out_proj = torch.nn.Linear(hidden, 2).double()
    input_ids = torch.randint(3, 120, (B, 24), device=DEV)
    labels = torch.tensor([0, 1, 0, 0, 1, 1])
    feats = roberta(input_ids, attention_mask=input_ids.ne(1))[0]            # [B, 24, hidden] (linevul_model.py:63)

    def head(cls_feature, flow, dense_, proj_):
        x = torch.cat((cls_feature, flow), dim=1)
        return proj_(torch.tanh(dense_(x)))

    # oracle side (fp64, CPU)
    cls_ref = feats[:, 0, :].detach().cpu().double()
    loss_ref = torch.nn.functional.cross_entropy(head(cls_ref, o(b), dense, out_proj), labels)
    loss_ref.backward()
    # ours: GPU, fp32, the same head weights
    dense32, proj32 = torch.nn.Linear(hidden + 256, hidden).to(DEV), torch.nn.Linear(hidden, 2).to(DEV)
    dense32.load_state_dict({k: v.float() for k, v in dense.state_dict().items()})
    proj32.load_state_dict({k: v.float() for k, v in out_proj.state_dict().items()})
    flow = m(b, {})
    assert flow.shape == (B, 256)
    loss = torch.nn.functional.cross_entropy(head(feats[:, 0, :], flow, dense32, proj32), labels.to(DEV))
    loss.backward()
    assert abs(float(loss) - float(loss_ref)) < 2e-4
    tol = 1e-4 if engine == "simt" else 1e-3
    for (name, p), (_, q) in zip(m.named_parameters(), o.named_parameters()):
        assert (p.grad.cpu().double() - q.grad).abs().max() <= tol * max(1.0, float(q.grad.abs().max())) + 1e-7, name
    assert roberta.embeddings.word_embeddings.weight.grad is not None       # the transformer side of the joint graph got its gradient


@pytest.mark.gpu
def test_test_step_writes_reference_profiling_records(tmp_path):
    """SURVEY.md §8 f4: test_step with time / profile emits timedata.jsonl / profiledata.jsonl rows in the schema
    scripts/report_profiling.py reads (base_module.py:238-291), only for steps after the third."""
    import json
    b = synth.make_batch(12, 40, seed=4, vuln_rate=0.3).to(DEV)
    for flag, fname, keys in (("time", "timedata.jsonl", {"step", "batch_size", "runtime"}),
                              ("profile", "profiledata.jsonl", {"step", "flops", "params", "macs", "batch_size"})):
        m = D.FlowGNNGGNNModule(FEAT, 1002, 32, 4, 2, concat_all_absdf=True, **{flag: True}).to(DEV)
        m.profile_output_dir = str(tmp_path)
        outs = [m.test_step((b, {}), i) for i in range(6)]
        rows = [json.loads(l) for l in open(tmp_path / fname)]
        assert [r["step"] for r in rows] == [3, 4, 5] and all(set(r) == keys and r["batch_size"] == 12 for r in rows)
        if flag == "time":
            assert all(0.0 < r["runtime"] < 1e3 for r in rows)
        else:
            flops, macs, params = m.analytic_counts(b.num_nodes(), 12)
            for r in rows:      # the parsing rule of report_profiling.py
                count, unit = r["flops"].split(" ")
                assert abs(float(count) * {"G": 1e9, "M": 1e6, "K": 1e3}[unit] - flops) <= 0.005 * {"G": 1e9, "M": 1e6, "K": 1e3}[unit]
        loss, prob, labels = outs[-1]
        ref_loss, ref_prob, ref_labels = m.validation_step((b, {}), 0)
        assert torch.equal(prob, ref_prob) and torch.equal(labels, ref_labels) and float(loss) == float(ref_loss)


@pytest.mark.gpu
def test_graph_caps_degrade_to_eager():
    """A stream of ever-new batch shapes must not accumulate captured graphs: beyond max_graph_shapes the same kernels run
    eagerly and the results stay those of the eager trainer."""
    batches = [synth.make_batch(8, 20 + 3 * i, seed=90 + i, vuln_rate=0.3) for i in range(5)]     # 5 different shapes
    order = [0, 1, 2, 3, 4, 0, 1, 2, 3, 4, 0, 1]
    losses = {}
    for mode in ("eager", "graph"):
        torch.manual_seed(2)
        m = D.FlowGNNGGNNModule(FEAT, 1002, 32, 3, 2, concat_all_absdf=True, engine="tcgen05").to(DEV)
        tr = D.FusedTrainer(m, use_cuda_graph=(mode == "graph"), max_graph_shapes=2)
        losses[mode] = [float(tr.step(batches[i])) for i in order]
        if mode == "graph":
            assert len(tr._stream_slots) == 2
    for a, b in zip(losses["eager"], losses["graph"]):
        assert abs(a - b) < 1e-5 * max(1.0, abs(a))


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
def test_module_matches_reference_control_flow_goldens(engine):
    """The CUDA module against outputs of the reference's own ggnn.py / base_module.py code (fixture written by
    tests/golden/make_reference_ctrlflow_golden.py; small widths, so the SIMT engine): logits / pooled embedding, graph labels,
    training loss and parameter gradients."""
    from deepdfa_b200.batched_graph import BatchedCFG
    from golden_params import load, sample_error
    data = load("reference_ctrlflow_golden.pt.xz")
    checked_grads = 0
    for case in data["cases"]:
        gd = case["graph"]
        g = BatchedCFG(gd["src"], gd["dst"], gd["batch_num_nodes"], gd["ndata"])
        if engine == "tcgen05" and case["ctor"]["hidden_dim"] * (4 if case["ctor"].get("concat_all_absdf") else 1) != 128:
            continue                                                      # the tensor-core engine is the width-128 one
        m = D.FlowGNNGGNNModule(**case["ctor"], engine=engine)
        m.load_state_dict(case["state_dict"])
        m.to(DEV)
        with torch.no_grad():
            out = m(g, {})
        assert out.shape == case["out"].shape, case["name"]
        assert (out.cpu() - case["out"]).abs().max() < (1e-4 if engine == "simt" else 1e-3), case["name"]   # north-star bound 1e-3
        assert torch.equal((out.cpu() > 0), (case["out"] > 0)), case["name"]                                # identical decisions
        assert torch.equal(m.get_label(g).cpu(), case["label"]), case["name"]
        if "train_loss" in case:
            m.zero_grad(set_to_none=True)
            loss = m.training_step((g, {}), 0)
            loss.backward()
            assert abs(float(loss) - float(case["train_loss"])) < 1e-4, case["name"]
            for k, p in m.named_parameters():
                if k in case["grads"]:
                    ref = case["grads"][k]
                    tol = 2e-4 if engine == "simt" else 2e-3
                    assert sample_error(p.grad, ref) < tol * max(1.0, ref["absmax"]), (case["name"], k)
            checked_grads += 1
    assert checked_grads >= 1, "no reference-code gradient case ran for this engine"


@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
def test_node_label_style_with_undersampling_matches_oracle(engine):
    """label_style="node" (ggnn.py:101-107 without the pooling; base_module.py:84-85 labels; base_module.py:96-135,178-183 the
    undersampled training loss): per-node logits, per-node labels, validation loss, and the training step with
    undersample_node_on_loss_factor — same `random` seed on both sides, so the same nodes are drawn."""
    import random
    hd = 32 if engine == "tcgen05" else 8
    ctor = dict(feat=FEAT, input_dim=50, hidden_dim=hd, n_steps=3, num_output_layers=2, concat_all_absdf=True, label_style="node",
                positive_weight=1.5)
    g = synth.make_batch(sizes=[12, 40, 1, 7, 25], seed=5, vuln_rate=0.8, input_dim=50)
    assert 0 < int(g.ndata["_VULN"].sum()) < g.num_nodes() // 2
    torch.manual_seed(7)
    o = O.OracleFlowGNNGGNN(**ctor)
    m = D.FlowGNNGGNNModule(**ctor, undersample_node_on_loss_factor=1.0, engine=engine)
    m.load_state_dict(o.state_dict())
    m.to(DEV)
    with torch.no_grad():
        ref = o(g).double()
    vloss, prob, labels = m.validation_step((g, {}), 0)
    assert prob.shape == (g.num_nodes(),) and torch.equal(labels.cpu(), o.get_label(g).int())
    assert (torch.logit(prob.double().cpu()) - ref).abs().max() < (1e-4 if engine == "simt" else 1e-3)
    assert abs(float(vloss) - float(o.loss_fn(ref.float(), o.get_label(g)))) < 1e-4
    random.seed(3)
    loss = m.training_step((g, {}), 0)
    loss.backward()
    random.seed(3)
    out, label = o(g), o.get_label(g)
    vi = label.nonzero().flatten().tolist()
    idx = vi + random.sample((label == 0).nonzero().flatten().tolist(), round(len(vi) * 1.0))
    lo = o.loss_fn(out[idx], label[idx])
    lo.backward()
    assert abs(float(loss) - float(lo)) < 1e-4
    ref_g = dict(o.named_parameters())
    tol = 2e-4 if engine == "simt" else 2e-3
    for k, p in m.named_parameters():
        r = ref_g[k].grad
        assert (p.grad.cpu() - r).abs().max() < tol * max(1.0, float(r.abs().max())), k


def test_module_path_is_immune_to_garbage_in_recycled_memory():
    """The autograd path allocates its activation images fresh every step and clears only the tile that can hold padding rows
    (engine._FreshAlloc.get_image).  Poison the caching allocator's free blocks with NaNs and check that a training step over a
    batch whose node count is not a multiple of the 128-row tile still gives the same finite loss and gradients."""
    if not tc_available():
        pytest.skip("tcgen05 engine not compiled into libddfa_b200.so")
    g = synth.make_batch(sizes=[150, 3, 77, 140, 1, 129], seed=21, vuln_rate=0.5, input_dim=64)
    assert g.num_nodes() % 128 != 0
    torch.manual_seed(3)
    m = D.FlowGNNGGNNModule(FEAT, 64, 32, 8, 2, concat_all_absdf=True, engine="tcgen05").to(DEV)

    def run():
        m.zero_grad(set_to_none=True)
        loss = m.training_step((g, {}), 0)
        loss.backward()
        return float(loss), {k: p.grad.clone() for k, p in m.named_parameters()}

    loss0, grads0 = run()
    for _ in range(2):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        junk = [torch.full((n,), float("nan"), device=DEV) for n in (1 << 14, 1 << 18, 1 << 22, 1 << 24)]
        del junk                              # freed blocks go back to the caching allocator and are handed out again, unzeroed
        loss1, grads1 = run()
        assert loss1 == loss1 and abs(loss1 - loss0) < 1e-6
        for k, g0 in grads0.items():
            assert torch.isfinite(grads1[k]).all(), k
            assert (grads1[k] - g0).abs().max() <= 1e-5 * max(1.0, float(g0.abs().max())), k
