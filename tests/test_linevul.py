"""LineVul + DeepDFA combined head (SURVEY.md §8 f3, BASELINE configs[4]): ``deepdfa_b200.linevul.LineVulCombined`` against
outputs of the reference's own ``linevul_model.Model`` (tests/golden/make_reference_linevul_golden.py), and the eval harness
of ``linevul_main.evaluate`` (F1 at the 0.5 threshold) with the CUDA encoder against the oracle encoder under one frozen head."""
import time

import numpy as np
import pytest
import torch

from deepdfa_b200 import synth
from deepdfa_b200.batched_graph import BatchedCFG
from deepdfa_b200.linevul import LineVulCombined, evaluate
from golden_params import load
from oracle import ggnn_oracle as O

GOLDEN = "reference_linevul_golden.pt.xz"
DEV = "cuda:0"


def _build(data, flow, device="cpu", overlap=True):
    from transformers import RobertaConfig, RobertaForSequenceClassification
    config = RobertaConfig(**data["roberta"])
    model = LineVulCombined(RobertaForSequenceClassification(config), flow, config, overlap=overlap)
    sd = {k: v for k, v in data["state_dict"].items() if not k.startswith(("roberta.", "flowgnn_encoder."))}
    missing, unexpected = model.load_state_dict(sd, strict=False)
    # the reference class inherits an unused second RoBERTa ("roberta.*"); everything else must line up by name
    assert not unexpected and all(k.startswith("flowgnn_encoder.") for k in missing), (missing, unexpected)
    flow.load_state_dict({k[len("flowgnn_encoder."):]: v for k, v in data["state_dict"].items() if k.startswith("flowgnn_encoder.")})
    return model.to(device).eval()


def _graph(data):
    gd = data["graph"]
    return BatchedCFG(gd["src"], gd["dst"], gd["batch_num_nodes"], gd["ndata"])


def test_wrapper_reproduces_reference_model_on_cpu():
    """Control flow, head and state_dict naming of the wrapper are the reference's: with the oracle as flowgnn_encoder (what the
    fixture was generated with) the outputs are identical."""
    data = load(GOLDEN)
    model = _build(data, O.OracleFlowGNNGGNN(**data["flow"]))
    g = _graph(data)
    with torch.no_grad():
        loss, prob = model(input_ids=data["input_ids"], labels=data["labels"], graphs=g)
        prob_only = model(input_ids=data["input_ids"], graphs=g)
    assert torch.allclose(prob, data["prob"], atol=1e-6) and torch.allclose(loss, data["loss"], atol=1e-6)
    assert torch.equal(prob, prob_only)
    res = evaluate(model, [(data["input_ids"], data["labels"], g)])
    assert set(res) >= {"eval_recall", "eval_precision", "eval_f1", "eval_threshold"}      # linevul_main.py:296-301


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
def test_cuda_encoder_under_the_reference_head(engine):
    import deepdfa_b200 as D
    data = load(GOLDEN)
    flow = D.FlowGNNGGNNModule(**data["flow"], engine=engine)
    model = _build(data, flow, DEV)
    g = _graph(data)
    with torch.no_grad():
        loss, prob = model(input_ids=data["input_ids"].to(DEV), labels=data["labels"].to(DEV), graphs=g)
    err = float((prob.cpu() - data["prob"]).abs().max())
    print(f"LineVul head, engine={engine}: max|dprob| vs the reference model = {err:.2e}")
    assert err < 1e-3 and abs(float(loss) - float(data["loss"])) < 1e-3
    decisive = (data["prob"][:, 1] - 0.5).abs() > 5e-3
    assert torch.equal((prob.cpu()[:, 1] > 0.5)[decisive], (data["prob"][:, 1] > 0.5)[decisive])


@pytest.mark.gpu
def test_eval_f1_gpu_encoder_vs_oracle_encoder_and_stream_overlap():
    """BASELINE configs[4]: DDFA GPU embeddings fed to a FROZEN LineVul classifier, eval F1.  2 048 synthetic functions (graph +
    token ids); the head is fitted once on oracle embeddings (frozen encoders, 800 Adam steps on 1 024 other functions) so the F1
    is that of a working classifier; then ``linevul_main.evaluate``'s rule scores the same frozen head with (a) the oracle
    encoder on the CPU and (b) the CUDA encoder — with and without the side-stream overlap."""
    import deepdfa_b200 as D
    learnable_batch = synth.make_learnable_batch
    data = load(GOLDEN)
    torch.manual_seed(1)
    oracle_flow = O.OracleFlowGNNGGNN(**data["flow"])
    cpu_model = _build(data, oracle_flow)
    flow_sd = oracle_flow.state_dict()

    def batches(seed0, n, device):
        out = []
        for i in range(n):
            g = learnable_batch(128, 40, seed=seed0 + i)
            gen = torch.Generator().manual_seed(seed0 + i)
            ids = torch.randint(3, 120, (128, 24), generator=gen)
            ids[:, 0] = 0
            offs = np.concatenate([[0], np.cumsum(g.batch_num_nodes().numpy())])
            y = torch.from_numpy(np.maximum.reduceat(g.ndata["_VULN"].numpy(), offs[:-1]).astype(np.int64))
            out.append((ids.to(device), y.to(device), g))
        return out

    # fit a fresh head on oracle embeddings (encoders frozen; the fixture's head is scaled for spread, not for training) — CPU, ~1 s
    from transformers import RobertaConfig
    from deepdfa_b200.linevul import RobertaClassificationHead
    for p in cpu_model.parameters():
        p.requires_grad_(False)
    torch.manual_seed(2)
    cpu_model.classifier = RobertaClassificationHead(RobertaConfig(**data["roberta"]), oracle_flow.out_dim).eval()
    opt = torch.optim.Adam(cpu_model.classifier.parameters(), lr=3e-3)
    train = batches(2000, 8, "cpu")
    with torch.no_grad():
        feats = [(cpu_model.encoder.roberta(ids, attention_mask=ids.ne(1))[0], oracle_flow(g), y) for ids, y, g in train]
    for step in range(800):
        h, f, y = feats[step % len(feats)]
        opt.zero_grad()
        loss = torch.nn.functional.cross_entropy(cpu_model.classifier(h, f), y)
        loss.backward()
        opt.step()
    cpu_model.eval()
    head_sd = {k: v.clone() for k, v in cpu_model.classifier.state_dict().items()}

    held_cpu = batches(3000, 16, "cpu")                     # 2 048 functions
    t0 = time.perf_counter()
    res_cpu = evaluate(cpu_model, held_cpu)
    t_cpu = time.perf_counter() - t0

    results = {}
    for overlap in (True, False):
        flow = D.FlowGNNGGNNModule(**data["flow"], engine="tcgen05")
        gpu_model = _build(data, flow, DEV, overlap=overlap)
        flow.load_state_dict(flow_sd)
        gpu_model.classifier.load_state_dict(head_sd)
        held_gpu = [(ids.to(DEV), y.to(DEV), g.to(DEV)) for ids, y, g in held_cpu]
        evaluate(gpu_model, held_gpu)                       # warm-up pass over the SAME batches: device CSRs cached, the caching
                                                            # allocator's per-stream pools filled (the side stream has its own)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = evaluate(gpu_model, held_gpu)
        torch.cuda.synchronize()
        results[overlap] = (res, time.perf_counter() - t0)
    res_gpu = results[True][0]
    agree = float(((res_gpu["probs"][:, 1] > 0.5) == (res_cpu["probs"][:, 1] > 0.5)).mean())
    dprob = float(np.abs(res_gpu["probs"] - res_cpu["probs"]).max())
    print(f"configs[4] eval, 2048 functions, frozen head: F1 oracle-encoder {res_cpu['eval_f1']:.4f} vs CUDA-encoder {res_gpu['eval_f1']:.4f}; "
          f"decision agreement {agree:.4f}; max|dprob| {dprob:.2e}; wall: cpu {t_cpu:.2f}s, gpu overlap {results[True][1] * 1e3:.1f} ms, "
          f"gpu serial {results[False][1] * 1e3:.1f} ms")
    assert res_cpu["eval_f1"] > 0.75                         # the frozen head is a working classifier
    assert agree >= 0.998 and abs(res_gpu["eval_f1"] - res_cpu["eval_f1"]) <= 0.005 and dprob < 5e-3
    assert np.array_equal(results[True][0]["probs"], results[False][0]["probs"])     # overlap changes scheduling, not numbers


@pytest.mark.gpu
def test_side_stream_overlap_at_roberta_base_size():
    """The same A/B with a transformer of the size LineVul uses (RoBERTa-base shape: 12 layers x 768, random weights — no
    checkpoint can be downloaded here), batch 16 x 512 tokens as in linevul_main.py's defaults, graphs of Big-Vul size: wall time of
    the combined forward with the DDFA encoder on the side stream vs on the main stream; identical outputs."""
    import deepdfa_b200 as D
    from transformers import RobertaConfig, RobertaForSequenceClassification
    torch.manual_seed(0)
    config = RobertaConfig(vocab_size=50265, hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072,
                           max_position_embeddings=514, num_labels=2)
    encoder = RobertaForSequenceClassification(config).to(DEV).eval()
    FEAT = "_ABS_DATAFLOW_api_all_limitall_1000_limitsubkeys_1000"
    flow = D.FlowGNNGGNNModule(FEAT, 1002, 32, 5, 3, concat_all_absdf=True, encoder_mode=True).to(DEV)
    g = synth.make_batch(16, 150, seed=3, variable=True).to(DEV)
    ids = torch.randint(3, 50000, (16, 512), device=DEV)
    out = {}
    for overlap in (False, True):
        model = LineVulCombined(encoder, flow, config, overlap=overlap).to(DEV).eval()
        with torch.no_grad():
            for _ in range(3):
                prob = model(input_ids=ids, graphs=g)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(10):
                prob = model(input_ids=ids, graphs=g)
            torch.cuda.synchronize()
        out[overlap] = ((time.perf_counter() - t0) / 10, prob)
    print(f"LineVul forward, RoBERTa-base shape, 16 x 512 tokens + 16 CFGs: serial {out[False][0] * 1e3:.2f} ms, side-stream overlap {out[True][0] * 1e3:.2f} ms")
    assert out[False][1].shape == (16, 2)
