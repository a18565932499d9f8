"""Golden for the LineVul + DeepDFA combined head (SURVEY.md §8 f3, BASELINE configs[4]) — produced by the reference's OWN
``LineVul/linevul/linevul_model.py`` (``Model`` + ``RobertaClassificationHead``, imported unmodified: it needs only torch and
transformers, both installed) around a tiny random-weight RoBERTa and the oracle's encoder_mode GGNN as ``flowgnn_encoder``.

The parameters, except the output projection rescaled below, are set from tests/golden_params.py's hash before the model runs;
the fixture stores their names, shapes and bounds instead of their values.

Run with a checkout of ISU-PAAL/DeepDFA:   python tests/golden/make_reference_linevul_golden.py <DeepDFA>/LineVul/linevul
Writes tests/golden/reference_linevul_golden.pt.xz; read by tests/test_linevul.py (CPU: our wrapper + oracle encoder reproduce it;
GPU: our wrapper + the CUDA encoder reproduce it within the 1e-3 bound with identical decisions).
"""
import os
import sys
from types import SimpleNamespace

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from golden_params import hash_params, save, stored_state  # noqa: E402
from deepdfa_b200 import synth  # noqa: E402
from oracle import ggnn_oracle as O  # noqa: E402

FEAT = "_ABS_DATAFLOW_api_all_limitall_1000_limitsubkeys_1000"
ROBERTA = dict(vocab_size=120, hidden_size=64, num_hidden_layers=2, num_attention_heads=4, intermediate_size=128,
               max_position_embeddings=40, num_labels=2)
FLOW = dict(feat=FEAT, input_dim=1002, hidden_dim=32, n_steps=5, num_output_layers=3, concat_all_absdf=True, encoder_mode=True)


def main(reference):
    sys.path.insert(0, reference)
    from transformers import RobertaConfig, RobertaForSequenceClassification
    from linevul_model import Model as RefModel          # the reference class, unmodified
    torch.manual_seed(0)
    config = RobertaConfig(**ROBERTA)
    encoder = RobertaForSequenceClassification(config)
    flow = O.OracleFlowGNNGGNN(**FLOW)
    ref = RefModel(encoder, flow, config, tokenizer=None, args=SimpleNamespace(no_flowgnn=False))
    params = hash_params(ref, 0, skip=("classifier.out_proj.",))
    with torch.no_grad():                                  # spread the probabilities away from 0.5 (random init gives ~0.5 +- 0.01)
        ref.classifier.out_proj.weight.mul_(40.0)
    ref.eval()
    g = synth.make_batch(8, 30, seed=31, variable=True, vuln_rate=0.4)
    input_ids = torch.randint(3, 120, (8, 24))
    input_ids[:, 0] = 0
    input_ids[5, 20:] = 1                                  # padding tokens (id 1): exercises the attention mask
    labels = torch.tensor([0, 1, 0, 0, 1, 1, 0, 1])
    with torch.no_grad():                                  # centre the decision boundary inside the batch: mixed decisions
        p0 = ref(input_ids=input_ids, graphs=g)
        ref.classifier.out_proj.bias[1] -= torch.log(p0[:, 1] / p0[:, 0]).median()
    with torch.no_grad():
        loss, prob = ref(input_ids=input_ids, labels=labels, graphs=g)
        prob_only = ref(input_ids=input_ids, graphs=g)
        loss_a, prob_a, att = ref(input_ids=input_ids, labels=labels, graphs=g, output_attentions=True)
    assert torch.equal(prob, prob_only) and torch.allclose(prob, prob_a)
    out = {"roberta": ROBERTA, "flow": FLOW, "state_dict": stored_state(ref, params), "params": params,
           "input_ids": input_ids, "labels": labels,
           "graph": {"src": g.edges()[0], "dst": g.edges()[1], "batch_num_nodes": g.batch_num_nodes(), "ndata": dict(g.ndata)},
           "loss": loss.clone(), "prob": prob.clone(), "num_attentions": len(att),
           "note": "outputs of the reference's own linevul_model.Model; flowgnn_encoder = oracle/ggnn_oracle.py (encoder_mode)"}
    path = save(out, "reference_linevul_golden.pt.xz")
    print("wrote", path, float(loss), prob[:, 1])


if __name__ == "__main__":
    main(sys.argv[1])
