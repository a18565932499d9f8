"""Pins the oracle's restatement of the reference's OWN code — by running that code.

The reference module cannot be imported as shipped: `ggnn.py` / `base_module.py` import dgl, pytorch_lightning, torchmetrics,
deepspeed and nni, none of which is installed (no network).  But everything those imports are used for on this path is either
bookkeeping (Lightning hooks, metrics, profiler) or the two DGL operators.  This script installs minimal stand-ins for the
bookkeeping packages and lets the REAL reference classes run:

    DDFA/code_gnn/models/flow_gnn/ggnn.py      FlowGNNGGNNModule.__init__ / forward          (ggnn.py:23-109)
    DDFA/code_gnn/models/base_module.py        BaseModule.__init__ / get_label / training_step (:27-95, :171-199)

with `dgl.nn.pytorch.GatedGraphConv` / `GlobalAttentionPooling` / `dgl.unbatch` bound to the restatements in
oracle/ggnn_oracle.py and deepdfa_b200.batched_graph (those remain the UNPINNED part: DGL itself is not here).  What the
fixture therefore pins, against the reference's own executing code: parameter construction and state_dict naming, the
feature-key and embedding order, the concatenations, where pooling and the MLP sit, `.squeeze()`, `encoder_mode`, the
graph-label rule (`dgl.unbatch` + max of `_VULN`), `BCEWithLogitsLoss(pos_weight)` and the training-step loss.

The parameters are set from tests/golden_params.py's hash before the reference code runs, so the fixture stores their names,
shapes and bounds instead of their values, and a sample of each large gradient (see that module).

Run with a checkout of ISU-PAAL/DeepDFA:   python tests/golden/make_reference_ctrlflow_golden.py <DeepDFA>/DDFA
Writes tests/golden/reference_ctrlflow_golden.pt.xz; tests/test_oracle.py::test_oracle_matches_reference_control_flow reads it.
"""
import inspect
import os
import sys
import types

import torch
from torch import nn

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from golden_params import hash_params, sample, save, stored_state  # noqa: E402
from deepdfa_b200 import batched_graph as BG  # noqa: E402
from deepdfa_b200 import synth  # noqa: E402
from oracle import ggnn_oracle as O  # noqa: E402


def install_stand_ins():
    """Bookkeeping packages the reference imports but this path does not compute with."""
    class _HParams(dict):
        __getattr__ = dict.__getitem__

    class LightningModule(nn.Module):
        def save_hyperparameters(self):      # Lightning: the calling __init__'s arguments, merged over the class hierarchy
            frame = inspect.currentframe().f_back
            args = inspect.getargvalues(frame)
            hp = self.__dict__.setdefault("_hp", _HParams())
            for name in args.args:
                if name != "self":
                    hp[name] = args.locals[name]
            if args.keywords:
                hp.update(args.locals[args.keywords])

        @property
        def hparams(self):
            return self.__dict__["_hp"]

        def log(self, *a, **k):
            pass

        def log_dict(self, *a, **k):
            pass

    pl = types.ModuleType("pytorch_lightning")
    pl.LightningModule = LightningModule
    util = types.ModuleType("pytorch_lightning.utilities")
    cli = types.ModuleType("pytorch_lightning.utilities.cli")
    cli.MODEL_REGISTRY = lambda cls: cls
    pl.utilities, util.cli = util, cli

    class _Metric(nn.Module):
        def __init__(self, *a, **k):
            super().__init__()

        def clone(self, prefix=None):
            return _Metric()

        def update(self, *a, **k):
            pass

        def forward(self, x=None, *a, **k):
            return x

        def compute(self):
            return {}

        def reset(self):
            pass

    tm = types.ModuleType("torchmetrics")
    for n in ("MetricCollection", "Accuracy", "Precision", "Recall", "F1Score", "PrecisionRecallCurve", "BinnedPrecisionRecallCurve",
              "CatMetric", "ConfusionMatrix", "MeanMetric"):
        setattr(tm, n, _Metric)

    ds = [types.ModuleType(n) for n in ("deepspeed", "deepspeed.profiling", "deepspeed.profiling.flops_profiler",
                                        "deepspeed.profiling.flops_profiler.profiler")]
    ds[3].FlopsProfiler = lambda module: None
    nni = types.ModuleType("nni")

    # the two DGL operators and dgl.unbatch: the oracle's restatements (the part that stays unpinned)
    dgl = types.ModuleType("dgl")
    dgl_nn = types.ModuleType("dgl.nn")
    dgl_nn_pt = types.ModuleType("dgl.nn.pytorch")
    dgl_nn_pt.GatedGraphConv = O.GatedGraphConvRestated
    dgl_nn_pt.GlobalAttentionPooling = O.GlobalAttentionPoolingRestated
    dgl.nn, dgl_nn.pytorch = dgl_nn, dgl_nn_pt
    dgl.unbatch = lambda g, node_split=None, edge_split=None: BG.unbatch(g)

    mods = {"pytorch_lightning": pl, "pytorch_lightning.utilities": util, "pytorch_lightning.utilities.cli": cli, "torchmetrics": tm,
            "nni": nni, "dgl": dgl, "dgl.nn": dgl_nn, "dgl.nn.pytorch": dgl_nn_pt}
    mods.update({m.__name__: m for m in ds})
    sys.modules.update(mods)


def main(reference):
    install_stand_ins()
    sys.path.insert(0, reference)
    from code_gnn.models.flow_gnn.ggnn import FlowGNNGGNNModule as RefModule      # the real reference class

    feat = "_ABS_DATAFLOW_datatype_all_limitall_1000_limitsubkeys_1000"
    cases = []
    specs = [
        dict(name="concat_T5_L3_pw", ctor=dict(feat=feat, input_dim=64, hidden_dim=8, n_steps=5, num_output_layers=3, concat_all_absdf=True,
                                               positive_weight=7.5), graphs=dict(sizes=[1, 2, 40, 9, 150, 3], seed=11, vuln_rate=0.3, input_dim=64)),
        dict(name="single_T3_L2", ctor=dict(feat=feat, input_dim=60, hidden_dim=24, n_steps=3, num_output_layers=2, concat_all_absdf=False),
             graphs=dict(sizes=[5, 17, 1, 30], seed=12, vuln_rate=0.5, input_dim=60)),
        dict(name="encoder_T4", ctor=dict(feat=feat, input_dim=64, hidden_dim=8, n_steps=4, num_output_layers=3, concat_all_absdf=True,
                                          encoder_mode=True), graphs=dict(sizes=[12, 7, 33], seed=13, vuln_rate=0.2, input_dim=64)),
        dict(name="one_graph_squeeze", ctor=dict(feat=feat, input_dim=64, hidden_dim=8, n_steps=2, num_output_layers=1, concat_all_absdf=True),
             graphs=dict(sizes=[21], seed=14, vuln_rate=0.4, input_dim=64)),
        # hidden width 128 (what the tcgen05 engine runs): forward only
        dict(name="concat_D128_T8_L1_fwd", ctor=dict(feat=feat, input_dim=64, hidden_dim=32, n_steps=8, num_output_layers=1, concat_all_absdf=True),
             graphs=dict(sizes=[150, 3, 77, 140, 1, 129], seed=15, vuln_rate=0.3, input_dim=64), forward_only=True),
        # hidden width 128 WITH the reference's training step: loss + parameter gradients for the tcgen05 backward kernels
        dict(name="concat_D128_T8_L2_pw_train", ctor=dict(feat=feat, input_dim=64, hidden_dim=32, n_steps=8, num_output_layers=2,
                                                         concat_all_absdf=True, positive_weight=3.0),
             graphs=dict(sizes=[150, 3, 77, 140, 1, 129, 260, 31], seed=16, vuln_rate=0.4, input_dim=64)),
        # label_style="node" (ggnn.py:101-107 without the pooling; base_module.py:84-85 per-node labels), training step without
        # the undersampling (undersample_node_on_loss_factor=None, the ctor default)
        dict(name="node_single_T3_L2_train", ctor=dict(feat=feat, input_dim=60, hidden_dim=24, n_steps=3, num_output_layers=2,
                                                      concat_all_absdf=False, label_style="node", positive_weight=2.0),
             graphs=dict(sizes=[5, 17, 1, 30], seed=17, vuln_rate=0.5, input_dim=60)),
        dict(name="node_concat_D128_T4_L2_train", ctor=dict(feat=feat, input_dim=64, hidden_dim=32, n_steps=4, num_output_layers=2,
                                                           concat_all_absdf=True, label_style="node"),
             graphs=dict(sizes=[150, 3, 77, 1, 129], seed=18, vuln_rate=0.4, input_dim=64)),
    ]
    for i, spec in enumerate(specs):
        torch.manual_seed(100 + i)
        ref = RefModule(**spec["ctor"])
        with torch.no_grad():
            ref.ggnn.linears[0].bias.uniform_(-0.1, 0.1)             # DGL zero-initialises it; make the bias path visible
        params = hash_params(ref, 100 + i)
        g = synth.make_batch(**spec["graphs"])
        if not spec["ctor"].get("concat_all_absdf"):
            g.ndata["_ABS_DATAFLOW"] = g.ndata["_ABS_DATAFLOW_datatype"] % spec["ctor"]["input_dim"]
        case = {"name": spec["name"], "ctor": spec["ctor"], "state_dict": stored_state(ref, params), "params": params,
                "graph": {"src": g.edges()[0], "dst": g.edges()[1], "batch_num_nodes": g.batch_num_nodes(), "ndata": dict(g.ndata)}}
        ref.eval()
        with torch.no_grad():
            case["out"] = ref(g, {}).clone()
            case["label"] = ref.get_label(g).clone()
        # (a one-graph batch cannot take the reference's training step: `.squeeze()` makes the logit 0-d and BCEWithLogitsLoss
        #  rejects it against the [1] label — reference behaviour, base_module.py:183)
        if not spec["ctor"].get("encoder_mode") and g.batch_size > 1 and not spec.get("forward_only"):
            ref.train()
            ref.zero_grad()
            loss = ref.training_step((g, {}), 0)
            loss.backward()
            case["train_loss"] = loss.detach().clone()
            case["grads"] = {k: sample(p.grad, 100 * i + j) for j, (k, p) in enumerate(ref.named_parameters()) if p.grad is not None}
        cases.append(case)
    out = save({"cases": cases, "note": "outputs of the reference's own ggnn.py / base_module.py code; DGL ops bound to the oracle restatements"},
               "reference_ctrlflow_golden.pt.xz")
    print("wrote", out, {c["name"]: tuple(c["out"].shape) for c in cases})


if __name__ == "__main__":
    main(sys.argv[1])
