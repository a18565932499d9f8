"""ORACLE — CPU restatement of the DDFA ``code_gnn`` GGNN hot path.  TEST INFRASTRUCTURE ONLY.

This file is the checker, never the product: only ``tests/``, ``__graft_entry__.smoke()``
and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may import it.  The product
package ``deepdfa_b200`` never imports anything under ``oracle/`` and has no CPU path.

PARITY STATUS: **partially pinned**.
  * The reference cannot run here: ``ggnn.py`` imports ``dgl`` (:5) and
    ``pytorch_lightning`` (:11), neither installed, no network (SURVEY.md §8c).
  * Everything the reference delegates to **torch** (``nn.Embedding`` ggnn.py:48-54,
    ``nn.Linear`` :67,:71-80, ``nn.GRUCell`` inside DGL's GatedGraphConv,
    ``BCEWithLogitsLoss`` base_module.py:72-74, ``optim.Adam`` config_default.yaml:43-47)
    is executed here by the *real* torch modules — that part is the reference's own
    dependency running in this container, and ``tests/test_oracle.py`` additionally pins the
    explicit-formula restatement (``gru_cell_formula``) against ``torch.nn.GRUCell``.
  * The reference's OWN code for this path — ``FlowGNNGGNNModule.__init__ / forward`` (ggnn.py:23-109) and
    ``BaseModule.__init__ / get_label / training_step`` (base_module.py:27-95, 171-199) — has been EXECUTED in the build
    container with stand-ins for its bookkeeping imports (Lightning, torchmetrics, deepspeed, nni) and with the two DGL
    operators bound to the restatements below (``tests/golden/make_reference_ctrlflow_golden.py``); its outputs, labels,
    training loss, gradients (the larger ones sampled) and state_dict are committed (``tests/golden/reference_ctrlflow_golden.pt.xz``) and
    ``tests/test_oracle.py::test_oracle_matches_reference_control_flow`` pins this oracle against them.  So parameter
    construction and naming, embedding order, concatenations, pooling / MLP placement, ``squeeze``, ``encoder_mode``, the
    graph-label rule and the loss are pinned to the reference's executing code.
  * The two **DGL** ops are restated from the pinned upstream version (``dgl<1.1.3``,
    ``environment.yml:10``; ``dgl-cu113==0.9.0`` in ``LineVul/requirements.txt``), whose
    source is NOT vendored in ``/root/reference`` and is not installed:
      - ``dgl.nn.pytorch.conv.GatedGraphConv.forward`` (n_etypes == 1 fast path):
        zero-pad ``feat`` to ``out_feats``; repeat ``n_steps`` times
        ``graph.ndata['h'] = linears[0](feat)``;
        ``update_all(fn.copy_u('h','m'), fn.sum('m','a'))``; ``feat = gru(a, feat)``.
        ``reset_parameters``: ``xavier_normal_(linear.weight, gain=calculate_gain('relu'))``,
        ``zeros_(linear.bias)``, ``gru.reset_parameters()``.
      - ``dgl.nn.pytorch.glob.GlobalAttentionPooling.forward`` (feat_nn=None):
        ``gate = gate_nn(feat)``; ``gate = softmax_nodes(graph, 'gate')``;
        ``readout = sum_nodes(graph, feat * gate)``.
    No reference test pins these numerics (SURVEY.md §4) => **parity unpinned for the DGL
    portion**; the restatement below *is* the contract.  ``tests/test_oracle.py`` upgrades
    itself to compare against real DGL modules whenever ``import dgl`` succeeds.

Control flow follows ``DDFA/code_gnn/models/flow_gnn/ggnn.py:82-109`` line by line;
state_dict keys/shapes equal the reference's (SURVEY.md §5 checkpoint row).
"""
from __future__ import annotations

import torch
from torch import nn

allfeats = ["api", "datatype", "literal", "operator"]  # ggnn.py:17-19


# --------------------------------------------------------------------------------------
# DGL restatements
# --------------------------------------------------------------------------------------
class GatedGraphConvRestated(nn.Module):
    """dgl.nn.pytorch.GatedGraphConv (n_etypes=1) — call site ggnn.py:57-60,95."""

    def __init__(self, in_feats, out_feats, n_steps, n_etypes=1, bias=True):
        super().__init__()
        if n_etypes != 1:
            raise NotImplementedError("reference uses n_etypes=1 (ggnn.py:60)")
        if in_feats > out_feats:
            raise ValueError("GatedGraphConv requires in_feats <= out_feats")
        self._in_feats, self._out_feats, self._n_steps = in_feats, out_feats, n_steps
        self.linears = nn.ModuleList([nn.Linear(out_feats, out_feats) for _ in range(n_etypes)])
        self.gru = nn.GRUCell(out_feats, out_feats, bias=bias)
        self.reset_parameters()

    def reset_parameters(self):
        gain = nn.init.calculate_gain("relu")
        self.gru.reset_parameters()
        for linear in self.linears:
            nn.init.xavier_normal_(linear.weight, gain=gain)
            nn.init.zeros_(linear.bias)

    def forward(self, graph, feat, return_all_steps=False):
        src, dst = graph.edges()
        src, dst = src.to(torch.int64), dst.to(torch.int64)
        n = feat.shape[0]
        zero_pad = feat.new_zeros((n, self._out_feats - feat.shape[1]))
        feat = torch.cat([feat, zero_pad], -1)
        steps = [feat]
        for _ in range(self._n_steps):
            h = self.linears[0](feat)                      # graph.ndata['h'] = linears[0](feat)
            a = torch.zeros_like(h).index_add_(0, dst, h.index_select(0, src))  # copy_u + sum
            feat = self.gru(a, feat)
            steps.append(feat)
        return (feat, steps) if return_all_steps else feat


def segment_ids(batch_num_nodes: torch.Tensor) -> torch.Tensor:
    bnn = batch_num_nodes.to(torch.int64)
    return torch.repeat_interleave(torch.arange(bnn.shape[0], device=bnn.device), bnn)


class GlobalAttentionPoolingRestated(nn.Module):
    """dgl.nn.pytorch.GlobalAttentionPooling(gate_nn, feat_nn=None) — call site ggnn.py:66-68,102."""

    def __init__(self, gate_nn):
        super().__init__()
        self.gate_nn = gate_nn

    def forward(self, graph, feat, get_attention=False):
        bnn = graph.batch_num_nodes().to(feat.device)
        nb = bnn.shape[0]
        gid = segment_ids(bnn)
        gate = self.gate_nn(feat)
        assert gate.shape[-1] == 1, "The output of gate_nn should have size 1 at the last axis."
        g = gate.squeeze(-1)
        # softmax_nodes: softmax over each graph's node segment
        gmax = torch.full((nb,), float("-inf"), dtype=g.dtype, device=g.device)
        gmax = gmax.scatter_reduce(0, gid, g, reduce="amax", include_self=True)
        e = torch.exp(g - gmax.index_select(0, gid))
        denom = torch.zeros(nb, dtype=g.dtype, device=g.device).index_add_(0, gid, e)
        alpha = (e / denom.index_select(0, gid)).unsqueeze(-1)
        # sum_nodes(feat * gate)
        readout = torch.zeros(nb, feat.shape[1], dtype=feat.dtype, device=feat.device)
        readout.index_add_(0, gid, feat * alpha)
        return (readout, alpha) if get_attention else readout


# --------------------------------------------------------------------------------------
# The model (ggnn.py:21-109) and the step contract (base_module.py:72-95,171-199)
# --------------------------------------------------------------------------------------
class OracleFlowGNNGGNN(nn.Module):
    """FlowGNNGGNNModule restated without Lightning.  Same ctor args (ggnn.py:23-32),
    same submodule names => same state_dict keys."""

    def __init__(self, feat, input_dim, hidden_dim, n_steps, num_output_layers,
                 label_style="graph", concat_all_absdf=False, encoder_mode=False,
                 positive_weight=None, **kwargs):
        super().__init__()
        if "_ABS_DATAFLOW" in feat:                        # ggnn.py:36-37
            feat = "_ABS_DATAFLOW"
        self.feature_keys = {"feature": feat}
        self.input_dim = input_dim
        self.concat_all_absdf = concat_all_absdf
        self.label_style = label_style
        self.encoder_mode = encoder_mode
        embedding_dim = hidden_dim
        if concat_all_absdf:                               # ggnn.py:47-52
            self.all_embeddings = nn.ModuleDict({of: nn.Embedding(input_dim, embedding_dim) for of in allfeats})
            embedding_dim *= len(allfeats)
            hidden_dim *= len(allfeats)
        else:
            self.embedding = nn.Embedding(input_dim, embedding_dim)
        self.ggnn = GatedGraphConvRestated(in_feats=embedding_dim, out_feats=hidden_dim,
                                           n_steps=n_steps, n_etypes=1)
        output_in_size = embedding_dim + hidden_dim
        self.out_dim = output_in_size                      # ggnn.py:64
        if label_style == "graph":
            self.pooling = GlobalAttentionPoolingRestated(nn.Linear(output_in_size, 1))
        if not encoder_mode:                               # ggnn.py:70-80
            layers = []
            for i in range(num_output_layers):
                last = i == num_output_layers - 1
                layers.append(nn.Linear(output_in_size, 1 if last else output_in_size))
                if not last:
                    layers.append(nn.ReLU())
            self.output_layer = nn.Sequential(*layers)
        if positive_weight is not None:                    # base_module.py:72-74
            positive_weight = torch.tensor([positive_weight])
        self.loss_fn = nn.BCEWithLogitsLoss(pos_weight=positive_weight)

    def embed(self, graph):
        if self.concat_all_absdf:                          # ggnn.py:84-89
            cfeats = [self.all_embeddings[of](graph.ndata[f"_ABS_DATAFLOW_{of}"]) for of in allfeats]
            return torch.cat(cfeats, dim=1)
        return self.embedding(graph.ndata[self.feature_keys["feature"]])   # ggnn.py:91-92

    def forward(self, graph, extrafeats=None):
        feat_embed = self.embed(graph)
        ggnn_out = self.ggnn(graph, feat_embed)            # ggnn.py:95
        out = torch.cat([ggnn_out, feat_embed], -1)        # ggnn.py:98
        if self.label_style == "graph":
            out = self.pooling(graph, out)                 # ggnn.py:102
        if self.encoder_mode:
            return out                                     # ggnn.py:104-105
        return self.output_layer(out).squeeze()            # ggnn.py:107

    def get_label(self, batch):
        """base_module.py:83-95, label_style == 'graph': per-graph max of _VULN."""
        if self.label_style == "node":
            return batch.ndata["_VULN"].float()
        if self.label_style != "graph":
            raise NotImplementedError(self.label_style)
        bnn = batch.batch_num_nodes()
        vuln = batch.ndata["_VULN"]
        gid = segment_ids(bnn.to(vuln.device))
        lab = torch.zeros(bnn.shape[0], dtype=vuln.dtype, device=vuln.device)
        lab = lab.scatter_reduce(0, gid, vuln, reduce="amax", include_self=False)
        return lab.float()

    def training_loss(self, batch, extrafeats=None):
        """base_module.py:171-183 without the logging."""
        label = self.get_label(batch)
        out = self.forward(batch, extrafeats)
        if out.dim() == 0:
            out = out.unsqueeze(0)
        return self.loss_fn(out, label.to(out.dtype)), out


def make_optimizer(model, lr=1e-3, weight_decay=1e-2):
    """config_default.yaml:43-47 — torch.optim.Adam with coupled L2 (NOT AdamW)."""
    return torch.optim.Adam(model.parameters(), lr=lr, weight_decay=weight_decay)


# --------------------------------------------------------------------------------------
# Explicit formulas (Appendix A/B of SURVEY.md) used to pin the restatement against torch
# --------------------------------------------------------------------------------------
def gru_cell_formula(a, h, w_ih, w_hh, b_ih, b_hh):
    """torch.nn.GRUCell written out: gate order (r, z, n)."""
    gi = a @ w_ih.t() + b_ih
    gh = h @ w_hh.t() + b_hh
    d = h.shape[1]
    r = torch.sigmoid(gi[:, :d] + gh[:, :d])
    z = torch.sigmoid(gi[:, d:2 * d] + gh[:, d:2 * d])
    n = torch.tanh(gi[:, 2 * d:] + r * gh[:, 2 * d:])
    return (1 - z) * n + z * h


def folded_step_formula(h, src, dst, w, b, w_ih, w_hh, b_ih, b_hh):
    """One propagation step with the re-association the CUDA path uses:
    a_v = W (sum_u h_u) + indeg(v) b  =>  gi = s (W_ih W)^T + indeg (W_ih b) + b_ih."""
    n = h.shape[0]
    s = torch.zeros_like(h).index_add_(0, dst, h.index_select(0, src))
    deg = torch.zeros(n, dtype=h.dtype).index_add_(0, dst, torch.ones(dst.shape[0], dtype=h.dtype))
    w_fold = w_ih @ w
    b_fold = w_ih @ b
    gi = s @ w_fold.t() + deg[:, None] * b_fold[None, :] + b_ih
    gh = h @ w_hh.t() + b_hh
    d = h.shape[1]
    r = torch.sigmoid(gi[:, :d] + gh[:, :d])
    z = torch.sigmoid(gi[:, d:2 * d] + gh[:, d:2 * d])
    nn_ = torch.tanh(gi[:, 2 * d:] + r * gh[:, 2 * d:])
    return (1 - z) * nn_ + z * h
