"""GPU: the tcgen05 backward kernels at the sizes the training step runs them at, and the D = 128 edge gathers on graphs with
controlled degree extremes — each against an fp64 reference computed on the GPU.

The backward kernels are persistent: a CTA walks many 32-row blocks (gate_bwd_tma_kernel, 3-slot TMA ring), many tiles
(dgrad3_kernel) or many (tile, step) work items (wgrad_kernel).  Slot reuse and barrier-phase flips only start beyond a few
thousand rows, so the sizes below straddle those thresholds, including a ragged last tile and a ragged last 32-row block.
The degree tests build graphs whose hubs, empty rows and 4-row-group boundaries sit exactly where the gathers switch code
paths (prefetched neighbour ids vs reloads past 32 edges, the out-edge tail of the folded transposed gather).

Every case prints its worst error, relative to max(1, |ref|max) unless noted."""
import ctypes

import numpy as np
import pytest
import torch

import deepdfa_b200 as D
from deepdfa_b200 import synth
from deepdfa_b200._lib import (ENGINE_SIMT, ENGINE_TCGEN05, TUNE_GATE_BWD_TMA, TUNE_GATHER_SRC_GROUPS, DdfaError, lib,
                               ptr_array)
from deepdfa_b200.batched_graph import BatchedCFG
from deepdfa_b200.engine import _p, _stream_ptr, prepare_graph
from oracle import ggnn_oracle as O
from parity_helpers import GRAD_TOL, decode_gates, decode_image, gru_reference

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FEAT = "_ABS_DATAFLOW_api_all_limitall_1000_limitsubkeys_1000"
DIM = 128
TILE_BYTES = 65536                 # one 128-row tile of an activation image
C0_N, C1_N, C1_VAR_N = 38400, 153600, 157377
STEP_TOL = 3e-4                    # the image-entry backward bound of test_kernels_gpu.py, relative to max(1, |ref|max)


@pytest.fixture(autouse=True)
def _needs_tcgen05():
    if lib().call("ddfa_engine_available", ENGINE_TCGEN05) != 1:
        pytest.skip("tcgen05 engine not compiled into libddfa_b200.so")
    yield
    torch.cuda.synchronize()
    torch.cuda.empty_cache()        # a C1 case holds several GB: give it back before the next one


def st():
    return _stream_ptr()


def rel_err(got, ref):
    return float((got.double() - ref).abs().max()) / max(1.0, float(ref.abs().max()))


def batch_of_size(N):
    """The bench batches at C0 / C1 (fixed and variable sizes); other N: 150-node graphs plus one ragged graph."""
    if N == C0_N:
        return synth.make_batch(256, 150, seed=0)
    if N == C1_N:
        return synth.make_batch(1024, 150, seed=0)
    if N == C1_VAR_N:
        return synth.make_batch(1024, 150, seed=11, variable=True)
    sizes = [150] * (N // 150) + ([N % 150] if N % 150 else [])
    return synth.make_batch(sizes=sizes, seed=N)


def step_weights(seed, wf_scale=1.5, bf_scale=1.0):
    g = torch.Generator().manual_seed(seed)
    k = 1.0 / DIM ** 0.5
    mk = lambda *sh: ((torch.rand(*sh, dtype=torch.float64, generator=g) * 2 - 1) * k).to(DEV)
    wf, bf, bih, whh, bhh = mk(3 * DIM, DIM) * wf_scale, mk(3 * DIM) * bf_scale, mk(3 * DIM), mk(3 * DIM, DIM), mk(3 * DIM)
    return [wf, bf, bih, whh, bhh]


def image_of(x32):
    N = x32.shape[0]
    img = torch.zeros(lib().call("ddfa_act_image_bytes", N), dtype=torch.uint8, device=DEV)
    lib().call("ddfa_act_to_image", _p(x32), N, DIM, _p(img), st())
    return img


def gather_image_src(dg, h_img, N):
    s_img = torch.zeros_like(h_img)
    lib().call("ddfa_gather_sum_image_src", _p(dg.indptr), _p(dg.indices), _p(h_img), N, DIM, _p(s_img), st())
    return s_img


class Fwd:
    """The forward step's prepared weight workspace (independent of N)."""

    def __init__(self, w):
        L = lib()
        self.w32 = [t.float().contiguous() for t in w]
        self.wsb = L.call("ddfa_gru_step_workspace_bytes", 0, DIM, ENGINE_TCGEN05)
        self.ws = torch.empty(self.wsb, dtype=torch.uint8, device=DEV)
        L.call("ddfa_gru_step_prepare", *[_p(t) for t in self.w32], DIM, ENGINE_TCGEN05, _p(self.ws), self.wsb, st())

    def __call__(self, s_img, h_img, indptr, N):
        """Middle-step form (h only as its image): -> (image of h', packed gates, fp32 h')."""
        L = lib()
        o_img = torch.zeros_like(h_img)
        gates = torch.empty(L.call("ddfa_gru_gates_packed_bytes", N, DIM), dtype=torch.uint8, device=DEV)
        h_out = torch.empty(N, DIM, device=DEV)
        L.call("ddfa_gru_step_fwd_image_v2", _p(s_img), _p(h_img), None, _p(indptr), N, DIM, None, _p(o_img), _p(gates),
               _p(self.ws), self.wsb, st())
        L.call("ddfa_gru_step_fwd_image_v2", _p(s_img), _p(h_img), None, _p(indptr), N, DIM, _p(h_out), None, None,
               _p(self.ws), self.wsb, st())
        return o_img, gates, h_out


class Bwd:
    """A prepared backward workspace for N nodes and `steps` kept q-image slots."""

    def __init__(self, w32, N, steps=1):
        L = lib()
        self.N = N
        self.wsb = L.call("ddfa_gru_step_bwd_workspace_bytes_steps", N, DIM, ENGINE_TCGEN05, steps)
        self.ws = torch.empty(self.wsb, dtype=torch.uint8, device=DEV)
        L.call("ddfa_gru_step_prepare_bwd", _p(w32[0]), _p(w32[3]), DIM, ENGINE_TCGEN05, _p(self.ws), self.wsb, st())

    @staticmethod
    def new_acc():
        return {k: torch.zeros(sh, device=DEV) for k, sh in (("dwf", (3 * DIM, DIM)), ("dbf", (3 * DIM,)), ("dbih", (3 * DIM,)),
                                                           ("dwhh", (3 * DIM, DIM)), ("dbhh", (3 * DIM,)))}

    def __call__(self, dh_part, h_img, s_img, gates, indptr, acc, ds_prev=None, indptr_t=None, indices_t=None, wgrad_mode=0,
                 wsb=None):
        N = self.N
        ds, dh = torch.empty(N, DIM, device=DEV), torch.empty(N, DIM, device=DEV)
        lib().call("ddfa_gru_step_bwd_image_v2", _p(dh_part), _p(ds_prev), _p(indptr_t), _p(indices_t), None, _p(h_img), _p(s_img),
                   _p(gates), _p(indptr), N, DIM, _p(ds), _p(dh), _p(acc["dwf"]), _p(acc["dbf"]), _p(acc["dbih"]), _p(acc["dwhh"]),
                   _p(acc["dbhh"]), _p(self.ws), self.wsb if wsb is None else wsb, wgrad_mode, st())
        return ds, dh


def step_reference(s, h, deg, w, dh_in):
    """fp64 autograd of one step: gradients of <h', dh_in> w.r.t. s, h and the five step parameters."""
    leaves = [t.detach().clone().requires_grad_(True) for t in (s, h, *w)]
    h_ref = gru_reference(leaves[0], leaves[1], deg, *leaves[2:])[0]
    (h_ref * dh_in).sum().backward()
    return dict(zip(("ds", "dh", "dwf", "dbf", "dbih", "dwhh", "dbhh"), (t.grad for t in leaves)))


def transposed_gather(src, dst, x):
    """(A^T x)[u] = sum over edges u -> v of x[v]: the gradient the folded gather adds."""
    return torch.zeros_like(x).index_add_(0, src, x[dst])


def check_outputs(label, got, ref, tol=STEP_TOL):
    errs = {k: rel_err(got[k], ref[k]) for k in ref}
    print(f"{label}: " + ", ".join(f"{k}={v:.1e}" for k, v in errs.items()))
    bad = {k: v for k, v in errs.items() if not v < tol}
    assert not bad, (label, bad)


class StepCase:
    """One step's inputs at the kernels' own precision: h as its activation image, s = A h gathered from that image, the packed
    gates of the forward step; fp64 copies of exactly what the images carry."""

    def __init__(self, g, dg, fwd, seed):
        self.N = N = g.num_nodes()
        gen = torch.Generator(device=DEV).manual_seed(seed)
        self.h_img = image_of(torch.tanh(torch.randn(N, DIM, device=DEV, generator=gen)))
        self.s_img = gather_image_src(dg, self.h_img, N)
        self.h = decode_image(self.h_img, N, DEV)
        self.s = decode_image(self.s_img, N, DEV)
        self.o_img, self.gates, self.h_out = fwd(self.s_img, self.h_img, dg.indptr, N)
        self.dh_part32 = torch.randn(N, DIM, device=DEV, generator=gen)
        self.dh_part = self.dh_part32.double()


def deg_of(dst, N):
    return torch.bincount(dst, minlength=N).double()


# ------------------------------------------------------------------------------------------------------------------------------
# A. one step backward at bench sizes, all three gate-backward forms
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [4736, 9473, 14240, 28449, C0_N, C1_N, C1_VAR_N])
def test_step_backward_at_bench_sizes(N):
    """gate_bwd_tma_kernel reuses ring slots from Npad > 3 x 148 x 32 = 14 208 rows (and flips the barrier parity again above
    28 416), dgrad3_kernel takes more than one tile per CTA pair from N > 9 472: ds, dh and the five parameter gradients of
    ddfa_gru_step_bwd_image_v2 with the transposed gather folded in, against fp64 autograd, in all three
    DDFA_TUNE_GATE_BWD_TMA modes; ds and dh bit-identical across the modes."""
    g = batch_of_size(N)
    assert g.num_nodes() == N
    dg = prepare_graph(g, DEV)
    src, dst = [t.to(DEV) for t in g.edges()]
    w = step_weights(N)
    fwd = Fwd(w)
    c = StepCase(g, dg, fwd, seed=N)
    s_ref = torch.zeros_like(c.h).index_add_(0, dst, c.h[src])
    assert rel_err(c.s, s_ref) < 2e-5
    ds_prev = torch.randn(N, DIM, device=DEV, dtype=torch.float64, generator=torch.Generator(device=DEV).manual_seed(N + 1))
    ds_prev32 = ds_prev.float()
    ref = step_reference(c.s, c.h, deg_of(dst, N), w, c.dh_part + transposed_gather(src, dst, ds_prev32.double()))
    bwd = Bwd(fwd.w32, N)
    outs = {}
    try:
        for mode in (2, 1, 0):        # 2 (default): TMA ring + pipelined CSR scalars; 1: TMA ring; 0: register path
            lib().call("ddfa_tuning_set", TUNE_GATE_BWD_TMA, mode)
            acc = Bwd.new_acc()
            ds, dh = bwd(c.dh_part32, c.h_img, c.s_img, c.gates, dg.indptr, acc, ds_prev32, dg.indptr_t, dg.indices_t)
            torch.cuda.synchronize()
            check_outputs(f"step bwd N={N} tma_mode={mode}", dict(ds=ds, dh=dh, **acc), ref)
            outs[mode] = (ds, dh)
    finally:
        lib().call("ddfa_tuning_set", TUNE_GATE_BWD_TMA, 2)
    for mode in (1, 0):
        assert torch.equal(outs[mode][0], outs[2][0]) and torch.equal(outs[mode][1], outs[2][1]), (N, mode)


# ------------------------------------------------------------------------------------------------------------------------------
# B. tile-slice invariance
# ------------------------------------------------------------------------------------------------------------------------------
def test_tile_slices_are_bit_identical_at_c1():
    """Row v of the forward step (h', its image row, its packed gates) depends only on row v's s, h and in-degree, and row v of
    the backward's ds and dh (no folded gather) only on row v's inputs.  So any 128-row-aligned slice of the variable C1 batch,
    run on its own, must reproduce the big run's rows bit for bit — whichever CTA, ring slot or barrier phase handled them."""
    N = C1_VAR_N
    g = batch_of_size(N)
    dg = prepare_graph(g, DEV)
    tiles = (N + 127) // 128
    w = step_weights(3)
    fwd = Fwd(w)
    c = StepCase(g, dg, fwd, seed=3)
    bwd = Bwd(fwd.w32, N)
    ds, dh = bwd(c.dh_part32, c.h_img, c.s_img, c.gates, dg.indptr, Bwd.new_acc())
    gates_rows = c.gates.view(N, DIM * 8)
    assert tiles == 1230 and N % 128 and N % 32
    for a, b in ((0, 1), (36, 38), (73, 75), (147, 149), (tiles - 1, tiles), (500, 510)):
        n0, n1 = a * 128, min(b * 128, N)
        n = n1 - n0
        img = slice(a * TILE_BYTES, b * TILE_BYTES)
        indptr = (dg.indptr[n0:n1 + 1] - dg.indptr[n0]).contiguous()
        s_img, h_img = c.s_img[img].contiguous(), c.h_img[img].contiguous()
        o_img, gates, h_out = fwd(s_img, h_img, indptr, n)
        assert torch.equal(o_img, c.o_img[img]), (a, b)
        assert torch.equal(gates.view(n, DIM * 8), gates_rows[n0:n1]), (a, b)
        assert torch.equal(h_out, c.h_out[n0:n1]), (a, b)
        ds_s, dh_s = Bwd(fwd.w32, n)(c.dh_part32[n0:n1].contiguous(), h_img, s_img, gates, indptr, Bwd.new_acc())
        assert torch.equal(ds_s, ds[n0:n1]) and torch.equal(dh_s, dh[n0:n1]), (a, b)
    print(f"tile slices of N={N}: forward image / gates / h' and backward ds / dh bit-identical")


# ------------------------------------------------------------------------------------------------------------------------------
# C. weight gradients accumulated over steps
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [C0_N, C1_N])
def test_weight_gradients_over_steps(N):
    """16 independent steps (own h, s, gates, incoming gradient each): dw_fold / dw_hh (and the bias sums) against the fp64 sum
    of the per-step references, through the three ways of accumulating them — kept q images + ONE batched launch (T = 1, 8, 16),
    the deferred per-CTA partials (wgrad_mode 1, 2, ..., 2 + ddfa_gru_step_bwd_finish), and the immediate form (wgrad_mode 0)."""
    T = 16
    g = batch_of_size(N)
    dg = prepare_graph(g, DEV)
    dst = g.edges()[1].to(DEV)
    deg = deg_of(dst, N)
    w = step_weights(100 + N)
    fwd = Fwd(w)
    cases, prefix = [], {}
    total = None
    for t in range(T):
        c = StepCase(g, dg, fwd, seed=1000 * N + t)
        r = step_reference(c.s, c.h, deg, w, c.dh_part)
        del c.h, c.s, c.dh_part, c.o_img, c.h_out            # keep only what the kernels read
        cases.append(c)
        r = {k: v for k, v in r.items() if k not in ("ds", "dh")}
        total = r if total is None else {k: total[k] + r[k] for k in r}
        if t + 1 in (1, 8, 16):
            prefix[t + 1] = dict(total)
    L = lib()
    # (1) kept q images, one weight-gradient launch over the first T steps
    bwd = Bwd(fwd.w32, N, steps=T)
    for steps in (1, 8, 16):
        acc = Bwd.new_acc()
        for t in range(steps):
            bwd(cases[t].dh_part32, cases[t].h_img, cases[t].s_img, cases[t].gates, dg.indptr, acc, wgrad_mode=16 + t)
        L.call("ddfa_gru_bwd_wgrad_batched", ptr_array([_p(c.s_img) for c in cases[:steps]]), ptr_array([_p(c.h_img) for c in cases[:steps]]),
               steps, N, DIM, _p(acc["dwf"]), _p(acc["dwhh"]), _p(bwd.ws), bwd.wsb, st())
        torch.cuda.synchronize()
        check_outputs(f"wgrad batched N={N} T={steps}", acc, prefix[steps])
    # the batched form takes at most 16 steps, and a workspace with room for all of them
    s_ptrs, h_ptrs = [_p(c.s_img) for c in cases], [_p(c.h_img) for c in cases]
    with pytest.raises(DdfaError, match="steps"):
        L.call("ddfa_gru_bwd_wgrad_batched", ptr_array(s_ptrs + s_ptrs[:1]), ptr_array(h_ptrs + h_ptrs[:1]), 17, N, DIM,
               _p(acc["dwf"]), _p(acc["dwhh"]), _p(bwd.ws), bwd.wsb, st())
    short = L.call("ddfa_gru_step_bwd_workspace_bytes_steps", N, DIM, ENGINE_TCGEN05, T - 1)
    assert short < bwd.wsb
    with pytest.raises(DdfaError, match="workspace"):
        L.call("ddfa_gru_bwd_wgrad_batched", ptr_array(s_ptrs), ptr_array(h_ptrs), T, N, DIM, _p(acc["dwf"]), _p(acc["dwhh"]),
               _p(bwd.ws), short, st())
    c = cases[0]
    with pytest.raises(DdfaError, match="wgrad_mode"):      # there is no 17th slot
        bwd(c.dh_part32, c.h_img, c.s_img, c.gates, dg.indptr, acc, wgrad_mode=16 + T)
    with pytest.raises(DdfaError, match="workspace"):       # slot 15 needs the 16-slot workspace
        bwd(c.dh_part32, c.h_img, c.s_img, c.gates, dg.indptr, acc, wgrad_mode=16 + T - 1, wsb=short)
    del bwd
    # (2) deferred: per-CTA partials accumulated over the steps, added once by ddfa_gru_step_bwd_finish; (3) immediate
    bwd = Bwd(fwd.w32, N)
    for label, modes in (("deferred", [1] + [2] * (T - 1)), ("immediate", [0] * T)):
        acc = Bwd.new_acc()
        for c, mode in zip(cases, modes):
            bwd(c.dh_part32, c.h_img, c.s_img, c.gates, dg.indptr, acc, wgrad_mode=mode)
        if label == "deferred":
            L.call("ddfa_gru_step_bwd_finish", N, DIM, _p(acc["dwf"]), _p(acc["dwhh"]), _p(bwd.ws), bwd.wsb, st())
        torch.cuda.synchronize()
        check_outputs(f"wgrad {label} N={N} T={T}", acc, prefix[T])


def ggnn_case(g, T, seed, msg_scale=1.0):
    """fp64 GatedGraphConv on the GPU, its output and gradients for a random incoming gradient.  msg_scale shrinks
    linears[0] so that messages summed over thousands of in-edges do not saturate every gate."""
    torch.manual_seed(seed)
    conv = O.GatedGraphConvRestated(DIM, DIM, T).double().to(DEV)
    with torch.no_grad():
        conv.linears[0].bias.uniform_(-0.2, 0.2)          # DGL initialises it to zero; exercise the bias path
        conv.linears[0].weight.mul_(msg_scale)
        conv.linears[0].bias.mul_(msg_scale)
    N = g.num_nodes()
    x = (torch.randn(N, DIM, dtype=torch.float64, device=DEV) * 0.5).requires_grad_(True)
    h_ref = conv(g.to(DEV), x)
    dh_T = torch.randn(N, DIM, dtype=torch.float64, device=DEV)
    (h_ref * dh_T).sum().backward()
    par = dict(w_msg=conv.linears[0].weight, b_msg=conv.linears[0].bias, w_ih=conv.gru.weight_ih, w_hh=conv.gru.weight_hh,
               b_ih=conv.gru.bias_ih, b_hh=conv.gru.bias_hh)
    return x, h_ref.detach(), dh_T, par


def run_ggnn_drivers(label, g, dg, T, engines, x, h_ref, dh_T, par):
    """ddfa_ggnn_fwd / ddfa_ggnn_bwd against the fp64 references, with the bounds of test_kernels_gpu.py::test_ggnn_fused_drivers."""
    N = g.num_nodes()
    pd = {k: v.detach().float().contiguous() for k, v in par.items()}
    xd, dhd = x.detach().float().contiguous(), dh_T.float()
    L = lib()
    for engine in engines:
        wsb = L.call("ddfa_ggnn_workspace_bytes", N, DIM, T, engine, 1)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        h_out = torch.full((N, DIM), float("nan"), device=DEV)
        L.call("ddfa_ggnn_fwd", _p(dg.indptr), _p(dg.indices), _p(xd), N, DIM, T, _p(pd["w_msg"]), _p(pd["b_msg"]), _p(pd["w_ih"]),
               _p(pd["w_hh"]), _p(pd["b_ih"]), _p(pd["b_hh"]), _p(h_out), _p(ws), wsb, 1, engine, st())
        dx = torch.full((N, DIM), float("nan"), device=DEV)
        gr = {k: torch.zeros_like(v) for k, v in pd.items()}
        L.call("ddfa_ggnn_bwd", _p(dg.indptr), _p(dg.indptr_t), _p(dg.indices_t), _p(xd), N, DIM, T, _p(pd["w_msg"]), _p(pd["b_msg"]),
               _p(pd["w_ih"]), _p(pd["w_hh"]), _p(dhd), _p(dx), _p(gr["w_msg"]), _p(gr["b_msg"]), _p(gr["w_ih"]), _p(gr["w_hh"]),
               _p(gr["b_ih"]), _p(gr["b_hh"]), _p(ws), wsb, engine, st())
        torch.cuda.synchronize()
        name = "simt" if engine == ENGINE_SIMT else "tcgen05"
        err_h = float((h_out.double() - h_ref).abs().max())
        errs = {"dx": rel_err(dx, x.grad), **{k: rel_err(gr[k], par[k].grad) for k in par}}
        print(f"{label} T={T} {name}: |dh_T| abs={err_h:.1e}, " + ", ".join(f"{k}={v:.1e}" for k, v in errs.items()))
        assert err_h < (3e-5 if engine == ENGINE_SIMT else 2e-4) * T, (label, name, err_h)
        bound = (1e-4 if engine == ENGINE_SIMT else 5e-4) * T ** 0.5
        bad = {k: v for k, v in errs.items() if not v < bound}
        assert not bad, (label, name, bad)
        del ws


@pytest.mark.parametrize("T", [8, 18])
def test_ggnn_drivers_at_c0(T):
    """The whole GatedGraphConv behind ddfa_ggnn_fwd / ddfa_ggnn_bwd at C0 size; T = 18 takes the deferred weight-gradient path
    (more steps than the batched launch keeps)."""
    g = batch_of_size(C0_N)
    dg = prepare_graph(g, DEV)
    run_ggnn_drivers("ggnn C0", g, dg, T, [ENGINE_SIMT, ENGINE_TCGEN05], *ggnn_case(g, T, seed=T))


# ------------------------------------------------------------------------------------------------------------------------------
# D. degree extremes at D = 128
# ------------------------------------------------------------------------------------------------------------------------------
HUB_N = 10003                       # not a multiple of 4; the last tile is ragged
IN_HUBS = {0: 5000, 31: 33, 32: 32, 127: 31, 128: 1000, 4003: 64, 6001: 33, HUB_N - 1: 5000}
OUT_HUBS = {0: 1000, 31: 32, 32: 33, 127: 5000, 128: 31, 4003: 5000, 7002: 64, HUB_N - 1: 64}
# 4-row groups whose 33rd edge (index 32 from the group's first edge) lands in the 3rd row (1000..1003) and the 4th row (2000..2003)
GROUP_DEGREES = {1000: 10, 1001: 12, 1002: 20, 1003: 5, 2000: 8, 2001: 8, 2002: 8, 2003: 20}
NO_IN = [5, 129, 3001, 3002, 8190]          # zero in-degree
NO_OUT = [6, 130, 3003, 8191, 9999]         # zero out-degree
ISOLATED = [7, 4444, HUB_N - 2]             # neither


def hub_graph():
    rng = np.random.default_rng(17)
    N = HUB_N
    special = set(IN_HUBS) | set(OUT_HUBS) | set(GROUP_DEGREES)
    no_in, no_out = set(NO_IN) | set(ISOLATED), set(NO_OUT) | set(ISOLATED)
    assert not (special & (no_in | no_out))
    fixed_in = set(IN_HUBS) | set(GROUP_DEGREES)          # rows whose in-degree is exactly what the tables say
    fixed_out = set(OUT_HUBS)
    free_src = np.array(sorted(set(range(N)) - no_out - fixed_out))
    free_dst = np.array(sorted(set(range(N)) - no_in - fixed_in))
    src, dst = [], []
    # background: every free row gets ~2 in-edges from free sources (incl. self-loops where allowed)
    for _ in range(2):
        src.append(rng.choice(free_src, free_dst.shape[0])); dst.append(free_dst)
    for v, d in {**IN_HUBS, **GROUP_DEGREES}.items():
        s = rng.choice(free_src, d)
        s[:8] = s[0]                                        # a run of duplicate edges
        src.append(s); dst.append(np.full(d, v))
    for u, d in OUT_HUBS.items():
        t = rng.choice(free_dst, d)
        t[d // 2: d // 2 + 8] = t[d // 2]
        src.append(np.full(d, u)); dst.append(t)
    src, dst = np.concatenate(src), np.concatenate(dst)
    g = BatchedCFG(torch.from_numpy(src), torch.from_numpy(dst), torch.tensor([N]))
    indeg, outdeg = np.bincount(dst, minlength=N), np.bincount(src, minlength=N)
    for v, d in {**IN_HUBS, **GROUP_DEGREES}.items():
        assert indeg[v] == d, (v, indeg[v], d)
    for u, d in OUT_HUBS.items():
        assert outdeg[u] == d, (u, outdeg[u], d)
    assert (indeg[sorted(no_in)] == 0).all() and (outdeg[sorted(no_out)] == 0).all()
    return g


def self_loop_graph():
    N = 301
    loops = torch.arange(N)
    return BatchedCFG(loops.clone(), loops.clone(), torch.tensor([N]))


GRAPHS = {"hubs": hub_graph, "self_loops": self_loop_graph}


def tma_wait_timeouts():
    v = ctypes.c_int32(-1)
    lib().call("ddfa_debug_read", 4, ctypes.addressof(v), 4)
    return v.value


@pytest.mark.parametrize("graph", list(GRAPHS))
def test_gathers_at_degree_extremes(graph):
    """ddfa_gather_sum and every ddfa_gather_sum_variant (0-9 register shapes, 10 / 11 TMA-staged), forward and transposed with
    accumulate; ddfa_gather_sum_image (+ fp32 copy); ddfa_gather_sum_image_src with 1, 2 and 4 row groups per warp."""
    g = GRAPHS[graph]()
    dg = prepare_graph(g, DEV)
    N = g.num_nodes()
    src, dst = [t.to(DEV) for t in g.edges()]
    gen = torch.Generator(device=DEV).manual_seed(5)
    h = torch.randn(N, DIM, device=DEV, generator=gen)
    base = torch.randn(N, DIM, device=DEV, generator=gen)
    ref = torch.zeros(N, DIM, dtype=torch.float64, device=DEV).index_add_(0, dst, h.double()[src])
    ref_t = base.double() + transposed_gather(src, dst, h.double())
    L = lib()
    before = tma_wait_timeouts()
    worst = {}
    outs = {}
    for variant in [None] + list(range(12)):
        out, out_t = torch.full_like(h, float("nan")), base.clone()
        if variant is None:
            L.call("ddfa_gather_sum", _p(dg.indptr), _p(dg.indices), _p(h), N, DIM, _p(out), 0, st())
            L.call("ddfa_gather_sum", _p(dg.indptr_t), _p(dg.indices_t), _p(h), N, DIM, _p(out_t), 1, st())
        else:
            L.call("ddfa_gather_sum_variant", variant, _p(dg.indptr), _p(dg.indices), _p(h), N, DIM, _p(out), 0, st())
            L.call("ddfa_gather_sum_variant", variant, _p(dg.indptr_t), _p(dg.indices_t), _p(h), N, DIM, _p(out_t), 1, st())
        torch.cuda.synchronize()
        worst[variant] = (rel_err(out, ref), rel_err(out_t, ref_t))     # forward, transposed + accumulate
        outs[variant] = (out, out_t)
    after = tma_wait_timeouts()
    # fp32 rounding of an n-term sum grows like sqrt(n) against the result's scale: the 1e-5 of test_kernels_gpu.py holds for the
    # <= 82-edge rows there; it is widened by that factor for the 5 000-edge rows here (every variant sums in neighbour order)
    max_deg = int(max(torch.bincount(dst, minlength=N).max(), torch.bincount(src, minlength=N).max()))
    tol = 1e-5 * max(1.0, (max_deg / 500) ** 0.5)
    print(f"gather {graph} N={N} (max degree {max_deg}, bound {tol:.1e}): worst rel. error (forward / transposed) per variant "
          + ", ".join(f"{k if k is not None else 'default'}={a:.1e}/{b:.1e}" for k, (a, b) in worst.items())
          + f"; timed-out TMA waits before / after: {before} / {after}")
    assert before == 0 and after == 0
    bad = {k: v for k, v in worst.items() if not (v[0] < tol and v[1] < tol)}      # NaN (an unwritten row) fails too
    assert not bad, bad
    for v in (10, 11):              # gather_tma.cu: same summation order as the register variant 9
        assert torch.equal(outs[v][0], outs[9][0]) and torch.equal(outs[v][1], outs[9][1]), v
    # fp32 source -> image (+ fp32 copy)
    s_img = torch.zeros(L.call("ddfa_act_image_bytes", N), dtype=torch.uint8, device=DEV)
    s_f = torch.empty(N, DIM, device=DEV)
    L.call("ddfa_gather_sum_image", _p(dg.indptr), _p(dg.indices), _p(h), N, DIM, _p(s_img), _p(s_f), st())
    e_f32, e_img = rel_err(s_f, ref), rel_err(decode_image(s_img, N, DEV), ref)
    # image source -> image, 1 / 2 / 4 row groups per warp
    h_img = image_of(h)
    hd = decode_image(h_img, N, DEV)
    ref_i = torch.zeros_like(hd).index_add_(0, dst, hd[src])
    imgs = {}
    try:
        for groups in (1, 2, 4):
            L.call("ddfa_tuning_set", TUNE_GATHER_SRC_GROUPS, groups)
            imgs[groups] = gather_image_src(dg, h_img, N)
    finally:
        L.call("ddfa_tuning_set", TUNE_GATHER_SRC_GROUPS, 0)
    e_src = rel_err(decode_image(imgs[1], N, DEV), ref_i)
    print(f"gather image {graph}: fp32 copy {e_f32:.1e}, image {e_img:.1e}; image source {e_src:.1e}")
    assert e_f32 < tol and e_img < 2 * tol and e_src < 2 * tol
    assert torch.equal(imgs[2], imgs[1]) and torch.equal(imgs[4], imgs[1])


@pytest.mark.parametrize("graph", list(GRAPHS))
def test_step_at_degree_extremes(graph):
    """The forward step (its deg x b_fold term at in-degree 0 and 5 000) and the backward with the folded transposed gather (out-edge
    lists far past the two prefetched neighbours) in all three gate-backward modes.  w_fold and b_fold are scaled down so the
    gates stay out of saturation at the hubs and both terms stay visible in h' there; a second forward with b_fold at full scale
    pins the term at in-degrees 0 to 3."""
    g = GRAPHS[graph]()
    dg = prepare_graph(g, DEV)
    N = g.num_nodes()
    src, dst = [t.to(DEV) for t in g.edges()]
    deg = deg_of(dst, N)
    w = step_weights(21, wf_scale=0.05, bf_scale=2e-3)
    fwd = Fwd(w)
    c = StepCase(g, dg, fwd, seed=9)
    h_ref, r_ref, z_ref, n_ref, ghn_ref = gru_reference(c.s, c.h, deg, *w)
    err_h = float((decode_image(c.o_img, N, DEV) - h_ref).abs().max())
    err_h32 = float((c.h_out.double() - h_ref).abs().max())
    gk = decode_gates(c.gates, N, DEV)
    err_g = [float((a - b).abs().max()) for a, b in zip(gk[:3], (r_ref, z_ref, n_ref))] + [rel_err(gk[3], ghn_ref)]
    print(f"step fwd {graph}: |dh'| image {err_h:.1e} fp32 {err_h32:.1e}; gates r/z/n/gh_n " + ", ".join(f"{e:.1e}" for e in err_g))
    assert err_h < 1e-4 and err_h32 < 1e-4 and all(e < 1.5e-4 for e in err_g)
    if graph == "hubs":             # the deg x b_fold term moves h' at the 5 000-edge hub: the check above would see it missing
        no_bias = gru_reference(c.s, c.h, torch.zeros_like(deg), *w)[0]
        assert float((no_bias[HUB_N - 1] - h_ref[HUB_N - 1]).abs().max()) > 1e-2
        assert int((deg == 0).sum()) >= len(NO_IN) + len(ISOLATED)
    # the same forward with b_fold at full scale, where one in-edge more or less moves h' of every low-degree row (in-degree 0 to 3)
    # by far more than the bound: a kernel that got those degrees wrong would fail here
    w_b = step_weights(22, wf_scale=0.05)
    h_b = Fwd(w_b)(c.s_img, c.h_img, dg.indptr, N)[2]
    ref_b = gru_reference(c.s, c.h, deg, *w_b)[0]
    err_b = float((h_b.double() - ref_b).abs().max())
    shift = (gru_reference(c.s, c.h, deg + 1, *w_b)[0] - ref_b).abs().amax(1)[deg <= 3]
    print(f"step fwd {graph}, full-scale b_fold: |dh'| {err_b:.1e}; smallest effect of one extra in-edge on a row of in-degree <= 3: "
          f"{float(shift.min()):.1e}")
    assert err_b < 1e-4 and float(shift.min()) > 1e-3
    ds_prev = torch.randn(N, DIM, device=DEV, generator=torch.Generator(device=DEV).manual_seed(10)).float()
    ref = step_reference(c.s, c.h, deg, w, c.dh_part + transposed_gather(src, dst, ds_prev.double()))
    bwd = Bwd(fwd.w32, N)
    outs = {}
    try:
        for mode in (2, 1, 0):
            lib().call("ddfa_tuning_set", TUNE_GATE_BWD_TMA, mode)
            acc = Bwd.new_acc()
            ds, dh = bwd(c.dh_part32, c.h_img, c.s_img, c.gates, dg.indptr, acc, ds_prev, dg.indptr_t, dg.indices_t)
            torch.cuda.synchronize()
            check_outputs(f"step bwd {graph} tma_mode={mode}", dict(ds=ds, dh=dh, **acc), ref)
            outs[mode] = (ds, dh)
    finally:
        lib().call("ddfa_tuning_set", TUNE_GATE_BWD_TMA, 2)
    for mode in (1, 0):
        assert torch.equal(outs[mode][0], outs[2][0]) and torch.equal(outs[mode][1], outs[2][1]), (graph, mode)


@pytest.mark.parametrize("graph", list(GRAPHS))
def test_ggnn_drivers_at_degree_extremes(graph):
    g = GRAPHS[graph]()
    dg = prepare_graph(g, DEV)
    run_ggnn_drivers(f"ggnn {graph}", g, dg, 3, [ENGINE_SIMT, ENGINE_TCGEN05], *ggnn_case(g, 3, seed=4, msg_scale=0.05))


# ------------------------------------------------------------------------------------------------------------------------------
# E. module gradients at C1
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("engine", ["simt", "tcgen05"])
@pytest.mark.parametrize("variable", [False, True])
def test_module_gradients_at_c1(engine, variable):
    """FlowGNNGGNNModule.training_step + backward at 1024 CFGs x 150 nodes (fixed and lognormal sizes) against the fp64 oracle
    run on the GPU, per parameter.  The head is one linear layer: with ReLU layers, 1024 graphs put hidden pre-activations within
    1e-7 of zero, where a forward difference of that size flips a ReLU and moves whole gradients by 1e-3 (measured); the
    kernels' gradients are only comparable where the loss is smooth.  The ReLU head's backward at this batch size is checked by
    test_mlp_head_backward_at_c1_batch, on the reference's own activations."""
    g = synth.make_batch(1024, 150, seed=5, variable=variable, vuln_rate=0.3)
    gd = g.to(DEV)
    torch.manual_seed(1)
    o = O.OracleFlowGNNGGNN(FEAT, 1002, 32, 8, 1, concat_all_absdf=True, positive_weight=4.0).double().to(DEV)
    loss_ref, _ = o.training_loss(gd)
    loss_ref.backward()
    m = D.FlowGNNGGNNModule(FEAT, 1002, 32, 8, 1, concat_all_absdf=True, positive_weight=4.0, engine=engine)
    m.load_state_dict({k: v.float() for k, v in o.state_dict().items()})
    m.to(DEV)
    loss = m.training_step((gd, {}), 0)
    loss.backward()
    assert abs(float(loss.detach()) - float(loss_ref.detach())) < 1e-4
    worst = {}
    for (name, p), (_, q) in zip(m.named_parameters(), o.named_parameters()):
        scale = max(float(q.grad.abs().max()), 1e-3)      # pooling.gate_nn.bias: true gradient 0 (shift-invariant softmax)
        worst[name] = float((p.grad.double() - q.grad).abs().max()) / scale
    print(f"module gradients C1 N={g.num_nodes()} engine={engine}: " + ", ".join(f"{k}={v:.1e}" for k, v in worst.items()))
    bad = {k: v for k, v in worst.items() if not v < GRAD_TOL[engine]}
    assert not bad, bad


@pytest.mark.parametrize("L", [2, 3])
def test_mlp_head_backward_at_c1_batch(L):
    """ddfa_mlp_bwd (the output MLP's backward, ReLU between layers) at the C1 batch of 1024 graphs against fp64 autograd.  The
    kernel is handed the reference's own post-ReLU activations, so both sides use the same ReLU masks and the comparison holds
    even for pre-activations next to zero."""
    B, D2 = 1024, 2 * DIM
    torch.manual_seed(30 + L)
    lins = [torch.nn.Linear(D2, 1 if i == L - 1 else D2).double().to(DEV) for i in range(L)]
    pooled = torch.randn(B, D2, dtype=torch.float64, device=DEV).float().double().requires_grad_(True)
    cur, acts = pooled, []
    for i, lin in enumerate(lins):
        cur = lin(cur)
        if i != L - 1:
            cur = torch.relu(cur)
            acts.append(cur)
    dout = torch.randn(B, dtype=torch.float64, device=DEV).float()
    (cur.squeeze(-1) * dout.double()).sum().backward()
    mw = [m.weight.detach().float().contiguous() for m in lins]
    act = torch.stack([a.detach().float() for a in acts]).contiguous()
    p32 = pooled.detach().float().contiguous()
    dpooled, scratch = torch.empty(B, D2, device=DEV), torch.empty(2, B, D2, device=DEV)
    gw, gb = [torch.zeros_like(t) for t in mw], [torch.zeros(t.shape[0], device=DEV) for t in mw]
    lib().call("ddfa_mlp_bwd", _p(dout), _p(p32), _p(act), ptr_array([_p(t) for t in mw]), B, DIM, L, _p(dpooled),
               ptr_array([_p(t) for t in gw]), ptr_array([_p(t) for t in gb]), _p(scratch), st())
    torch.cuda.synchronize()
    errs = {"dpooled": rel_err(dpooled, pooled.grad)}
    for i, m in enumerate(lins):
        errs[f"w{i}"], errs[f"b{i}"] = rel_err(gw[i], m.weight.grad), rel_err(gb[i], m.bias.grad)
    print(f"mlp head backward B={B} L={L}: " + ", ".join(f"{k}={v:.1e}" for k, v in errs.items()))
    bad = {k: v for k, v in errs.items() if not v < 1e-4}
    assert not bad, bad
