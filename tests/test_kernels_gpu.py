"""GPU: every C-ABI entry point against the oracle's building blocks on the same seeded inputs.
All calls go through libddfa_b200.so (ctypes); torch only holds the device buffers."""
import numpy as np
import pytest
import torch

from deepdfa_b200 import synth
from deepdfa_b200._lib import ENGINE_SIMT, ENGINE_TCGEN05, DdfaError, lib, ptr_array
from deepdfa_b200.engine import _p, _stream_ptr, prepare_graph
from oracle import ggnn_oracle as O
from parity_helpers import decode_gates, decode_image
from parity_helpers import gru_reference as _gru_reference

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def dev(t):
    return t.to(DEV).contiguous()


_KEEP = []


def dk(t):
    """dev() for tensors passed inline as pointers: keeps the device tensor alive so two temporaries in one call
    can never alias through the caching allocator."""
    x = dev(t)
    _KEEP.append(x)
    if len(_KEEP) > 64:
        torch.cuda.synchronize()
        del _KEEP[:32]
    return x


def st():
    return _stream_ptr()


def engines_for(D):
    tc = lib().call("ddfa_engine_available", ENGINE_TCGEN05) == 1
    return [ENGINE_SIMT, ENGINE_TCGEN05] if (D == 128 and tc) else [ENGINE_SIMT]


# ---------------------------------------------------------------------------------------------
def test_device_is_blackwell():
    assert lib().call("ddfa_device_supported") == 1


@pytest.mark.parametrize("idx_dtype", [torch.int64, torch.int32])
def test_build_csr_matches_numpy(idx_dtype):
    rng = np.random.default_rng(0)
    N, E = 1000, 5000
    src = rng.integers(0, N, E); dst = rng.integers(0, N, E)
    dst[:600] = 7            # a hub row with a long neighbour list
    src[100:200] = 3         # duplicates
    s, d = dev(torch.from_numpy(src).to(idx_dtype)), dev(torch.from_numpy(dst).to(idx_dtype))
    L = lib()
    indptr = torch.empty(N + 1, dtype=torch.int32, device=DEV); indices = torch.empty(E, dtype=torch.int32, device=DEV)
    indptr_t = torch.empty_like(indptr); indices_t = torch.empty_like(indices)
    wsb = L.call("ddfa_build_csr_workspace_bytes", E, N)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    L.call("ddfa_build_csr", _p(s), _p(d), s.element_size(), E, N, _p(indptr), _p(indices), _p(indptr_t), _p(indices_t), _p(ws), wsb, st())
    torch.cuda.synchronize()
    order = np.lexsort((src, dst))
    assert np.array_equal(indices.cpu().numpy(), src[order])
    assert np.array_equal(indptr.cpu().numpy(), np.concatenate([[0], np.cumsum(np.bincount(dst, minlength=N))]))
    order_t = np.lexsort((dst, src))
    assert np.array_equal(indices_t.cpu().numpy(), dst[order_t])
    assert np.array_equal(indptr_t.cpu().numpy(), np.concatenate([[0], np.cumsum(np.bincount(src, minlength=N))]))
    assert int(ws[:4].view(torch.int32)[0]) == 0


def test_build_csr_large_scan_empty_and_out_of_range():
    L = lib()
    # > 4096 rows exercises the multi-pass scan carry
    g = synth.make_batch(200, 150, seed=3, variable=True)
    dg = prepare_graph(g, DEV)
    src, dst = [t.numpy() for t in g.edges()]
    torch.cuda.synchronize()
    assert np.array_equal(dg.indptr.cpu().numpy(), np.concatenate([[0], np.cumsum(np.bincount(dst, minlength=g.num_nodes()))]))
    assert np.array_equal(dg.indices.cpu().numpy()[: g.num_edges()], src[np.lexsort((src, dst))])
    assert np.array_equal(dg.graph_ptr.cpu().numpy(), np.concatenate([[0], np.cumsum(g.batch_num_nodes().numpy())]))
    # the multi-CTA scan (N > 16 384 rows: block sums -> scan of the sums -> per-block scan) at ragged sizes, both orientations
    rng = np.random.default_rng(5)
    for N, E in ((16385, 40000), (20481, 30000), (153677, 307201), (70000, 18)):
        src = rng.integers(0, N, E); dst = rng.integers(0, N, E)
        s, d = dev(torch.from_numpy(src)), dev(torch.from_numpy(dst))
        indptr = torch.empty(N + 1, dtype=torch.int32, device=DEV); indices = torch.empty(E, dtype=torch.int32, device=DEV)
        indptr_t = torch.empty_like(indptr); indices_t = torch.empty_like(indices)
        wsb = L.call("ddfa_build_csr_workspace_bytes", E, N); ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        L.call("ddfa_build_csr", _p(s), _p(d), 8, E, N, _p(indptr), _p(indices), _p(indptr_t), _p(indices_t), _p(ws), wsb, st())
        torch.cuda.synchronize()
        assert np.array_equal(indptr.cpu().numpy(), np.concatenate([[0], np.cumsum(np.bincount(dst, minlength=N))])), (N, E)
        assert np.array_equal(indptr_t.cpu().numpy(), np.concatenate([[0], np.cumsum(np.bincount(src, minlength=N))])), (N, E)
        assert np.array_equal(indices.cpu().numpy(), src[np.lexsort((src, dst))]) and np.array_equal(indices_t.cpu().numpy(), dst[np.lexsort((dst, src))])
    # empty edge list
    indptr = torch.full((6,), -1, dtype=torch.int32, device=DEV); indices = torch.empty(1, dtype=torch.int32, device=DEV)
    wsb = L.call("ddfa_build_csr_workspace_bytes", 0, 5); ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    L.call("ddfa_build_csr", None, None, 8, 0, 5, _p(indptr), _p(indices), None, None, _p(ws), wsb, st())
    assert indptr.cpu().tolist() == [0] * 6
    # out-of-range ids are dropped and counted
    s = dev(torch.tensor([0, 1, 9, 2])); d = dev(torch.tensor([1, 2, 0, -1]))
    indptr = torch.empty(4, dtype=torch.int32, device=DEV); indices = torch.zeros(4, dtype=torch.int32, device=DEV)
    wsb = L.call("ddfa_build_csr_workspace_bytes", 4, 3); ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    L.call("ddfa_build_csr", _p(s), _p(d), 8, 4, 3, _p(indptr), _p(indices), None, None, _p(ws), wsb, st())
    assert indptr.cpu().tolist() == [0, 0, 1, 2] and indices.cpu().tolist()[:2] == [0, 1]
    assert int(ws[:4].view(torch.int32)[0]) == 2
    with pytest.raises(DdfaError, match="workspace"):
        L.call("ddfa_build_csr", _p(s), _p(d), 8, 4, 3, _p(indptr), _p(indices), None, None, _p(ws), 8, st())


@pytest.mark.parametrize("D", [20, 32, 64, 128, 256, 512, 1024])
def test_gather_sum_matches_index_add(D):
    g = synth.make_edge_cases() if D != 128 else synth.make_batch(64, 150, seed=1, variable=True)
    dg = prepare_graph(g, DEV)
    N = g.num_nodes()
    torch.manual_seed(D)
    h = torch.randn(N, D)
    src, dst = g.edges()
    ref = torch.zeros(N, D, dtype=torch.float64).index_add_(0, dst, h.double()[src])
    hd, out = dev(h), torch.empty(N, D, device=DEV)
    lib().call("ddfa_gather_sum", _p(dg.indptr), _p(dg.indices), _p(hd), N, D, _p(out), 0, st())
    assert (out.cpu().double() - ref).abs().max() < 1e-5 * max(1.0, float(ref.abs().max()))
    # accumulate over the transposed graph = backward of the op
    base = torch.randn(N, D)
    ref_t = base.double() + torch.zeros(N, D, dtype=torch.float64).index_add_(0, src, h.double()[dst])
    out2 = dev(base)
    lib().call("ddfa_gather_sum", _p(dg.indptr_t), _p(dg.indices_t), _p(hd), N, D, _p(out2), 1, st())
    assert (out2.cpu().double() - ref_t).abs().max() < 1e-5 * max(1.0, float(ref_t.abs().max()))


def test_gather_sum_is_deterministic_and_rejects_bad_shapes():
    g = synth.make_batch(64, 150, seed=1)
    dg = prepare_graph(g, DEV)
    h = torch.randn(g.num_nodes(), 128, device=DEV)
    a, b = torch.empty_like(h), torch.empty_like(h)
    for o in (a, b):
        lib().call("ddfa_gather_sum", _p(dg.indptr), _p(dg.indices), _p(h), g.num_nodes(), 128, _p(o), 0, st())
    assert torch.equal(a, b)
    with pytest.raises(DdfaError, match="D=130"):
        lib().call("ddfa_gather_sum", _p(dg.indptr), _p(dg.indices), _p(h), 10, 130, _p(a), 0, st())
    with pytest.raises(DdfaError, match="in-place"):
        lib().call("ddfa_gather_sum", _p(dg.indptr), _p(dg.indices), _p(h), 10, 128, _p(h), 0, st())


@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("shape", [(300, 384, 128), (37, 5, 19), (384, 128, 5000), (1, 256, 200), (256, 1, 256)])
def test_sgemm(ta, tb, shape):
    M, N, K = shape
    torch.manual_seed(M * 7 + N)
    A = torch.randn((K, M) if ta else (M, K)); B = torch.randn((N, K) if tb else (K, N)); C0 = torch.randn(M, N)
    opA = A.t() if ta else A; opB = B.t() if tb else B
    ref = 0.5 * opA.double() @ opB.double() + 2.0 * C0.double()
    Ad, Bd, Cd = dev(A), dev(B), dev(C0)
    lib().call("ddfa_sgemm", ta, tb, M, N, K, 0.5, _p(Ad), A.shape[1], _p(Bd), B.shape[1], 2.0, _p(Cd), N, 1, st())
    tol = 1e-5 * (K ** 0.5) * 4
    assert (Cd.cpu().double() - ref).abs().max() < tol * max(1.0, float(ref.abs().max()) / 10)
    # split-K accumulates into C (beta must be 1)
    Cd = dev(C0)
    lib().call("ddfa_sgemm", ta, tb, M, N, K, 1.0, _p(Ad), A.shape[1], _p(Bd), B.shape[1], 1.0, _p(Cd), N, 7, st())
    ref2 = opA.double() @ opB.double() + C0.double()
    assert (Cd.cpu().double() - ref2).abs().max() < tol * max(1.0, float(ref2.abs().max()) / 10)
    with pytest.raises(DdfaError, match="beta"):
        lib().call("ddfa_sgemm", ta, tb, M, N, K, 1.0, _p(Ad), A.shape[1], _p(Bd), B.shape[1], 0.0, _p(Cd), N, 4, st())


@pytest.mark.parametrize("K,H", [(4, 32), (1, 32), (4, 8), (1, 20)])
def test_embed_concat_fwd_bwd(K, H):
    V, N = 50, 3000
    torch.manual_seed(K * 100 + H)
    tables = [torch.randn(V, H) for _ in range(K)]
    g = synth.make_batch(sizes=[N], input_dim=V, seed=K)
    idx = [g.ndata[f"_ABS_DATAFLOW_{k}"] for k in ("api", "datatype", "literal", "operator")][:K]
    ref = torch.cat([t[i] for t, i in zip(tables, idx)], 1)
    td, idd = [dev(t) for t in tables], [dev(i) for i in idx]
    x = torch.empty(N, K * H, device=DEV); oob = torch.zeros(1, dtype=torch.int32, device=DEV)
    lib().call("ddfa_embed_concat_fwd", ptr_array([_p(i) for i in idd]), ptr_array([_p(t) for t in td]), K, V, H, N, _p(x), _p(oob), st())
    assert torch.equal(x.cpu(), ref) and int(oob) == 0
    if K * H == 128:      # fused form: the same rows AND h_0's activation image, bit-equal to a separate ddfa_act_to_image pass
        ib = lib().call("ddfa_act_image_bytes", N)
        img_a, img_b = torch.zeros(ib, dtype=torch.uint8, device=DEV), torch.zeros(ib, dtype=torch.uint8, device=DEV)
        x2 = torch.empty_like(x)
        lib().call("ddfa_embed_concat_fwd_image", ptr_array([_p(i) for i in idd]), ptr_array([_p(t) for t in td]), K, V, H, N, _p(x2), _p(img_a), _p(oob), st())
        lib().call("ddfa_act_to_image", _p(x), N, K * H, _p(img_b), st())
        assert torch.equal(x2, x) and torch.equal(img_a, img_b) and int(oob) == 0
        with pytest.raises(DdfaError, match="NULL image"):
            lib().call("ddfa_embed_concat_fwd_image", ptr_array([_p(i) for i in idd]), ptr_array([_p(t) for t in td]), K, V, H, N, _p(x2), None, _p(oob), st())
    dx, dx2 = torch.randn(N, K * H), torch.randn(N, K * H)
    dx_d, dx2_d = dev(dx), dev(dx2)          # keep the device tensors alive across the call (no aliasing temporaries)
    for second in (None, dx2):
        tot = dx + (second if second is not None else 0)
        ref_g = [torch.zeros(V, H, dtype=torch.float64).index_add_(0, i, tot[:, k * H:(k + 1) * H].double()) for k, i in enumerate(idx)]
        gd = [torch.zeros(V, H, device=DEV) for _ in range(K)]
        lib().call("ddfa_embed_concat_bwd", ptr_array([_p(i) for i in idd]), _p(dx_d), _p(dx2_d) if second is not None else None,
                   K, V, H, N, ptr_array([_p(t) for t in gd]), st())
        for a, b in zip(gd, ref_g):
            assert (a.cpu().double() - b).abs().max() < 2e-4 * max(1.0, float(b.abs().max()))
    # out-of-range indices are clamped and counted
    bad = [i.clone() for i in idx]; bad[0][5] = V + 3; bad[0][6] = -2
    lib().call("ddfa_embed_concat_fwd", ptr_array([_p(dk(i)) for i in bad]), ptr_array([_p(t) for t in td]), K, V, H, N, _p(x), _p(oob), st())
    assert int(oob) == 2


def test_fold_weights_fwd_bwd():
    D = 128
    torch.manual_seed(5)
    W = torch.randn(D, D, dtype=torch.float64, requires_grad=True); b = torch.randn(D, dtype=torch.float64, requires_grad=True)
    Wih = torch.randn(3 * D, D, dtype=torch.float64, requires_grad=True)
    wf, bf = Wih @ W, Wih @ b
    dwf, dbf = torch.randn(3 * D, D, dtype=torch.float64), torch.randn(3 * D, dtype=torch.float64)
    ((wf * dwf).sum() + (bf * dbf).sum()).backward()
    Wd, bd, Wihd = dev(W.detach().float()), dev(b.detach().float()), dev(Wih.detach().float())
    wfd, bfd = torch.empty(3 * D, D, device=DEV), torch.empty(3 * D, device=DEV)
    lib().call("ddfa_fold_weights_fwd", _p(Wd), _p(bd), _p(Wihd), D, _p(wfd), _p(bfd), st())
    assert (wfd.cpu().double() - wf.detach()).abs().max() < 1e-3 and (bfd.cpu().double() - bf.detach()).abs().max() < 1e-3
    gW, gb, gWih = torch.ones(D, D, device=DEV), torch.ones(D, device=DEV), torch.ones(3 * D, D, device=DEV)   # += semantics
    lib().call("ddfa_fold_weights_bwd", _p(Wd), _p(bd), _p(Wihd), _p(dk(dwf.float())), _p(dk(dbf.float())), D, _p(gW), _p(gb), _p(gWih), st())
    for got, ref in ((gW, W.grad), (gb, b.grad), (gWih, Wih.grad)):
        assert (got.cpu().double() - 1.0 - ref).abs().max() < 1e-3 * max(1.0, float(ref.abs().max()) / 10)


@pytest.mark.parametrize("D", [32, 128, 256])
def test_gru_step_fwd_bwd(D):
    g = synth.make_batch(24, 60, seed=2, variable=True)
    dg = prepare_graph(g, DEV)
    N = g.num_nodes()
    torch.manual_seed(D)
    k = 1.0 / D ** 0.5
    mk = lambda *sh: (torch.rand(*sh, dtype=torch.float64) * 2 - 1) * k
    wf, bf, bih, whh, bhh = mk(3 * D, D) * 1.5, mk(3 * D), mk(3 * D), mk(3 * D, D), mk(3 * D)
    s = torch.randn(N, D, dtype=torch.float64) * 2; h = torch.tanh(torch.randn(N, D, dtype=torch.float64))
    deg = torch.bincount(g.edges()[1], minlength=N).double()
    leaves = [t.requires_grad_(True) for t in (s, h, wf, bf, bih, whh, bhh)]
    h_ref, r_ref, z_ref, n_ref, ghn_ref = _gru_reference(*leaves[:2], deg, *leaves[2:])
    dh_out = torch.randn(N, D, dtype=torch.float64)
    (h_ref * dh_out).sum().backward()
    f32 = [dev(t.detach().float()) for t in leaves]
    sd, hd, wfd, bfd, bihd, whhd, bhhd = f32
    for engine in engines_for(D):
        L = lib()
        wsb = max(L.call("ddfa_gru_step_workspace_bytes", N, D, engine), 16)
        ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
        L.call("ddfa_gru_step_prepare", _p(wfd), _p(bfd), _p(bihd), _p(whhd), _p(bhhd), D, engine, _p(ws), wsb, st())
        wsb_b = max(L.call("ddfa_gru_step_bwd_workspace_bytes", N, D, engine), 16)
        ws_b = torch.empty(wsb_b, dtype=torch.uint8, device=DEV)
        L.call("ddfa_gru_step_prepare_bwd", _p(wfd), _p(whhd), D, engine, _p(ws_b), wsb_b, st())
        h_out = torch.empty(N, D, device=DEV); gates = torch.empty(4, N, D, device=DEV)
        L.call("ddfa_gru_step_fwd", _p(sd), _p(hd), _p(dg.indptr), _p(wfd), _p(bfd), _p(bihd), _p(whhd), _p(bhhd), N, D, _p(h_out),
               _p(gates), _p(ws), wsb, engine, st())
        # SIMT: fp32 FFMA + accurate expf/tanhf; tcgen05: bf16x3 operands (~2^-16 rel.) + ex2.approx gate math
        tol_h = 2e-5 if engine == ENGINE_SIMT else 1e-4
        assert (h_out.cpu().double() - h_ref.detach()).abs().max() < tol_h, f"engine {engine}"
        for got, ref in zip(gates.cpu().double(), (r_ref, z_ref, n_ref, ghn_ref)):
            assert (got - ref.detach()).abs().max() < 2.5 * tol_h
        # without gate saving
        h_out2 = torch.empty(N, D, device=DEV)
        L.call("ddfa_gru_step_fwd", _p(sd), _p(hd), _p(dg.indptr), _p(wfd), _p(bfd), _p(bihd), _p(whhd), _p(bhhd), N, D, _p(h_out2),
               None, _p(ws), wsb, engine, st())
        assert torch.equal(h_out, h_out2)
        # backward
        ds, dh = torch.empty(N, D, device=DEV), torch.empty(N, D, device=DEV)
        acc = {n_: torch.zeros(sh, device=DEV) for n_, sh in (("dwf", (3 * D, D)), ("dbf", (3 * D,)), ("dbih", (3 * D,)), ("dwhh", (3 * D, D)), ("dbhh", (3 * D,)))}
        L.call("ddfa_gru_step_bwd", _p(dk(dh_out.float())), _p(hd), _p(sd), _p(gates), _p(dg.indptr), _p(wfd), _p(whhd), N, D, _p(ds), _p(dh),
               _p(acc["dwf"]), _p(acc["dbf"]), _p(acc["dbih"]), _p(acc["dwhh"]), _p(acc["dbhh"]), _p(ws_b), wsb_b, engine, st())
        checks = [(ds, s.grad), (dh, h.grad), (acc["dwf"], wf.grad), (acc["dbf"], bf.grad), (acc["dbih"], bih.grad), (acc["dwhh"], whh.grad), (acc["dbhh"], bhh.grad)]
        for got, ref in checks:
            scale = max(1.0, float(ref.abs().max()))
            assert (got.cpu().double() - ref).abs().max() < 2e-4 * scale, f"engine {engine}"
    with pytest.raises(DdfaError, match="tcgen05"):
        lib().call("ddfa_gru_step_fwd", _p(sd), _p(hd), _p(dg.indptr), _p(wfd), _p(bfd), _p(bihd), _p(whhd), _p(bhhd), N, 64 if D != 64 else 32,
                   _p(h_out), None, _p(ws), wsb, ENGINE_TCGEN05, st())


@pytest.mark.parametrize("graphs,nodes", [(3, 50), (24, 60), (40, 150)])     # N = 150 (2 tiles, ragged) .. 6000 (47 tiles)
def test_gru_step_image_entries(graphs, nodes):
    """The image-level entry points the training driver uses (tcgen05 engine): gather -> image, forward on images, backward
    on images with the transposed gather of the previous step's ds folded in — against fp64 autograd of the same math."""
    D = 128
    g = synth.make_batch(graphs, nodes, seed=graphs, variable=True)
    dg = prepare_graph(g, DEV)
    N = g.num_nodes()
    src, dst = g.edges()
    torch.manual_seed(graphs)
    k = 1.0 / D ** 0.5
    mk = lambda *sh: (torch.rand(*sh, dtype=torch.float64) * 2 - 1) * k
    wf, bf, bih, whh, bhh = mk(3 * D, D) * 1.5, mk(3 * D), mk(3 * D), mk(3 * D, D), mk(3 * D)
    h = torch.tanh(torch.randn(N, D, dtype=torch.float64))
    deg = torch.bincount(dst, minlength=N).double()
    dh_part = torch.randn(N, D, dtype=torch.float64)
    ds_prev = torch.randn(N, D, dtype=torch.float64)
    leaves = [t.requires_grad_(True) for t in (h, wf, bf, bih, whh, bhh)]
    s_ref = torch.zeros(N, D, dtype=torch.float64).index_add(0, dst, leaves[0][src])            # s = A h
    s_leaf = s_ref.detach().requires_grad_(True)
    h_ref, r_ref, z_ref, n_ref, ghn_ref = _gru_reference(s_leaf, leaves[0], deg, *leaves[1:])
    # incoming gradient of the step = dh_part + A^T ds_prev
    dh_in = dh_part + torch.zeros(N, D, dtype=torch.float64).index_add(0, src, ds_prev[dst])
    (h_ref * dh_in).sum().backward()
    L = lib()
    hd, wfd, bfd, bihd, whhd, bhhd = [dev(t.detach().float()) for t in leaves]
    ib = L.call("ddfa_act_image_bytes", N)
    assert ib == ((N + 127) // 128) * 65536
    h_img = torch.zeros(ib, dtype=torch.uint8, device=DEV); s_img = torch.zeros(ib, dtype=torch.uint8, device=DEV)
    o_img = torch.zeros(ib, dtype=torch.uint8, device=DEV); s_f = torch.empty(N, D, device=DEV)
    L.call("ddfa_act_to_image", _p(hd), N, D, _p(h_img), st())
    L.call("ddfa_gather_sum_image", _p(dg.indptr), _p(dg.indices), _p(hd), N, D, _p(s_img), _p(s_f), st())
    assert (s_f.cpu().double() - s_ref.detach()).abs().max() < 1e-5
    wsb = L.call("ddfa_gru_step_workspace_bytes", N, D, ENGINE_TCGEN05)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    L.call("ddfa_gru_step_prepare", _p(wfd), _p(bfd), _p(bihd), _p(whhd), _p(bhhd), D, ENGINE_TCGEN05, _p(ws), wsb, st())
    h_out = torch.empty(N, D, device=DEV); gates = torch.empty(4, N, D, device=DEV)
    L.call("ddfa_gru_step_fwd_image", _p(s_img), _p(h_img), _p(hd), _p(dg.indptr), N, D, _p(h_out), _p(o_img), _p(gates), _p(ws), wsb, st())
    assert (h_out.cpu().double() - h_ref.detach()).abs().max() < 1e-4
    for got, ref in zip(gates.cpu().double(), (r_ref, z_ref, n_ref, ghn_ref)):
        assert (got - ref.detach()).abs().max() < 2.5e-4
    # the image of h' the kernel wrote == the image ddfa_act_to_image makes of h' (including the zero tail rows)
    ref_img = torch.zeros(ib, dtype=torch.uint8, device=DEV)
    L.call("ddfa_act_to_image", _p(h_out), N, D, _p(ref_img), st())
    assert torch.equal(o_img, ref_img)
    # inference form (no image, no gates) gives the same h'
    h_out2 = torch.empty(N, D, device=DEV)
    L.call("ddfa_gru_step_fwd_image", _p(s_img), _p(h_img), _p(hd), _p(dg.indptr), N, D, _p(h_out2), None, None, _p(ws), wsb, st())
    assert torch.equal(h_out, h_out2)
    # backward on images, with and without the folded transposed gather
    wsb_b = L.call("ddfa_gru_step_bwd_workspace_bytes", N, D, ENGINE_TCGEN05)
    ws_b = torch.empty(wsb_b, dtype=torch.uint8, device=DEV)
    L.call("ddfa_gru_step_prepare_bwd", _p(wfd), _p(whhd), D, ENGINE_TCGEN05, _p(ws_b), wsb_b, st())
    dpart_d, dsprev_d = dev(dh_part.float()), dev(ds_prev.float())
    results = []
    for fused in (True, False):
        ds, dh = torch.empty(N, D, device=DEV), torch.empty(N, D, device=DEV)
        acc = {n_: torch.zeros(sh, device=DEV) for n_, sh in (("dwf", (3 * D, D)), ("dbf", (3 * D,)), ("dbih", (3 * D,)), ("dwhh", (3 * D, D)), ("dbhh", (3 * D,)))}
        if fused:
            d_in, args = dpart_d, (_p(dsprev_d), _p(dg.indptr_t), _p(dg.indices_t))
        else:       # the caller gathers: d_in = dh_part + A^T ds_prev through ddfa_gather_sum (accumulate)
            d_in = dpart_d.clone()
            L.call("ddfa_gather_sum", _p(dg.indptr_t), _p(dg.indices_t), _p(dsprev_d), N, D, _p(d_in), 1, st())
            args = (None, None, None)
        L.call("ddfa_gru_step_bwd_image", _p(d_in), *args, _p(hd), _p(h_img), _p(s_img), _p(gates), _p(dg.indptr), N, D, _p(ds), _p(dh),
               _p(acc["dwf"]), _p(acc["dbf"]), _p(acc["dbih"]), _p(acc["dwhh"]), _p(acc["dbhh"]), _p(ws_b), wsb_b, 0, st())
        torch.cuda.synchronize()
        checks = [(ds, s_leaf.grad), (dh, leaves[0].grad),            # s_leaf is detached: h.grad is the GRU-only path, like the kernel's dh
                  (acc["dwf"], wf.grad), (acc["dbf"], bf.grad), (acc["dbih"], bih.grad), (acc["dwhh"], whh.grad), (acc["dbhh"], bhh.grad)]
        for got, ref in checks:
            scale = max(1.0, float(ref.abs().max()))
            assert (got.cpu().double() - ref).abs().max() < 3e-4 * scale, f"fused={fused}"
        results.append((ds, dh))
    assert (results[0][0] - results[1][0]).abs().max() < 1e-4 and (results[0][1] - results[1][1]).abs().max() < 1e-4
    with pytest.raises(DdfaError, match="alias"):
        L.call("ddfa_gru_step_bwd_image", _p(dpart_d), _p(ds), _p(dg.indptr_t), _p(dg.indices_t), _p(hd), _p(h_img), _p(s_img), _p(gates),
               _p(dg.indptr), N, D, _p(ds), _p(dh), _p(acc["dwf"]), _p(acc["dbf"]), _p(acc["dbih"]), _p(acc["dwhh"]), _p(acc["dbhh"]),
               _p(ws_b), wsb_b, 0, st())


@pytest.mark.parametrize("graphs,nodes", [(3, 50), (24, 60), (40, 150)])
def test_gru_step_image_entries_v2(graphs, nodes):
    """The round-2 form of the image entries (what engine.py and ddfa_ggnn_fwd/bwd drive): h_t only as its activation image
    (gather from the image, z*h from the image, backward from the image), gates saved as packed fp16."""
    D = 128
    g = synth.make_batch(graphs, nodes, seed=graphs, variable=True)
    dg = prepare_graph(g, DEV)
    N = g.num_nodes()
    src, dst = g.edges()
    torch.manual_seed(100 + graphs)
    k = 1.0 / D ** 0.5
    mk = lambda *sh: (torch.rand(*sh, dtype=torch.float64) * 2 - 1) * k
    wf, bf, bih, whh, bhh = mk(3 * D, D) * 1.5, mk(3 * D), mk(3 * D), mk(3 * D, D), mk(3 * D)
    L = lib()
    ib = L.call("ddfa_act_image_bytes", N)
    h32 = torch.tanh(torch.randn(N, D)).to(DEV)
    h_img = torch.zeros(ib, dtype=torch.uint8, device=DEV)
    L.call("ddfa_act_to_image", _p(h32), N, D, _p(h_img), st())
    h = decode_image(h_img, N)                      # the exact value the image carries (hi + lo): the reference runs on it
    assert (h - h32.cpu().double()).abs().max() < 2e-5
    deg = torch.bincount(dst, minlength=N).double()
    dh_part = torch.randn(N, D, dtype=torch.float64)
    ds_prev = torch.randn(N, D, dtype=torch.float64)
    leaves = [t.requires_grad_(True) for t in (h, wf, bf, bih, whh, bhh)]
    s_ref = torch.zeros(N, D, dtype=torch.float64).index_add(0, dst, leaves[0][src])
    # gather straight from the image
    s_img = torch.zeros(ib, dtype=torch.uint8, device=DEV)
    L.call("ddfa_gather_sum_image_src", _p(dg.indptr), _p(dg.indices), _p(h_img), N, D, _p(s_img), st())
    s_got = decode_image(s_img, N)
    assert (s_got - s_ref.detach()).abs().max() < 2e-5 * max(1.0, float(s_ref.abs().max()))
    # 1, 2 or 4 row groups per warp (CSR chain pipelined across groups): the same sums, bit for bit, incl. the ragged last warps
    from deepdfa_b200._lib import TUNE_GATHER_SRC_GROUPS
    try:
        for groups in (1, 2, 4):
            L.call("ddfa_tuning_set", TUNE_GATHER_SRC_GROUPS, groups)
            s_alt = torch.zeros(ib, dtype=torch.uint8, device=DEV)
            L.call("ddfa_gather_sum_image_src", _p(dg.indptr), _p(dg.indices), _p(h_img), N, D, _p(s_alt), st())
            assert torch.equal(s_alt, s_img), groups
    finally:
        L.call("ddfa_tuning_set", TUNE_GATHER_SRC_GROUPS, 0)
    s_leaf = s_got.clone().requires_grad_(True)     # the forward step below consumes exactly this image
    h_ref, r_ref, z_ref, n_ref, ghn_ref = _gru_reference(s_leaf, leaves[0], deg, *leaves[1:])
    dh_in = dh_part + torch.zeros(N, D, dtype=torch.float64).index_add(0, src, ds_prev[dst])
    (h_ref * dh_in).sum().backward()
    wfd, bfd, bihd, whhd, bhhd = [dev(t.detach().float()) for t in leaves[1:]]
    wsb = L.call("ddfa_gru_step_workspace_bytes", 0, D, ENGINE_TCGEN05)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    L.call("ddfa_gru_step_prepare", _p(wfd), _p(bfd), _p(bihd), _p(whhd), _p(bhhd), D, ENGINE_TCGEN05, _p(ws), wsb, st())
    gpb = L.call("ddfa_gru_gates_packed_bytes", N, D)
    assert gpb == N * D * 8
    gates = torch.empty(gpb, dtype=torch.uint8, device=DEV)
    o_img = torch.zeros(ib, dtype=torch.uint8, device=DEV)
    h_out = torch.empty(N, D, device=DEV)
    # middle step: h only as image in, image only out, packed gates
    L.call("ddfa_gru_step_fwd_image_v2", _p(s_img), _p(h_img), None, _p(dg.indptr), N, D, None, _p(o_img), _p(gates), _p(ws), wsb, st())
    assert (decode_image(o_img, N) - h_ref.detach()).abs().max() < 1e-4
    gk = decode_gates(gates, N)
    for i, (ref, tol) in enumerate(((r_ref, 1.5e-4), (z_ref, 1.5e-4), (n_ref, 1.5e-4), (ghn_ref, None))):
        err = (gk[i] - ref.detach()).abs()
        bound = tol if tol is not None else 1.5e-4 * max(1.0, float(ref.abs().max()))
        assert float(err.max()) < bound, (i, float(err.max()))
    # last step: fp32 out, no image; inference: nothing saved — same h'
    L.call("ddfa_gru_step_fwd_image_v2", _p(s_img), _p(h_img), None, _p(dg.indptr), N, D, _p(h_out), None, None, _p(ws), wsb, st())
    assert (h_out.cpu().double() - h_ref.detach()).abs().max() < 1e-4
    o_img2 = torch.zeros(ib, dtype=torch.uint8, device=DEV)
    L.call("ddfa_act_to_image", _p(h_out), N, D, _p(o_img2), st())
    assert torch.equal(o_img, o_img2)               # the image written directly == the image of the fp32 result
    # first step form: fp32 h operand given (h_0 = x)
    h_out0 = torch.empty(N, D, device=DEV)
    L.call("ddfa_gru_step_fwd_image_v2", _p(s_img), _p(h_img), _p(h32), _p(dg.indptr), N, D, _p(h_out0), None, None, _p(ws), wsb, st())
    assert (h_out0 - h_out).abs().max() < 2e-5
    with pytest.raises(DdfaError):
        L.call("ddfa_gru_step_fwd_image_v2", _p(s_img), _p(h_img), None, _p(dg.indptr), N, D, None, None, None, _p(ws), wsb, st())
    # backward from the image + packed gates, folded transposed gather
    wsb_b = L.call("ddfa_gru_step_bwd_workspace_bytes", N, D, ENGINE_TCGEN05)
    ws_b = torch.empty(wsb_b, dtype=torch.uint8, device=DEV)
    L.call("ddfa_gru_step_prepare_bwd", _p(wfd), _p(whhd), D, ENGINE_TCGEN05, _p(ws_b), wsb_b, st())
    ds, dh = torch.empty(N, D, device=DEV), torch.empty(N, D, device=DEV)
    acc = {n_: torch.zeros(sh, device=DEV) for n_, sh in (("dwf", (3 * D, D)), ("dbf", (3 * D,)), ("dbih", (3 * D,)), ("dwhh", (3 * D, D)), ("dbhh", (3 * D,)))}
    dpart_d, dsprev_d = dev(dh_part.float()), dev(ds_prev.float())        # (named: a temporary would be freed before the launch)
    L.call("ddfa_gru_step_bwd_image_v2", _p(dpart_d), _p(dsprev_d), _p(dg.indptr_t), _p(dg.indices_t), None, _p(h_img),
           _p(s_img), _p(gates), _p(dg.indptr), N, D, _p(ds), _p(dh), _p(acc["dwf"]), _p(acc["dbf"]), _p(acc["dbih"]), _p(acc["dwhh"]), _p(acc["dbhh"]),
           _p(ws_b), wsb_b, 0, st())
    torch.cuda.synchronize()
    checks = [("ds", ds, s_leaf.grad), ("dh", dh, leaves[0].grad), ("dwf", acc["dwf"], wf.grad), ("dbf", acc["dbf"], bf.grad),
              ("dbih", acc["dbih"], bih.grad), ("dwhh", acc["dwhh"], whh.grad), ("dbhh", acc["dbhh"], bhh.grad)]
    worst = {}
    for name, got, ref in checks:
        scale = max(1.0, float(ref.abs().max()))
        worst[name] = float((got.cpu().double() - ref).abs().max()) / scale
    print(f"image v2 backward (packed gates), N={N}: worst |err| / max(1, |ref|max) per output: " + ", ".join(f"{k_}={v:.1e}" for k_, v in worst.items()))
    assert max(worst.values()) < 3e-4, worst
    # the TMA-staged gate backward (default) and the register-path kernel: same q images -> identical ds / dh, same bias sums
    # up to the order of their float atomics; also the step-0 form (fp32 h operand given)
    from deepdfa_b200._lib import TUNE_GATE_BWD_TMA
    outs = {}
    try:
        for mode in (2, 1, 0):       # 2 (default): TMA-staged + pipelined CSR scalars; 1: TMA-staged; 0: register path
            L.call("ddfa_tuning_set", TUNE_GATE_BWD_TMA, mode)
            for h_arg in (None, _p(h32)):
                ds2, dh2 = torch.empty(N, D, device=DEV), torch.empty(N, D, device=DEV)
                acc2 = {n_: torch.zeros(sh, device=DEV) for n_, sh in (("dwf", (3 * D, D)), ("dbf", (3 * D,)), ("dbih", (3 * D,)), ("dwhh", (3 * D, D)), ("dbhh", (3 * D,)))}
                L.call("ddfa_gru_step_bwd_image_v2", _p(dpart_d), _p(dsprev_d), _p(dg.indptr_t), _p(dg.indices_t), h_arg, _p(h_img), _p(s_img), _p(gates),
                       _p(dg.indptr), N, D, _p(ds2), _p(dh2), _p(acc2["dwf"]), _p(acc2["dbf"]), _p(acc2["dbih"]), _p(acc2["dwhh"]), _p(acc2["dbhh"]),
                       _p(ws_b), wsb_b, 0, st())
                torch.cuda.synchronize()
                outs[(mode, h_arg is None)] = (ds2, dh2, acc2)
    finally:
        L.call("ddfa_tuning_set", TUNE_GATE_BWD_TMA, 2)
    for key in ((2, True), (2, False), (1, True), (1, False)):
        a, b = outs[key], outs[(0, key[1])]
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), key
        for n_ in ("dbf", "dbih", "dbhh"):
            assert (a[2][n_] - b[2][n_]).abs().max() < 1e-4 * max(1.0, float(b[2][n_].abs().max())), (key, n_)
    assert torch.equal(outs[(2, True)][0], ds) and torch.equal(outs[(2, True)][1], dh)
    assert (outs[(2, False)][0] - ds).abs().max() < 1e-3 * max(1.0, float(ds.abs().max()))      # fp32 h vs hi + lo: 2^-17 apart


@pytest.mark.parametrize("graphs,nodes", [(3, 50), (40, 150), (1024, 150)])
def test_forward_cta_pair_form_is_bit_identical(graphs, nodes):
    """DDFA_TUNE_FWD_PAIR: the forward GRU kernel launched as 2-CTA clusters issuing tcgen05.mma.cta_group::2 (each CTA stages
    half of every activation tile) multiplies the same operands in the same order — outputs must equal the single-CTA form
    bit for bit (image, fp32 h', packed gates), for ragged tails, few tiles and the C1 size."""
    from deepdfa_b200._lib import TUNE_FWD_PAIR
    D = 128
    g = synth.make_batch(graphs, nodes, seed=graphs, variable=graphs < 1000)
    dg = prepare_graph(g, DEV)
    N = g.num_nodes()
    torch.manual_seed(7)
    k = 1.0 / D ** 0.5
    mk = lambda *sh: ((torch.rand(*sh) * 2 - 1) * k).to(DEV)
    wf, bf, bih, whh, bhh = mk(3 * D, D) * 1.5, mk(3 * D), mk(3 * D), mk(3 * D, D), mk(3 * D)
    L = lib()
    ib = L.call("ddfa_act_image_bytes", N)
    h32 = torch.tanh(torch.randn(N, D)).to(DEV)
    h_img = torch.zeros(ib, dtype=torch.uint8, device=DEV); s_img = torch.zeros(ib, dtype=torch.uint8, device=DEV)
    L.call("ddfa_act_to_image", _p(h32), N, D, _p(h_img), st())
    L.call("ddfa_gather_sum_image_src", _p(dg.indptr), _p(dg.indices), _p(h_img), N, D, _p(s_img), st())
    wsb = L.call("ddfa_gru_step_workspace_bytes", 0, D, ENGINE_TCGEN05)
    ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
    L.call("ddfa_gru_step_prepare", _p(wf), _p(bf), _p(bih), _p(whh), _p(bhh), D, ENGINE_TCGEN05, _p(ws), wsb, st())
    gpb = L.call("ddfa_gru_gates_packed_bytes", N, D)
    outs = {}
    try:
        for pair in (0, 1):
            L.call("ddfa_tuning_set", TUNE_FWD_PAIR, pair)
            assert L.call("ddfa_tuning_get", TUNE_FWD_PAIR) == pair
            o_img = torch.zeros(ib, dtype=torch.uint8, device=DEV); gates = torch.zeros(gpb, dtype=torch.uint8, device=DEV)
            h_out = torch.empty(N, D, device=DEV)
            for _ in range(2):      # twice: barrier phases / stage wrap-around of a second launch
                L.call("ddfa_gru_step_fwd_image_v2", _p(s_img), _p(h_img), None, _p(dg.indptr), N, D, _p(h_out), _p(o_img), _p(gates), _p(ws), wsb, st())
            h_first = torch.empty(N, D, device=DEV)
            L.call("ddfa_gru_step_fwd_image_v2", _p(s_img), _p(h_img), _p(h32), _p(dg.indptr), N, D, _p(h_first), None, None, _p(ws), wsb, st())
            torch.cuda.synchronize()
            outs[pair] = (o_img, gates, h_out, h_first)
    finally:
        L.call("ddfa_tuning_set", TUNE_FWD_PAIR, 0)
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(a, b)
    assert torch.isfinite(outs[1][2]).all() and float(outs[1][2].abs().max()) > 0.1


@pytest.mark.parametrize("D,T", [(128, 3), (128, 8), (128, 18), (32, 4), (128, 1), (128, 0)])
def test_ggnn_fused_drivers(D, T):
    """ddfa_ggnn_fwd / ddfa_ggnn_bwd (the whole GatedGraphConv behind one call each) vs fp64 autograd of the oracle's
    restatement of dgl.nn.GatedGraphConv, both engines; T = 18 takes the per-step weight-gradient path (> 16 slots)."""
    g = synth.make_batch(9, 50, seed=T + D, variable=True)
    dg = prepare_graph(g, DEV)
    N = g.num_nodes()
    torch.manual_seed(D + T)
    conv = O.GatedGraphConvRestated(D, D, T).double()
    with torch.no_grad():
        conv.linears[0].bias.uniform_(-0.2, 0.2)          # DGL initialises it to zero; exercise the bias path
    x = (torch.randn(N, D, dtype=torch.float64) * 0.5).requires_grad_(True)
    h_ref = conv(g, x)
    dh_T = torch.randn(N, D, dtype=torch.float64)
    (h_ref * dh_T).sum().backward()
    par = dict(w_msg=conv.linears[0].weight, b_msg=conv.linears[0].bias, w_ih=conv.gru.weight_ih, w_hh=conv.gru.weight_hh,
               b_ih=conv.gru.bias_ih, b_hh=conv.gru.bias_hh)
    pd = {k: dev(v.detach().float()) for k, v in par.items()}
    xd, dhd = dev(x.detach().float()), dev(dh_T.float())
    L = lib()
    for engine in engines_for(D):
        for training in (1, 0):
            wsb = L.call("ddfa_ggnn_workspace_bytes", N, D, T, engine, training)
            assert wsb > 0
            ws = torch.empty(wsb, dtype=torch.uint8, device=DEV)
            h_out = torch.full((N, D), float("nan"), device=DEV)
            L.call("ddfa_ggnn_fwd", _p(dg.indptr), _p(dg.indices), _p(xd), N, D, T, _p(pd["w_msg"]), _p(pd["b_msg"]), _p(pd["w_ih"]),
                   _p(pd["w_hh"]), _p(pd["b_ih"]), _p(pd["b_hh"]), _p(h_out), _p(ws), wsb, training, engine, st())
            tol = (3e-5 if engine == ENGINE_SIMT else 2e-4) * max(1, T)
            assert (h_out.cpu().double() - h_ref.detach()).abs().max() < tol, (engine, training)
            if not training:
                continue
            dx = torch.full((N, D), float("nan"), device=DEV)
            gr = {k: torch.zeros_like(v) for k, v in pd.items()}
            L.call("ddfa_ggnn_bwd", _p(dg.indptr), _p(dg.indptr_t), _p(dg.indices_t), _p(xd), N, D, T, _p(pd["w_msg"]), _p(pd["b_msg"]),
                   _p(pd["w_ih"]), _p(pd["w_hh"]), _p(dhd), _p(dx), _p(gr["w_msg"]), _p(gr["b_msg"]), _p(gr["w_ih"]), _p(gr["w_hh"]),
                   _p(gr["b_ih"]), _p(gr["b_hh"]), _p(ws), wsb, engine, st())
            checks = [(dx, x.grad)] + [(gr[k], par[k].grad if T > 0 else torch.zeros_like(par[k])) for k in par]
            for got, ref in checks:
                scale = max(1.0, float(ref.abs().max()))
                assert (got.cpu().double() - ref).abs().max() < (1e-4 if engine == ENGINE_SIMT else 5e-4) * scale * max(1, T ** 0.5), engine
    with pytest.raises(DdfaError, match="workspace"):
        L.call("ddfa_ggnn_fwd", _p(dg.indptr), _p(dg.indices), _p(xd), N, D, max(T, 1), _p(pd["w_msg"]), _p(pd["b_msg"]), _p(pd["w_ih"]),
               _p(pd["w_hh"]), _p(pd["b_ih"]), _p(pd["b_hh"]), _p(h_out), _p(ws), 16, 1, ENGINE_SIMT, st())


@pytest.mark.parametrize("L", [1, 2, 3])
def test_readout_mlp_batched_head_for_large_training_batches(L):
    """B >= 256 with a place for the hidden activations (training): the readout kernel only pools, every hidden layer is one GEMM
    over the batch + bias / ReLU, the last layer a warp per graph.  Held to an fp64 reference and to the in-CTA path (same call
    without mlp_act, which keeps the whole MLP inside the pooling kernel)."""
    D, B = 128, 300
    D2 = 2 * D
    rng = np.random.default_rng(L)
    sizes = rng.integers(1, 24, B)
    bnn = torch.from_numpy(sizes)
    N = int(bnn.sum())
    torch.manual_seed(10 + L)
    h, x = torch.randn(N, D), torch.randn(N, D)
    gate = torch.nn.Linear(D2, 1)
    lins = [torch.nn.Linear(D2, 1 if i == L - 1 else D2) for i in range(L)]
    feat = torch.cat([h, x], 1).double()
    gl_ref = feat @ gate.weight.double().t() + gate.bias.double()
    pooled_ref = torch.zeros(B, D2, dtype=torch.float64)
    acts_ref, off = [], 0
    for b, n in enumerate(sizes):
        a = torch.softmax(gl_ref[off:off + n, 0], 0)
        pooled_ref[b] = (a[:, None] * feat[off:off + n]).sum(0)
        off += n
    cur = pooled_ref
    for i, lin in enumerate(lins):
        cur = cur @ lin.weight.double().t() + lin.bias.double()
        if i != L - 1:
            cur = torch.relu(cur)
            acts_ref.append(cur)
    out_ref = cur.squeeze(-1)
    graph_ptr = dev(torch.cat([torch.zeros(1, dtype=torch.int64), bnn.cumsum(0)]).to(torch.int32))
    hd, xd = dev(h), dev(x)
    wg, bg = dev(gate.weight.detach().reshape(-1)), dev(gate.bias.detach())
    mw, mb = [dev(m.weight.detach()) for m in lins], [dev(m.bias.detach()) for m in lins]
    Lb = lib()
    outs = {}
    for mode in ("batched", "in_cta"):
        pooled = torch.empty(B, D2, device=DEV); logits = torch.full((B,), float("nan"), device=DEV)
        gl = torch.empty(N, device=DEV); smax = torch.empty(B, device=DEV); ssum = torch.empty(B, device=DEV)
        act = torch.full((max(L - 1, 1), B, D2), float("nan"), device=DEV)
        Lb.call("ddfa_readout_mlp_fwd", _p(hd), _p(xd), _p(graph_ptr), B, D, _p(wg), _p(bg), ptr_array([_p(t) for t in mw]),
                ptr_array([_p(t) for t in mb]), L, _p(pooled), _p(logits), _p(gl), _p(smax), _p(ssum), _p(act) if mode == "batched" else None, st())
        torch.cuda.synchronize()
        outs[mode] = (pooled, logits, act)
        assert (pooled.cpu().double() - pooled_ref).abs().max() < 1e-5
        assert (logits.cpu().double() - out_ref.detach()).abs().max() < 2e-5 * max(1.0, float(out_ref.abs().max()))
    for i, a_ref in enumerate(acts_ref):
        assert (outs["batched"][2][i].cpu().double() - a_ref.detach()).abs().max() < 2e-5 * max(1.0, float(a_ref.abs().max()))
    assert torch.equal(outs["batched"][0], outs["in_cta"][0])
    assert (outs["batched"][1] - outs["in_cta"][1]).abs().max() < 1e-5


@pytest.mark.parametrize("D,L", [(128, 3), (128, 1), (32, 2), (64, 0), (256, 2)])
def test_readout_mlp_fwd_bwd(D, L):
    sizes = [1, 2, 300, 40, 5, 0, 17]          # includes an EMPTY graph (pooled = 0) and a 1-node graph
    g = synth.make_batch(sizes=[s for s in sizes if s > 0], input_dim=50, seed=D)
    bnn = torch.tensor(sizes)
    N, B, D2 = int(bnn.sum()), len(sizes), 2 * D
    torch.manual_seed(D + L)
    h = torch.randn(N, D, dtype=torch.float64, requires_grad=True); x = torch.randn(N, D, dtype=torch.float64, requires_grad=True)
    gate = torch.nn.Linear(D2, 1).double()
    layers = []
    for i in range(L):
        layers.append(torch.nn.Linear(D2, 1 if i == L - 1 else D2).double())
        if i != L - 1:
            layers.append(torch.nn.ReLU())
    mlp = torch.nn.Sequential(*layers)

    class _G:  # minimal graph for the oracle pooling
        def batch_num_nodes(self):
            return bnn
    pool = O.GlobalAttentionPoolingRestated(gate)
    pooled_ref = pool(_G(), torch.cat([h, x], 1))
    out_ref = mlp(pooled_ref).squeeze(-1) if L else pooled_ref
    dout = torch.randn_like(out_ref)
    (out_ref * dout).sum().backward()

    graph_ptr = dev(torch.cat([torch.zeros(1, dtype=torch.int64), bnn.cumsum(0)]).to(torch.int32))
    hd, xd = dev(h.detach().float()), dev(x.detach().float())
    wg, bg = dev(gate.weight.detach().float().reshape(-1)), dev(gate.bias.detach().float())
    lins = [m for m in mlp if isinstance(m, torch.nn.Linear)]
    mw, mb = [dev(m.weight.detach().float()) for m in lins], [dev(m.bias.detach().float()) for m in lins]
    pooled = torch.empty(B, D2, device=DEV); logits = torch.empty(B, device=DEV)
    gl = torch.empty(N, device=DEV); smax = torch.empty(B, device=DEV); ssum = torch.empty(B, device=DEV)
    act = torch.empty(max(L - 1, 1), B, D2, device=DEV)
    Lb = lib()
    Lb.call("ddfa_readout_mlp_fwd", _p(hd), _p(xd), _p(graph_ptr), B, D, _p(wg), _p(bg), ptr_array([_p(t) for t in mw]) if L else None,
            ptr_array([_p(t) for t in mb]) if L else None, L, _p(pooled), _p(logits) if L else None, _p(gl), _p(smax), _p(ssum), _p(act), st())
    assert (pooled.cpu().double() - pooled_ref.detach()).abs().max() < 1e-5
    assert float(pooled[5].abs().max()) == 0.0
    if L:
        assert (logits.cpu().double() - out_ref.detach()).abs().max() < 2e-5
        dpooled = torch.empty(B, D2, device=DEV); scratch = torch.empty(2, B, D2, device=DEV)
        gw, gb = [torch.zeros_like(t) for t in mw], [torch.zeros_like(t) for t in mb]
        Lb.call("ddfa_mlp_bwd", _p(dk(dout.float())), _p(pooled), _p(act), ptr_array([_p(t) for t in mw]), B, D, L, _p(dpooled),
                ptr_array([_p(t) for t in gw]), ptr_array([_p(t) for t in gb]), _p(scratch), st())
        for got, m in zip(gw, lins):
            assert (got.cpu().double() - m.weight.grad).abs().max() < 1e-4 * max(1.0, float(m.weight.grad.abs().max()))
        for got, m in zip(gb, lins):
            assert (got.cpu().double() - m.bias.grad).abs().max() < 1e-4 * max(1.0, float(m.bias.grad.abs().max()))
    else:
        dpooled = dev(dout.float())
    dh, dx = torch.zeros(N, D, device=DEV), torch.zeros(N, D, device=DEV)
    dwg, dbg = torch.zeros(D2, device=DEV), torch.zeros(1, device=DEV)
    Lb.call("ddfa_readout_bwd", _p(dpooled), _p(pooled), _p(hd), _p(xd), _p(graph_ptr), B, D, _p(wg), _p(gl), _p(smax), _p(ssum), _p(dh), _p(dx),
            _p(dwg), _p(dbg), st())
    assert (dh.cpu().double() - h.grad).abs().max() < 1e-4 * max(1.0, float(h.grad.abs().max()))
    assert (dx.cpu().double() - x.grad).abs().max() < 1e-4 * max(1.0, float(x.grad.abs().max()))
    assert (dwg.cpu().double() - gate.weight.grad.reshape(-1)).abs().max() < 2e-4 * max(1.0, float(gate.weight.grad.abs().max()))
    assert abs(float(dbg) - float(gate.bias.grad)) < 1e-4


@pytest.mark.parametrize("pw", [1.0, 2.5])
def test_graph_label_bce(pw):
    g = synth.make_batch(300, 20, seed=3, variable=True, vuln_rate=0.4)
    dg = prepare_graph(g, DEV)
    B = g.batch_size
    torch.manual_seed(1)
    logits = (torch.randn(B, dtype=torch.float64) * 4).requires_grad_(True)
    m = O.OracleFlowGNNGGNN("_ABS_DATAFLOW", 10, 4, 1, 1, positive_weight=pw)
    labels_ref = m.get_label(g)
    loss_ref = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor([pw], dtype=torch.float64))(logits, labels_ref.double())
    loss_ref.backward()
    labels = torch.empty(B, device=DEV); loss = torch.full((1,), 7.0, device=DEV); dl = torch.empty(B, device=DEV)
    lib().call("ddfa_graph_label_bce", _p(dk(logits.detach().float())), _p(dk(g.ndata["_VULN"])), _p(dg.graph_ptr), B, pw, 1.0 / B, 1.0 / B,
               _p(labels), _p(loss), _p(dl), st())
    assert torch.equal(labels.cpu(), labels_ref) and labels_ref.sum() > 10
    assert abs(float(loss) - float(loss_ref)) < 1e-5
    assert (dl.cpu().double() - logits.grad).abs().max() < 1e-7
    # labels only
    lib().call("ddfa_graph_label_bce", None, _p(dk(g.ndata["_VULN"])), _p(dg.graph_ptr), B, 1.0, 0.0, 0.0, _p(labels), None, None, st())
    assert torch.equal(labels.cpu(), labels_ref)


def test_adam_flat_matches_torch_adam():
    torch.manual_seed(0)
    n = 10007
    p0 = torch.randn(n)
    ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.Adam([ref], lr=1e-3, weight_decay=1e-2)        # config_default.yaml:43-47
    p, m, v = dev(p0), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    step = torch.zeros(1, dtype=torch.int32, device=DEV)
    for i in range(6):
        g = torch.randn(n) * (0.1 if i % 2 else 3.0)
        ref.grad = g.clone(); opt.step()
        lib().call("ddfa_adam_flat", _p(p), _p(dk(g)), _p(m), _p(v), _p(step), n, 1e-3, 0.9, 0.999, 1e-8, 1e-2, st())
    assert int(step) == 6
    assert (p.cpu() - ref.detach()).abs().max() < 2e-6


@pytest.mark.parametrize("world", [1, 2, 4])
def test_allreduce_adam_p2p_protocol_on_one_device(world):
    """ddfa_allreduce_adam_p2p (reduce-scatter + Adam + all-gather over peer memory, two flag barriers): `world` ranks emulated
    on ONE device — every rank has its own parameter / gradient / flag / moment buffers and its kernel runs on its own stream,
    concurrently with the others (they spin on each other's flags, as over NVLink).  Against torch.optim.Adam (coupled L2) on the
    summed gradient, several steps (epochs advance, flags are reused)."""
    torch.manual_seed(world)
    n = 64 * 97                                            # multiple of 64 like the trainer's flat buffers; not a multiple of world * 256
    p0 = torch.randn(n, device=DEV)
    params = [p0.clone() for _ in range(world)]
    grads = [torch.zeros(n + 64, device=DEV) for _ in range(world)]
    flags = [torch.zeros(64, dtype=torch.int32, device=DEV) for _ in range(world)]
    m = [torch.zeros(n, device=DEV) for _ in range(world)]
    v = [torch.zeros(n, device=DEV) for _ in range(world)]
    step = [torch.zeros(1, dtype=torch.int32, device=DEV) for _ in range(world)]
    ticket = [torch.zeros(1, dtype=torch.int32, device=DEV) for _ in range(world)]
    loss_out = [torch.zeros(1, device=DEV) for _ in range(world)]
    streams = [torch.cuda.Stream(device=DEV) for _ in range(world)]
    ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.Adam([ref], lr=1e-3, weight_decay=1e-2)
    L = lib()
    pp, pg, pf = ptr_array([_p(t) for t in params]), ptr_array([_p(t) for t in grads]), ptr_array([_p(t) for t in flags])
    for it in range(4):
        gs = [torch.randn(n, device=DEV) * 0.1 for _ in range(world)]
        for r in range(world):
            grads[r][:n].copy_(gs[r])
            grads[r][n] = float(r + 1 + it)               # the per-rank loss word
        torch.cuda.synchronize()
        for r in range(world):
            L.call("ddfa_allreduce_adam_p2p", pp, pg, pf, r, world, _p(m[r]), _p(v[r]), _p(step[r]), n, n, _p(loss_out[r]), _p(ticket[r]),
                   1e-3, 0.9, 0.999, 1e-8, 1e-2, streams[r].cuda_stream)
        torch.cuda.synchronize()
        ref.grad = torch.stack(gs).sum(0)
        opt.step()
        for r in range(world):
            assert (params[r] - ref.detach()).abs().max() < 2e-6, (it, r)
            assert torch.equal(params[r], params[0])      # every rank holds the same bits
            assert abs(float(loss_out[r]) - sum(q + 1 + it for q in range(world))) < 1e-5
            assert int(step[r]) == it + 1 and int(ticket[r]) == 0
    with pytest.raises(DdfaError):
        L.call("ddfa_allreduce_adam_p2p", pp, pg, pf, world, world, _p(m[0]), _p(v[0]), _p(step[0]), n, n, None, _p(ticket[0]),
               1e-3, 0.9, 0.999, 1e-8, 1e-2, st())
