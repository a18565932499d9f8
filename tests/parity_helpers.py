"""Shared pieces of the GPU parity tests (plain helpers, no fixtures): the module-gradient bound, decoders of the tcgen05
engine's saved state, and the fp64 GRU step the kernel tests compare against.  Every function runs on the device of its
inputs, or on `device` where one is given."""
import torch

# per-parameter gradient bound, relative to the largest entry of that parameter's reference gradient.  The fp32 oracle itself is
# ~1e-6 from fp64 on these; the tcgen05 engine multiplies with bf16x3 split operands (2^-16 per product) and uses ex2.approx
# gate math, which is what the measured worst case (printed, and recorded in DESIGN.md §4) reflects.
GRAD_TOL = {"simt": 1e-5, "tcgen05": 1e-4}       # measured worst case (r03a): simt 1.1e-6, tcgen05 1.6e-5 (ggnn.gru.weight_hh)


def decode_image(img: torch.Tensor, N: int, device="cpu") -> torch.Tensor:
    """Activation image (include/ddfa_b200.h) -> fp64 [N,128] = hi + lo, undoing the SWIZZLE_128B unit permutation."""
    tiles = img.numel() // 65536
    raw = img.to(device).view(torch.int16).view(tiles, 4, 128, 8, 8)            # [tile][chunk = 2 v + kb][row][physical 16-B unit][8 bf16]
    rows = torch.arange(128, device=raw.device).view(1, 1, 128, 1, 1)
    units = torch.arange(8, device=raw.device).view(1, 1, 1, 8, 1)
    phys = (units ^ (rows & 7)).expand(tiles, 4, 128, 8, 8)
    logical = torch.gather(raw, 3, phys)                                          # logical unit j sits at physical unit j ^ (row & 7)
    vals = (logical.to(torch.int32) << 16).view(torch.float32).double().view(tiles, 2, 2, 128, 64)   # [tile][v][kb][row][col in block]
    x = (vals[:, 0] + vals[:, 1]).permute(0, 2, 1, 3).reshape(tiles * 128, 128)   # hi + lo, [row][kb][64] -> 128 columns
    assert float(x[N:].abs().max()) == 0.0 if x.shape[0] > N else True           # rows past N are zero
    return x[:N]


def decode_gates(gates: torch.Tensor, N: int, device="cpu"):
    """Packed saved gates (csrc/tc_common.cuh: pack_gates) -> (r, z, n, gh_n) fp64 [N,128]."""
    w = gates.to(device).view(torch.int32).view(N, 128, 2).to(torch.int64) & 0xffffffff
    x, y = w[..., 0], w[..., 1]
    r = (x & 0x3fff).double() / 16383.0
    z = ((x >> 14) & 0x3fff).double() / 16383.0
    nq = y & 0xffff
    n = torch.where(nq >= 32768, nq - 65536, nq).double() / 32767.0
    g = ((y >> 16) << 4) | (x >> 28)
    e, m, sign = (g >> 14) & 31, (g & 0x3fff).double(), (g >> 19) & 1
    ghn = torch.where(e == 0, torch.zeros_like(m), torch.pow(2.0, (e - 15).double()) * (1.0 + m / 16384.0))
    return r, z, n, torch.where(sign == 1, -ghn, ghn)


def gru_reference(s, h, deg, wf, bf, bih, whh, bhh):
    """One GRU step in the folded form the kernels compute (include/ddfa_b200.h, K4): returns h', r, z, n, gh_n."""
    D = h.shape[1]
    gi = s @ wf.t() + deg[:, None] * bf[None, :] + bih
    gh = h @ whh.t() + bhh
    r = torch.sigmoid(gi[:, :D] + gh[:, :D]); z = torch.sigmoid(gi[:, D:2 * D] + gh[:, D:2 * D])
    n = torch.tanh(gi[:, 2 * D:] + r * gh[:, 2 * D:])
    return (1 - z) * n + z * h, r, z, n, gh[:, 2 * D:]
