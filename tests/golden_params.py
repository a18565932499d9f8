"""Compact storage for the reference-code goldens (tests/golden/make_reference_*_golden.py and the tests that read them).

Random parameters are not stored.  Before a generator runs the reference code it overwrites the module's parameters with
`hashed_uniform` values (integer hashing, no random-number library, so every machine rebuilds the same float32 values bit for
bit) and records each parameter's name, shape and bound; `load` puts them back into the fixture's ``state_dict``.  Gradients
larger than `SAMPLE` entries are stored as a fixed sample of entries plus the full tensor's max |g|, mean and mean |g|
(`sample`, `sample_error`), and the fixture is an xz-compressed `torch.save` file (`save`, `load`), so that each stays
well under 1 MB."""
import io
import lzma
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SAMPLE = 512


def hashed_uniform(shape, seed, bound):
    """float32 values in [-bound, bound) from splitmix64 of (seed, element index); 24 random bits each."""
    n = int(np.prod(shape, dtype=np.int64))
    with np.errstate(over="ignore"):
        z = np.arange(1, n + 1, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(seed) * np.uint64(0xD1B54A32D192ED03)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    u = ((z >> np.uint64(40)).astype(np.float64) * 2.0 ** -23 - 1.0).astype(np.float32)      # exact: 24 bits in [-1, 1)
    return torch.from_numpy((u * np.float32(bound)).reshape(tuple(shape)))


def hash_params(module, seed, skip=()):
    """Overwrites every parameter whose name does not start with one of `skip` with `hashed_uniform` values of the same
    root-mean-square as its current (initialised) values; returns the spec `load` rebuilds them from."""
    spec = []
    with torch.no_grad():
        for j, (name, p) in enumerate(module.named_parameters()):
            if name.startswith(tuple(skip)):
                continue
            bound = float(p.double().pow(2).mean().mul(3.0).sqrt())         # uniform on [-b, b) has rms b / sqrt(3)
            p.copy_(hashed_uniform(p.shape, seed * 1000 + j, bound))
            spec.append((name, tuple(p.shape), seed * 1000 + j, bound))
    return spec


def stored_state(module, spec):
    """The state_dict entries `spec` does not rebuild (buffers, parameters left out of the hashing)."""
    hashed = {s[0] for s in spec}
    return {k: v.clone() for k, v in module.state_dict().items() if k not in hashed}


def sample(t, seed):
    """A fixed sample of `t`'s entries (all of them up to SAMPLE) and three statistics of the whole tensor."""
    flat = t.detach().flatten()
    n = flat.numel()
    idx = np.arange(n) if n <= SAMPLE else np.sort(np.random.default_rng(seed).choice(n, SAMPLE, replace=False))
    idx = torch.from_numpy(idx.astype(np.int32))
    f64 = flat.double()
    return {"idx": idx, "val": flat[idx.long()].clone(), "absmax": float(f64.abs().max()), "mean": float(f64.mean()),
            "absmean": float(f64.abs().mean())}


def sample_error(got, s):
    """Largest of |got - ref| over the sampled entries and the differences of max |.|, mean and mean |.| over the whole
    tensor.  Each of these is at most the largest elementwise difference, so a bound on that bounds this too."""
    g = got.detach().cpu().double().flatten()
    return max(float((g[s["idx"].long()] - s["val"].double()).abs().max()), abs(float(g.abs().max()) - s["absmax"]),
               abs(float(g.mean()) - s["mean"]), abs(float(g.abs().mean()) - s["absmean"]))


def save(obj, name):
    buf = io.BytesIO()
    torch.save(obj, buf)
    path = os.path.join(GOLDEN_DIR, name)
    with open(path, "wb") as f:
        f.write(lzma.compress(buf.getvalue(), preset=9))
    return path


def load(name):
    """Reads tests/golden/<name> and rebuilds the full ``state_dict`` of the fixture (or of each of its ``cases``)."""
    with open(os.path.join(GOLDEN_DIR, name), "rb") as f:
        data = torch.load(io.BytesIO(lzma.decompress(f.read())), weights_only=False)
    for rec in data["cases"] if "cases" in data else [data]:
        sd = dict(rec["state_dict"])
        for pname, shape, seed, bound in rec.pop("params"):
            sd[pname] = hashed_uniform(shape, seed, bound)
        rec["state_dict"] = sd
    return data
