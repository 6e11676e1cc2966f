"""TEST INFRASTRUCTURE - compact golden records of reference outputs (tests/golden/ref_*.npz).

A reference output is stored as
  * a digest (sha256 of dtype, shape and bytes) where the test demands bit equality, or
  * where it allows a tolerance: a seeded sample of rows, checked element by element against atol + rtol * |ref|, plus seeded +-1
    projections of the whole tensor (float64).  The projections are a weaker check of the rows outside the sample: a result within the
    element-wise tolerance everywhere moves a projection by at most n * atol + rtol * sum|ref|, so only a deviation that adds up to
    more than that over the whole tensor (a systematic error, or a few grossly wrong elements) is caught there.  One wrong element
    outside the sample can pass; the sample (up to N_ROWS rows and MAX_SAMPLE elements, at least MIN_ROWS rows) bounds the file sizes.
Weights are not stored: `seeded_state` regenerates them from (name, shape) and a seed, on both sides.
"""
import hashlib
import json

import numpy as np
import torch

N_ROWS = 256
MAX_SAMPLE = 1024
MIN_ROWS = 32
N_PROJ = 4
_CHUNK = 1 << 20


def digest(t):
    a = np.ascontiguousarray(t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t))
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def _project(flat, seed):
    """N_PROJ seeded +-1 projections of a float64 vector, with the signs drawn chunk by chunk (int8) to bound host memory."""
    g = torch.Generator().manual_seed(seed)
    proj = torch.zeros(N_PROJ, dtype=torch.float64)
    for c in range(0, flat.numel(), _CHUNK):
        x = flat[c:c + _CHUNK]
        s = torch.randint(0, 2, (N_PROJ, x.numel()), generator=g, dtype=torch.int8)
        proj += 2 * (s.double() @ x) - x.sum()
    return proj


def _rows(n, k, seed):
    g = torch.Generator().manual_seed(seed + 1)
    return torch.randperm(n, generator=g)[:k].sort().values if n > k else torch.arange(n)


def record(out, name, t, exact=False, seed=0, rows=N_ROWS):
    """Adds the record of tensor `t` under `name` to the dict `out` (see save); `rows` rows are sampled."""
    t = t.detach().cpu()
    meta = out.setdefault("meta", {})
    m = meta[name] = {"shape": list(t.shape)}
    if exact:
        m["sha256"] = digest(t)
        return
    n = t.shape[0] if t.dim() else 1
    width = t.numel() // max(n, 1)
    idx = _rows(n, min(rows, max(MIN_ROWS, MAX_SAMPLE // max(width, 1))), seed)   # fewer rows when wide, never fewer than MIN_ROWS
    flat = t.reshape(-1).double()
    m.update(n_rows=len(idx), proj=_project(flat, seed).tolist(), abs_sum=float(flat.abs().sum()),
             abs_max=float(flat.abs().max()) if flat.numel() else 0.0)
    out[name] = t.reshape(n, -1)[idx].numpy()


def save(path, out):
    """np.savez_compressed of the arrays in `out`; the record metadata and any other non-array values go into one JSON string."""
    arrays = {k: v for k, v in out.items() if isinstance(v, np.ndarray)}
    arrays["meta"] = np.array(json.dumps({k: v for k, v in out.items() if not isinstance(v, np.ndarray)}))
    np.savez_compressed(path, **arrays)


def load(path):
    """The arrays of a saved record file plus its JSON values, in one dict."""
    z = np.load(path)
    d = {k: z[k] for k in z.files if k != "meta"}
    d.update(json.loads(str(z["meta"])))
    return d


def check(z, name, got, rtol=0.0, atol=0.0, seed=0):
    """Asserts that `got` matches the record `name` of a loaded record file `z` (exactly, or within rtol / atol element-wise)."""
    got = got.detach().cpu()
    m = z["meta"][name]
    assert list(got.shape) == m["shape"], f"{name}: shape {list(got.shape)} != {m['shape']}"
    if "sha256" in m:
        assert digest(got) == m["sha256"], f"{name}: differs from the reference (bit-exact record)"
        return
    n = got.shape[0] if got.dim() else 1
    rows = _rows(n, m["n_rows"], seed)
    ref = torch.from_numpy(z[name])
    torch.testing.assert_close(got.reshape(n, -1)[rows], ref, rtol=rtol, atol=atol, msg=lambda s: f"{name} (sampled rows): {s}")
    flat = got.reshape(-1).double()
    proj = _project(flat, seed)
    bound = flat.numel() * atol + (rtol + 1e-9) * m["abs_sum"]
    err = (proj - torch.tensor(m["proj"], dtype=torch.float64)).abs().max().item()
    assert err <= bound, f"{name}: projection error {err:.3e} > {bound:.3e} (a row outside the sample differs)"


def state_spec(module):
    """[(name, shape)] of the floating-point state of a module, in state-dict order."""
    return [(k, list(v.shape)) for k, v in module.state_dict().items() if v.dtype.is_floating_point]


def seeded_state(spec, seed):
    """Seeded weights for a state spec: matrices ~ N(0, 2/fan_in), norm scales around 1, biases / shifts ~ 0.2 N(0, 1),
    running variances in [0.5, 1.5).  `spec` is a state_spec list."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for name, shape in spec:
        if "running_var" in name:
            v = torch.rand(shape, generator=g) + 0.5
        elif "running_mean" in name:
            v = torch.randn(shape, generator=g) * 0.3
        elif name.endswith("tau"):
            v = torch.rand(shape, generator=g) * 0.5 + 0.05
        elif len(shape) >= 2:
            fan_in = int(np.prod(shape[1:])) if len(shape) == 2 else int(np.prod(shape[:-1]))
            v = torch.randn(shape, generator=g) * (2.0 / fan_in) ** 0.5
        else:
            v = torch.randn(shape, generator=g) * 0.2 + (1.0 if name.endswith("weight") else 0.0)
        out[name] = v
    return out


def load_seeded(module, spec, seed):
    """Copies seeded_state(spec, seed) into a module (the reference's, when the golden record is made)."""
    w = seeded_state(spec, seed)
    with torch.no_grad():
        for k, v in module.state_dict().items():
            if k in w:
                v.copy_(w[k])
    return w
