"""Shared helpers for the parity tests."""
import os

import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# north_star tolerance for fp32 results: 1e-5 relative.  Measured against the tensor's
# scale (max |ref|) for near-zero entries, as usual for reassociated fp32 sums.
RTOL = 1e-5


def load(name):
    return dict(np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False))


def t(a, dtype=None):
    x = torch.from_numpy(np.asarray(a))
    return x.to(dtype) if dtype is not None else x


def _np(a):
    if isinstance(a, torch.Tensor):
        a = a.detach().cpu().numpy()
    return np.asarray(a, dtype=np.float64)


def rel_err(got, ref, floor=0.0):
    got, ref = _np(got), _np(ref)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    if ref.size == 0:
        return 0.0
    scale = max(np.abs(ref).max(), floor, 1e-30)
    return float(np.abs(got - ref).max() / scale)


def assert_close(got, ref, rtol=RTOL, what="", floor=0.0):
    """max |got - ref| <= rtol * max(max |ref|, floor).

    `floor` is used for gradient groups: a tensor whose gradient is orders of magnitude below
    the group's largest one (cancelling sums; the reference's own fp32 result is noise there)
    is measured against GRAD_FLOOR x the group's scale instead of its own."""
    err = rel_err(got, ref, floor)
    assert err <= rtol, "%s: rel err %.3e > %.1e" % (what, err, rtol)


def keep_scale(seed, idx, p):
    """Bit-exact numpy restatement of the kernels' dropout multiplier (csrc/edis_common.cuh keep_scale):
    float32 inv_keep = 1 / (1 - p) where element `idx` is kept, 0 where it is dropped.  The layer kernels
    draw element csr_slot * C + channel of the attention weights with the layer's 64-bit seed."""
    idx = np.asarray(idx, dtype=np.uint64)
    seed = np.uint64(int(seed) & (2 ** 64 - 1))
    lo32 = np.uint64(0xFFFFFFFF)
    u32 = lambda v: (v & lo32).astype(np.uint32)   # noqa: E731
    with np.errstate(over="ignore"):
        x = u32(idx) ^ u32(seed)
        x = x * np.uint32(0x9E3779B1)
        x ^= u32(idx >> np.uint64(32)) * np.uint32(0x85EBCA77) + u32(seed >> np.uint64(32))
        x ^= x >> np.uint32(16)
        x = x * np.uint32(0x85EBCA6B)
        x ^= x >> np.uint32(13)
        x = x * np.uint32(0xC2B2AE35)
        x ^= x >> np.uint32(16)
    u = (x >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)
    inv_keep = np.float32(1) / (np.float32(1) - np.float32(p))
    return np.where(u >= np.float32(p), inv_keep, np.float32(0)).astype(np.float32)


def edge_keep(seed, e, C, p):
    """[e, C] dropout multipliers of a layer's attention weights (CSR slot x channel)."""
    return keep_scale(seed, np.arange(e * C, dtype=np.uint64), p).reshape(e, C)


GRAD_FLOOR = 1e-3


def group_floor(refs):
    """GRAD_FLOOR x the largest |value| over a group of reference tensors."""
    m = 0.0
    for r in refs:
        r = _np(r)
        if r.size:
            m = max(m, float(np.abs(r).max()))
    return GRAD_FLOOR * m


def params_from(g, prefix):
    """Collect `prefix + name` entries of a golden dict as float32 torch tensors."""
    return {k[len(prefix):]: t(v) for k, v in g.items() if k.startswith(prefix)}


class rounding_noise:
    """Context manager for float64 ARBITER runs of the oracle: the softmax weights exp(.) are multiplied by
    (1 + eps * u), u ~ U(-1, 1) -- a perturbation of the size fp32 rounding / MUFU approximations make
    (eps = 5e-7) -- and autograd differentiates the perturbed function exactly.

    Why: the gradient of this path is DISCONTINUOUS where a leaky-relu argument crosses zero (the att-3
    score a . lrelu(P_i + Q_j), the fuser, the MLP heads).  An argument closer to zero than fp32 rounding
    lands on either side of the kink depending on the evaluation order (the reference's own fp32 run
    included), both one-sided derivatives are valid subgradients, and one such element moves a weight
    gradient by ~5e-5 of its scale on chameleon (measured: tests/test_gpu_bundled.py).  A fixed tolerance
    cannot tell this from an inaccurate kernel; the arbiter's own response to rounding-sized noise can: away
    from kinks it is ~1e-6, next to one it shows the jump."""

    def __init__(self, eps, seed):
        self.eps, self.seed = eps, seed

    def __enter__(self):
        from oracle import disgat as od
        self._od, self._orig = od, od.sp_softmax
        gen = torch.Generator().manual_seed(self.seed)
        eps = self.eps

        def noisy(indices, values, n):
            row = indices[0]
            sh = torch.exp(values - values.max())
            sh = sh * (1 + eps * (2 * torch.rand(sh.shape, generator=gen, dtype=sh.dtype) - 1))
            den = torch.zeros(n, 1, dtype=values.dtype)
            den.scatter_add_(0, row.unsqueeze(1), sh)
            return sh / (den[row] + 1e-10)

        od.sp_softmax = noisy
        return self

    def __exit__(self, *exc):
        self._od.sp_softmax = self._orig
        return False


def kink_sensitivity(run_f64, base, floor, seeds=(1, 2, 3), eps=5e-7):
    """{name: max over noisy float64 runs of rel_err(noisy gradient, base gradient)}.  run_f64() -> {name: grad}."""
    out = {k: 0.0 for k in base}
    for s in seeds:
        with rounding_noise(eps, s):
            g = run_f64()
        for k in base:
            out[k] = max(out[k], rel_err(g[k], base[k], floor))
    return out
