"""Ring (bulk-copy) layer kernels on a graph large enough for their main structure to matter.

The ring kernels give each warp contiguous runs of work items (2 runs per resident warp); the copies of
a run go ahead across row boundaries (ring slot phase, neighbour window, next-row prefetch, split rows
inside a run, one `da` flush after many rows).  On the small graphs of test_gpu_parity.py a run holds one
or two items, so this file uses 100k rows -- at least 4 items per run on any occupancy -- and compares
every entry of the layer's outputs and gradients with a float64 oracle, in train mode with the kernels'
own dropout mask (helpers.keep_scale) and in eval mode.  F is small: it never reaches the sparse
kernels and keeps the CPU oracle cheap.
"""
import re

import numpy as np
import pytest
import torch

import edgedisentangle_ssl_b200 as edis
from edgedisentangle_ssl_b200 import layers
from edgedisentangle_ssl_b200.layers import run_channels
from edgedisentangle_ssl_b200.synthetic import power_law_graph
from oracle import disgat as od
from helpers import edge_keep, group_floor, rel_err, rounding_noise

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
N, M_RAW, F, D = 100_000, 250_000, 16, 64
P = 0.1                       # the benchmark's dropout
SEED = 0xD1B54A32D192ED03     # high word set
RT, RT_GRAD = 1e-5, 2e-5      # as test_gpu_parity.py


@pytest.fixture(scope="module")
def big():
    idx = power_law_graph(N, M_RAW, seed=3)
    graph = edis.Graph(N, idx[0], idx[1], device=DEV)
    info = graph.info
    # items >= 4 x (SMs x 64 resident warps x 2 runs per warp): every run holds several items
    need = 4 * torch.cuda.get_device_properties(0).multi_processor_count * 64 * 2
    assert info["dst_items"] >= need and info["src_items"] >= need, (info, need)
    assert info["max_in"] > 256 and info["dst_slots"] > 0, info     # split rows inside long runs
    return torch.from_numpy(idx), graph


def oracle(chs, gnn, x, idx, keep, r_out, r_e, dtype, channels=None):
    """The C-channel layer, one channel at a time: the loss is a sum over channels, so each channel is
    run and backpropagated on its own and only one channel's edge tensors are alive at a time.
    -> (out, edge_e, gx, {"c<k>.<param>": grad}); out / edge_e only when all channels run."""
    D_ = chs[0].out_features
    gx = torch.zeros(x.shape, dtype=dtype)
    outs, es, grads = [], [], {}
    for c in range(len(chs)) if channels is None else channels:
        p = {k: v.detach().cpu().to(dtype).requires_grad_(True) for k, v in chs[c].named_parameters()}
        xc = x.detach().clone().to(dtype).requires_grad_(True)
        o, e = od.disga_layer(p, "", xc, idx, 3, gnn, keep=None if keep is None else keep[:, c:c + 1])
        loss = (o * r_out[:, c * D_:(c + 1) * D_].to(dtype)).sum()
        if r_e is not None:
            loss = loss + (e[:, 0] * r_e[:, c].to(dtype)).sum()
        loss.backward()
        gx += xc.grad
        outs.append(o.detach())
        es.append(e.detach())
        grads.update({"c%d.%s" % (c, k): v.grad for k, v in p.items()})
    if channels is not None:
        return None, None, gx, grads
    return torch.cat(outs, 1), torch.cat(es, 1), gx, grads


class score_noise:
    """Arbiter runs: the att-3 score's leaky-relu argument z = [x_i || x_j] W moved by noise of the size fp32
    rounding gives it (5e-7 x sum_k |x_k W_k|).  With ~E x D = 4e7 such arguments some lie within rounding
    of the kink; their side decides a jump of 0.99 de_ij x_i in the score-weight gradient, and which side
    a kernel's (or the oracle's) own rounding picks is arbitrary.  Used together with
    helpers.rounding_noise."""

    def __init__(self, eps, seed):
        self.eps, self.seed = eps, seed

    def __enter__(self):
        self._orig = od.pair_logits
        gen = torch.Generator().manual_seed(self.seed)
        eps, orig = self.eps, self._orig

        def noisy(x, W, a, pairs, att):
            if att != 3:
                return orig(x, W, a, pairs, att)
            xi = torch.cat((x[pairs[0]], x[pairs[1]]), dim=1)
            z = xi @ W
            with torch.no_grad():
                scale = xi.abs() @ W.abs()
                z_n = eps * scale * (2 * torch.rand(z.shape, generator=gen, dtype=z.dtype) - 1)
            return torch.nn.functional.leaky_relu(z + z_n) @ a

        od.pair_logits = noisy
        return self

    def __exit__(self, *exc):
        od.pair_logits = self._orig
        return False


def cuda_kernels(prof):
    names = {ev.key for ev in prof.key_averages() if ev.device_type == torch.autograd.DeviceType.CUDA}
    assert names, "torch.profiler recorded no CUDA kernels"
    return names


CASES = [
    # (C, gnn, train, edge_e in the loss)
    (8, "AT", True, False),       # the benchmark's combination: dst pass without the logit gradient
    (8, "AT", False, True),
    (4, "AT", True, True),
    (2, "AT", True, False),
    (8, "GCN", True, True),       # bias
]


@pytest.mark.parametrize("C,gnn,train,gx_term", CASES, ids=lambda v: str(v))
def test_ring_kernels_on_long_runs_vs_float64(big, C, gnn, train, gx_term, monkeypatch):
    idx, graph = big
    e_cnt = idx.shape[1]
    monkeypatch.setenv("EDIS_AT_PLAN", "proj")        # the ring kernels belong to project-then-aggregate
    monkeypatch.setattr(layers, "_next_seed", lambda: SEED)
    torch.manual_seed(C)
    chs = [edis.DisGALayer(F, D, dropout=P, alpha=0.1, att_type=3, gnn_type=gnn) for _ in range(C)]
    x_cpu = torch.randn(N, F)
    r_out = torch.randn(N, C * D)
    r_e = torch.randn(e_cnt, C) if gx_term else None
    keep = torch.from_numpy(edge_keep(SEED, e_cnt, C, P)) if train else None

    for l in chs:
        l.to(DEV).train(train)
    x = x_cpu.to(DEV).requires_grad_(True)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out, e, _ = run_channels(chs, x, graph)
        loss = (out * r_out.to(DEV)).sum()
        if gx_term:
            loss = loss + (e * r_e.to(DEV)).sum()
        loss.backward()
        torch.cuda.synchronize()
    names = cuda_kernels(prof)
    flags = "%s, %s" % (str(train).lower(), str(gx_term).lower())
    for want in (r"k_disga_fwd_ring<", r"k_disga_bwd_dst_ring<.*, %s>" % flags, r"k_disga_bwd_src_ring<",
                 r"k_combine_"):
        assert any(re.search(want, nm) for nm in names), (want, sorted(names))
    got = {"gx": x.grad.cpu()}
    for c, l in enumerate(chs):
        got.update({"c%d.%s" % (c, k): v.grad.cpu() for k, v in l.named_parameters()})

    o64, e64, gx64, g64 = oracle(chs, gnn, x_cpu, idx, keep, r_out, r_e, torch.float64)
    assert rel_err(out.detach().cpu(), o64) <= RT, "out"
    assert rel_err(e.detach().cpu(), e64) <= RT, "edge_e"
    del o64, e64
    _, _, gx32, g32 = oracle(chs, gnn, x_cpu, idx, keep, r_out, r_e, torch.float32)
    g64["gx"], g32["gx"] = gx64, gx32
    floor = group_floor([v for k, v in g64.items() if k != "gx"])
    assert set(got) == set(g64)
    bad = []
    for k in sorted(got):
        fl = 0.0 if k == "gx" else floor
        err = rel_err(got[k], g64[k], fl)
        tol = max(RT_GRAD, 16.0 * rel_err(g32[k], g64[k], fl))
        if err > tol:
            # leaky-relu arguments within rounding of 0: the arbiter's own spread under rounding-sized noise
            chans = None if k == "gx" else [int(k[1:k.index(".")])]

            sens = 0.0
            for sd in (1, 2, 3):
                with rounding_noise(5e-7, sd), score_noise(5e-7, sd):
                    _, _, g, gr = oracle(chs, gnn, x_cpu, idx, keep, r_out, r_e, torch.float64, chans)
                gr["gx"] = g
                sens = max(sens, rel_err(gr[k], g64[k], fl))
            tol = max(tol, 2.0 * sens)
        if err > tol:
            bad.append("%s: rel err %.3e > %.1e" % (k, err, tol))
    assert not bad, bad
