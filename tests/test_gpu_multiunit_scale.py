"""Non-ring layer kernels and the SSL pair kernels where every warp walks many work units.

The persistent kernels cap their grid at ceil(units / 8) blocks of 8 warps, so on the small graphs of
test_gpu_parity.py each warp gets at most one unit and the state a warp carries from one unit to the
next is never exercised: the running `da` and its flush when the channel group changes, and the runs of
equal key in the pair backward.  A unit is item * G + group and a warp steps by 8 x (blocks per SM) x SMs
units; on a 148-SM B200 that is 2^5 * 37 * (blocks per SM), so at G = 2, 4, 8 a warp keeps one group for
life and only a G with another prime factor makes it switch groups mid-loop.  G = 3 and G = 5 cannot both
divide the warp count (blocks per SM <= 8), so the cases below, which have both, reach the switch.

Every case runs on a 100k-row power-law graph (and its ~2M-pair SSL sample) with at least 4 units per warp
at full occupancy, and asserts that precondition, the kernel variant it meant to reach, and -- for the layers
-- that no ring kernel ran.  Results are compared over all entries with a float64 restatement: the layers'
on the host, one channel at a time; the pair scoring's in float64 torch on the device (2M pairs x 768
elements are minutes on the host), chunked, with index_add_ for the gathered sides.

Exact score operands.  In att 3 the gradient jumps where an element of z = P_i + Q_j crosses 0.  Inputs are
built so that z is exact on every path: x entries are k/8 (k odd in [1, 15], positive) and each column of
W_top / W_bot has one sign with entries k/2^s (k odd in [1, 31]).  Every P and Q entry is then a nonzero sum
of same-signed dyadic terms, exact in fp32 and in the 3xTF32 projection (x and W lie on the TF32 grid, so
the low parts are 0), and z = P_i + Q_j is exact and takes both signs.  An exact cancellation gives z = +0,
which the kernels (w = -P - Q = +0, sign bit clear) and torch both treat as z <= 0.  So the sign of every
element has one right answer and no noise arbiter is needed.  s = 5 + ceil(log2 F) keeps |P| ~ 0.5, so the
logits stay O(1) and sigmoid(edge_e) does not saturate (with s = 6 at F = 16, |z| reaches ~8 and the score
gradient through the softmax all but vanishes).
"""
import math

import pytest
import torch

import edgedisentangle_ssl_b200 as edis
from edgedisentangle_ssl_b200 import functional as Fn
from edgedisentangle_ssl_b200 import layers
from edgedisentangle_ssl_b200.layers import run_channels
from edgedisentangle_ssl_b200.sampler import sample_pairs_device
from edgedisentangle_ssl_b200.synthetic import power_law_graph
from oracle import disgat as od
from helpers import edge_keep, group_floor, rel_err

DEV = "cuda:0"
N, M_RAW = 100_000, 250_000
P_DROP = 0.1                  # the benchmark's dropout
SEED = 0xD1B54A32D192ED03     # high word set
RT, RT_GRAD = 1e-5, 2e-5      # as test_gpu_parity.py
CHUNK = 1 << 18               # pairs per step of the pair restatement (bounds its memory)


# ------------------------------------------------------------------ exact operands
def exact_x(n, f, gen):
    """[n, f] entries k/8, k odd in [1, 15]: positive, 4 significant bits."""
    return (2 * torch.randint(0, 8, (n, f), generator=gen) + 1).float() / 8


def exact_w(f, d, gen, coherent=True):
    """[f, d] entries +-k/2^s, k odd in [1, 31], s = 5 + ceil(log2 f).  coherent: one random sign per column
    (x @ w is then nonzero in every entry for positive x); otherwise one per entry."""
    k = (2 * torch.randint(0, 16, (f, d), generator=gen) + 1).float()
    sign = 2 * torch.randint(0, 2, (1, d) if coherent else (f, d), generator=gen) - 1
    return sign * k / 2.0 ** (5 + math.ceil(math.log2(f)))


def units_needed():
    """4 units per warp with every SM at 64 resident warps."""
    return 4 * torch.cuda.get_device_properties(0).multi_processor_count * 64


def cuda_kernels(prof):
    """{kernel name: launches} of a torch.profiler trace."""
    names = {}
    for ev in prof.key_averages():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            # demanglers differ in printing int template arguments and the space in "> >"
            key = ev.key.replace("(int)", "").replace(" ", "")
            names[key] = names.get(key, 0) + ev.count
    assert names, "torch.profiler recorded no CUDA kernels"
    return names


def assert_ran(names, want, count=None):
    want = want.replace(" ", "")
    hit = [k for k in names if want in k]
    assert hit, (want, sorted(k for k in names if "edis::" in k))
    if count is not None:
        assert sum(names[k] for k in hit) == count, (want, {k: names[k] for k in hit}, count)


def grad_tol(got, g64, g32, floor):
    """The suite's gradient bound: max(2e-5, 16 x the fp32 restatement's own error against float64)."""
    return rel_err(got, g64, floor), max(RT_GRAD, 16.0 * rel_err(g32, g64, floor))


@pytest.fixture(scope="module")
def big():
    idx = power_law_graph(N, M_RAW, seed=3)
    graph = edis.Graph(N, idx[0], idx[1], device=DEV)
    assert graph.info["dst_slots"] > 0, graph.info        # split hub rows among the units
    return torch.from_numpy(idx), graph


@pytest.fixture(scope="module")
def sample(big):
    """The device sampler's pair list on the graph's keys: ~2M unique pairs, sorted by row."""
    idx, _ = big
    key = (idx[0] * N + idx[1]).to(DEV)
    gen = torch.Generator(device=DEV).manual_seed(7)
    pairs, label = sample_pairs_device(N, key, gen)
    assert bool((pairs[0, 1:] >= pairs[0, :-1]).all())
    return pairs, label


# ------------------------------------------------------------------ layers
def oracle(chs, att, gnn, x, idx, keep, r_out, r_e, dtype):
    """The C-channel layer one channel at a time (the loss is a sum over channels).
    -> (out, edge_e, gx, {"c<k>.<param>": grad})."""
    D_ = chs[0].out_features
    gx = torch.zeros(x.shape, dtype=dtype)
    outs, es, grads = [], [], {}
    for c in range(len(chs)):
        p = {k: v.detach().cpu().to(dtype).requires_grad_(True) for k, v in chs[c].named_parameters()}
        xc = x.detach().clone().to(dtype).requires_grad_(True)
        o, e = od.disga_layer(p, "", xc, idx, att, gnn, keep=None if keep is None else keep[:, c:c + 1])
        loss = (o * r_out[:, c * D_:(c + 1) * D_].to(dtype)).sum()
        if r_e is not None:
            loss = loss + (e[:, 0] * r_e[:, c].to(dtype)).sum()
        loss.backward()
        gx += xc.grad
        outs.append(o.detach())
        es.append(e.detach())
        grads.update({"c%d.%s" % (c, k): v.grad for k, v in p.items()})
    return torch.cat(outs, 1), torch.cat(es, 1), gx, grads


V4, V2, V1 = "edis::VecT<4, 16>", "edis::VecT<2, 16>", "edis::VecT<1, 16>"


def _std(T, att, usrc=1):
    """The project-then-aggregate kernels: fwd / dst pass with RX = 0, source pass with the V gradient."""
    return ("k_disga_fwd<%s, %d, 0," % (T, att), "k_disga_bwd_dst<%s, %d, 0," % (T, att),
            "k_disga_bwd_src<%s, %d, %d," % (T, att, usrc))


LAYER_CASES = [
    # (id, att, gnn, C, D, F, train, edge_e in the loss, EDIS_AT_PLAN, G, kernels)
    ("a3_AT_C16_G2", 3, "AT", 16, 64, 16, True, True, "proj", 2, _std(V4, 3)),
    ("a3_AT_C12_G3", 3, "AT", 12, 64, 16, True, False, "proj", 3, _std(V2, 3)),
    ("a3_GCN_C10_G5_eval", 3, "GCN", 10, 64, 16, False, True, "proj", 5, _std(V1, 3)),
    ("a2_AT_C8_G1", 2, "AT", 8, 64, 16, True, True, "proj", 1, _std(V4, 2)),
    ("a1_GCN_C6_G3", 1, "GCN", 6, 64, 16, True, True, "proj", 3, _std(V1, 1)),
    ("a3_AT_C5_D20_G5", 3, "AT", 5, 20, 16, True, True, "proj", 5, _std("edis::ScaT<1>", 3)),
    ("a3_SAGE_C12_F15_G3", 3, "SAGE", 12, 64, 15, True, True, "proj", 3,
     ("k_disga_fwd<%s, 3, 2," % V2, "k_disga_bwd_dst<%s, 3, 2," % V2, "k_disga_bwd_src<%s, 3, 0," % V2,
      "k_sage_bwd_src_x<2>")),
    ("a3_SAGE_C8_F64_shared", 3, "SAGE", 8, 64, 64, True, False, "proj", 1,
     ("k_disga_fwd<%s, 3, -1," % V4, "k_disga_bwd_dst<%s, 3, -1," % V4, "k_disga_bwd_src<%s, 3, 2," % V4)),
    ("a3_AT_C8_F64_aggplan", 3, "AT", 8, 64, 64, True, True, "agg", 1,
     ("k_disga_fwd<%s, 3, -1," % V4, "k_disga_bwd_dst<%s, 3, -1," % V4, "k_disga_bwd_src<%s, 3, 2," % V4)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", LAYER_CASES, ids=lambda c: c[0])
def test_layer_kernels_on_many_units_vs_float64(big, case, monkeypatch):
    name, att, gnn, C, D, F_, train, gx_term, plan, G, kernels = case
    idx, graph = big
    info = graph.info
    assert min(info["dst_items"], info["src_items"]) * G >= units_needed(), (info, G)
    assert info["dst_slots"] > 0, info
    e_cnt = idx.shape[1]
    monkeypatch.setenv("EDIS_AT_PLAN", plan)
    monkeypatch.setattr(layers, "_next_seed", lambda: SEED)
    torch.manual_seed(C * 100 + F_)
    gen = torch.Generator().manual_seed(C * 100 + F_)
    chs = [edis.DisGALayer(F_, D, dropout=P_DROP, alpha=0.1, att_type=att, gnn_type=gnn) for _ in range(C)]
    for l in chs:
        if att == 3:
            l.W.data = torch.cat([exact_w(F_, D, gen), exact_w(F_, D, gen)], 0)
        else:
            l.W.data = exact_w(F_, D, gen, coherent=False)
    x_cpu = exact_x(N, F_, gen)
    r_out = torch.randn(N, C * D)
    r_e = torch.randn(e_cnt, C) if gx_term else None
    keep = torch.from_numpy(edge_keep(SEED, e_cnt, C, P_DROP)) if train else None

    # the score operands come out of the device projection exactly (run_channels' GEMM path at this N)
    if att == 3:
        w_score = torch.cat([torch.cat([l.W[:F_] for l in chs], 1), torch.cat([l.W[F_:] for l in chs], 1)], 1)
    else:
        w_score = torch.cat([l.W for l in chs], 1)
    w_score = w_score.detach()
    with torch.no_grad():
        xd, wd = x_cpu.to(DEV), w_score.to(DEV)
        proj = Fn.Proj3xTF32.apply(xd, wd) if Fn.use_proj3x(N) else xd @ wd
    exact = x_cpu.double() @ w_score.double()
    assert torch.equal(proj.cpu().double(), exact), "score projection is not exact"
    if att == 3:
        assert bool((exact != 0).all())
    del proj, xd, wd, exact

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
    for want in kernels:
        assert_ran(names, want)
    assert not [k for k in names if "_ring" in k], sorted(names)
    got = {"gx": x.grad.cpu()}
    for c, l in enumerate(chs):
        got.update({"c%d.%s" % (c, k): v.grad.cpu() for k, v in l.named_parameters() if v.grad is not None})

    o64, e64, gx64, g64 = oracle(chs, att, gnn, x_cpu, idx, keep, r_out, r_e, torch.float64)
    assert rel_err(out.detach().cpu(), o64) <= RT, "out"
    assert rel_err(e.detach().cpu(), e64) <= RT, "edge_e"
    del o64, e64
    _, _, gx32, g32 = oracle(chs, att, gnn, x_cpu, idx, keep, r_out, r_e, torch.float32)
    g64["gx"], g32["gx"] = gx64, gx32
    floor = group_floor([v for k, v in g64.items() if k != "gx" and v is not None])
    assert set(got) == {k for k, v in g64.items() if v is not None}      # att 2 does not use a
    bad = []
    for k in sorted(got):
        err, tol = grad_tol(got[k], g64[k], g32[k], 0.0 if k == "gx" else floor)
        if k.endswith(".a"):
            # the suite's bound for the tiny score-vector gradients (test_gpu_trainers.py): the kernels' single-pass
            # softmax backward (t_i = <gh_i, agg_i> from the stored aggregate) is ill-conditioned for them, 6e-5 in
            # plain fp32 torch too (test_oracle_golden.py::test_single_pass_softmax_backward_conditioning)
            tol = max(tol, 1e-4)
        if err > tol:
            bad.append("%s: rel err %.3e > %.1e" % (k, err, tol))
    assert not bad, bad


# ------------------------------------------------------------------ pair scoring
def pair_restatement(att, pi, pj, P, Q, a, g, dtype, chunk=CHUNK):
    """Logits of channels [c_lo, c_hi) on the pairs (pi, pj) and their gradients for the upstream gradient g,
    in `dtype`, CHUNK pairs at a time.  P [nP, Cs, D] / Q [nQ, Cs, D] (att 2 / 3) or P [nP, Cs] / Q [nQ, Cs]
    (att 1) hold the range's channels, a [Cs, D] (att 3).
      att 1: P_i,c + Q_j,c      att 2: <P_i,c, Q_j,c>      att 3: lrelu_0.01(P_i,c + Q_j,c) . a_c
    -> (out [M, Cs], gP, gQ, ga, sum over pairs of |g lrelu(z)|); the last two are None unless att 3."""
    P, Q, g = P.to(dtype), Q.to(dtype), g.to(dtype)
    m = pi.numel()
    out = torch.empty((m,) + P.shape[1:2], dtype=dtype, device=P.device)
    gP, gQ = torch.zeros_like(P), torch.zeros_like(Q)
    ga = ga_abs = None
    if att == 3:
        a = a.to(dtype)
        ga, ga_abs = torch.zeros_like(a), torch.zeros_like(a)
    for s in range(0, m, chunk):
        i, j, gg = pi[s:s + chunk], pj[s:s + chunk], g[s:s + chunk]
        if att == 1:
            out[s:s + chunk] = P[i] + Q[j]
            gP.index_add_(0, i, gg)
            gQ.index_add_(0, j, gg)
            continue
        pI, qJ = P[i], Q[j]
        if att == 2:
            out[s:s + chunk] = (pI * qJ).sum(-1)
            gP.index_add_(0, i, gg.unsqueeze(-1) * qJ)
            gQ.index_add_(0, j, gg.unsqueeze(-1) * pI)
            continue
        z = pI + qJ
        pos = z > 0
        lr = torch.where(pos, z, 0.01 * z)
        out[s:s + chunk] = (lr * a).sum(-1)
        dz = gg.unsqueeze(-1) * a * torch.where(pos, z.new_ones(()), z.new_full((), 0.01))
        gP.index_add_(0, i, dz)
        gQ.index_add_(0, j, dz)
        t = gg.unsqueeze(-1) * lr
        ga += t.sum(0)
        ga_abs += t.abs().sum(0)
    return out, gP, gQ, ga, ga_abs


PAIR_CASES = [
    # (id, att, C, channel ranges, layout, G per range, backward kernel, P column offset, own rows of P or None)
    ("a3_C8_sign", 3, 8, [(0, 8)], V2, 2, "k_pair_bwd_sign<%s>" % V2, 0, None),
    ("a3_C8_halves", 3, 8, [(0, 4), (4, 8)], V2, 1, "k_pair_bwd_sign<%s>" % V2, 0, None),
    ("a3_C12_G3", 3, 12, [(0, 12)], V2, 3, "k_pair_bwd_sign<%s>" % V2, 0, None),
    ("a3_C10_halves_G5", 3, 10, [(0, 5), (5, 10)], "edis::ScaT<2>", 5, "k_pair_bwd_sign<edis::ScaT<2>>", 0, None),
    ("a3_C8_unaligned", 3, 8, [(0, 8)], "edis::ScaT<2>", 8, "k_pair_bwd<edis::ScaT<2>, 3>", 1, None),
    ("a2_C8", 2, 8, [(0, 8)], V2, 2, "k_pair_bwd<%s, 2>" % V2, 0, None),
    ("a1_C6", 1, 6, [(0, 6)], V1, 3, "k_pair_bwd<%s, 1>" % V1, 0, None),
    ("a3_C8_rect", 3, 8, [(0, 8)], V2, 2, "k_pair_bwd_sign<%s>" % V2, 0, 60_000),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", PAIR_CASES, ids=lambda c: c[0])
def test_pair_kernels_on_many_units_vs_float64(sample, case):
    name, att, C, ranges, layout, G, bwd_kernel, p0, n_own = case
    D, F_ = 64, 16
    CD = C * D
    pairs, _ = sample
    pl = Fn.PairList(pairs)
    m = pairs.shape[1] if n_own is None else int(torch.searchsorted(pairs[0], torch.tensor(n_own, device=DEV)))
    if n_own is not None:          # this rank's rows [0, n_own) against all N columns (own rows + halo)
        pl = Fn.PairList(pairs[:, :m])
        assert int(pairs[1, :m].max()) >= n_own
    assert math.ceil(m / 32) * G >= units_needed(), (m, G)
    gen = torch.Generator().manual_seed(C * 10 + att + p0)
    torch.manual_seed(C * 10 + att + p0)
    n_p = N if n_own is None else n_own
    if att == 1:
        P_cpu, Q_cpu, a_cpu = torch.randn(n_p, C), torch.randn(N, C), None
        P = P_cpu.to(DEV).requires_grad_(True)
        Q = Q_cpu.to(DEV).requires_grad_(True)
        blocks = {"P": P_cpu, "Q": Q_cpu}
    else:
        # P | Q | V column blocks of one projection buffer, as run_channels lays them out (exact construction)
        x = exact_x(N, F_, gen)
        w = exact_w(F_, 3 * CD, gen)
        buf_cpu = x @ w
        q0 = CD if p0 == 0 else 2 * CD              # the unaligned P keeps Q aligned on the third block
        if att == 2:
            q0 = p0                                  # one block: P = Q, as run_channels passes att 2
        for c0 in {p0, q0}:
            blk = x.double() @ w[:, c0:c0 + CD].double()
            assert torch.equal(buf_cpu[:, c0:c0 + CD].double(), blk) and bool((blk != 0).all())
        a_cpu = torch.randn(C, D) if att == 3 else None
        buf = buf_cpu.to(DEV).requires_grad_(True)
        P, Q = buf[:n_p, p0:p0 + CD], buf[:, q0:q0 + CD]
        blocks = {"P": buf_cpu[:n_p, p0:p0 + CD].reshape(n_p, C, D), "Q": buf_cpu[:, q0:q0 + CD].reshape(N, C, D)}
        if att == 3:
            # columns are sign-coherent: where the signs of P and Q differ, z = P_i + Q_j takes both signs
            assert bool((blocks["P"][0] * blocks["Q"][0] < 0).any())
    a = a_cpu.to(DEV).requires_grad_(True) if a_cpu is not None else None
    gs = [torch.randn(m, hi - lo, device=DEV) for lo, hi in ranges]

    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        outs = [Fn.PairScore.apply(att, C, D, pl.pi, pl.pj, lo, hi, P, Q, a, pl) for lo, hi in ranges]
        # the sign-record backward needs the forward's record: it exists exactly for the aligned att-3 cases
        assert all((o.grad_fn.saved_tensors[-1] is not None) == ("sign" in bwd_kernel) for o in outs)
        loss = sum((o * g).sum() for o, g in zip(outs, gs))
        loss.backward()
        torch.cuda.synchronize()
    names = cuda_kernels(prof)
    assert_ran(names, bwd_kernel, count=(2 if "sign" in bwd_kernel else 1) * len(ranges))
    outs = [o.detach().cpu() for o in outs]

    blocks = {k: v.to(DEV) for k, v in blocks.items()}
    a_d = None if a_cpu is None else a_cpu.to(DEV)

    def restate(dtype):
        res = {k: torch.zeros(v.shape, dtype=dtype, device=DEV) for k, v in blocks.items()}
        if att == 3:
            res["a"], res["a_abs"] = (torch.zeros(C, D, dtype=dtype, device=DEV) for _ in range(2))
        logits = []
        for (lo, hi), g in zip(ranges, gs):
            o, gP, gQ, ga, ga_abs = pair_restatement(att, pl.pi, pl.pj, blocks["P"][:, lo:hi], blocks["Q"][:, lo:hi],
                                                     None if a_d is None else a_d[lo:hi], g, dtype)
            logits.append(o.cpu())
            res["P"][:, lo:hi] += gP
            res["Q"][:, lo:hi] += gQ
            if att == 3:
                res["a"][lo:hi] += ga
                res["a_abs"][lo:hi] += ga_abs
        return logits, {k: v.cpu() for k, v in res.items()}

    l64, r64 = restate(torch.float64)
    for (lo, hi), o, ref in zip(ranges, outs, l64):
        assert rel_err(o, ref) <= RT, ("logits", lo, hi)
    _, r32 = restate(torch.float32)
    if att == 1:
        got = {"P": P.grad.cpu(), "Q": Q.grad.cpu()}
    else:
        gbuf = buf.grad.cpu()
        got = {"P": gbuf[:n_p, p0:p0 + CD].reshape(n_p, C, D), "Q": gbuf[:, q0:q0 + CD].reshape(N, C, D)}
        if att == 2:                                   # one block: its gradient is gP + gQ
            got = {"PQ": got["P"]}
            r64 = {"PQ": r64["P"] + r64["Q"]}
            r32 = {"PQ": r32["P"] + r32["Q"]}
        if att == 3:
            got["a"] = a.grad.cpu()
    floor = group_floor([r64[k] for k in got])
    bad = []
    for k in sorted(got):
        err, tol = grad_tol(got[k], r64[k], r32[k], floor)
        if k == "a":
            # ga sums g * lrelu(z) over every pair of the list (~2M terms per element, reduced by each warp
            # and then by atomics in an arbitrary order): first-order rounding bound 2^-24 x sum |terms|
            tol = max(tol, 2.0 ** -24 * float(r64["a_abs"].max()) / max(float(r64["a"].abs().max()), floor))
        if err > tol:
            bad.append("%s: rel err %.3e > %.1e" % (k, err, tol))
    assert not bad, bad


# ------------------------------------------------------------------ class-balanced MSE at the same M
def wmse_float64(s, y, n_pos, m_total):
    """utils.adj_mse_loss(sigmoid(s.sum(1)), y) with the pair set's total size and positive count."""
    pred = torch.sigmoid(s.sum(1))
    w = torch.where(y != 0, torch.ones_like(pred), torch.full_like(pred, n_pos / (m_total ** 2 - n_pos)))
    return (w * (pred - y) ** 2).sum() / m_total


@pytest.mark.gpu
@pytest.mark.parametrize("cs,parts", [(4, 1), (8, 1), (8, 3)], ids=["cs4", "cs8", "cs8_partitioned"])
def test_ssl_wmse_on_sampled_pairs_vs_float64(sample, cs, parts):
    _, label = sample
    m = label.numel()
    torch.manual_seed(cs + parts)
    s = torch.randn(m, cs)
    y = label.cpu()
    n_pos = int((y != 0).sum())
    m_total, n_pos_total = parts * m, parts * n_pos       # one rank's slice of a pair set `parts` times larger
    refs = {}
    for dt in (torch.float64, torch.float32):
        sr = s.detach().clone().to(dt).requires_grad_(True)
        if parts == 1:
            ref = od.adj_mse_loss(torch.sigmoid(sr.sum(1)), y.to(dt))
            assert abs(float(ref) - float(wmse_float64(sr.detach(), y.to(dt), n_pos, m))) <= 1e-12 * float(ref)
        else:
            ref = wmse_float64(sr, y.to(dt), n_pos_total, m_total)
        ref.backward()
        refs[dt] = (float(ref), sr.grad)
    sg = s.detach().to(DEV).requires_grad_(True)
    if parts == 1:
        loss = Fn.SslWmse.apply(sg, label, n_pos)
    else:
        loss = Fn.SslWmse.apply(sg, label, n_pos_total, m_total)
    loss.backward()
    ref64, g64 = refs[torch.float64]
    assert abs(loss.item() - ref64) <= RT * abs(ref64), (loss.item(), ref64)
    err, tol = grad_tol(sg.grad.cpu(), g64, refs[torch.float32][1], 0.0)
    assert err <= tol, (err, tol)


# ------------------------------------------------------------------ CPU: the construction and the restatement
def test_exact_operands_are_exact_and_take_both_signs():
    gen = torch.Generator().manual_seed(0)
    for f in (15, 16, 64):
        x = exact_x(4096, f, gen)
        wt, wb = exact_w(f, 64, gen), exact_w(f, 64, gen)
        for w in (wt, wb):
            # every entry is on the TF32 grid: the 3xTF32 split has zero low parts
            assert torch.equal(Fn._tf32_hi(w), w) and torch.equal(Fn._tf32_hi(x), x)
        P, Q = x @ wt, x @ wb
        assert torch.equal(P.double(), x.double() @ wt.double())
        assert torch.equal(Q.double(), x.double() @ wb.double())
        assert bool((P != 0).all()) and bool((Q != 0).all())
        i = torch.randint(0, 4096, (20000,), generator=gen)
        j = torch.randint(0, 4096, (20000,), generator=gen)
        z = P[i] + Q[j]
        assert torch.equal(z.double(), P[i].double() + Q[j].double())
        assert bool((z > 0).any()) and bool((z < 0).any())
        # the logits stay O(1): the softmax's sigmoid does not saturate
        assert float(z.abs().mean()) < 2.0


@pytest.mark.parametrize("att", [1, 2, 3])
def test_pair_restatement_matches_oracle_pair_logits(att):
    """pair_restatement (P / Q form) equals oracle.disgat.pair_logits ([x_i || x_j] W form, pinned by the
    goldens) in value and in the gradients of W and a, through W = [W_top; W_bot] (att 3) or h = x W."""
    torch.manual_seed(att)
    n, f, d, m = 60, 7, 5, 400
    x = torch.randn(n, f, dtype=torch.float64)
    pairs = torch.stack([torch.randint(0, n, (m,)), torch.randint(0, n, (m,))])
    pairs = pairs[:, torch.argsort(pairs[0])]
    W = torch.randn(2 * f if att == 3 else f, d, dtype=torch.float64, requires_grad=True)
    a = torch.randn(d if att == 3 else 2 * d, 1, dtype=torch.float64, requires_grad=True)
    g = torch.randn(m, 1, dtype=torch.float64)
    ref = od.pair_logits(x, W, a, pairs, att)
    (ref * g).sum().backward()
    Wd, ad = W.detach(), a.detach()
    if att == 3:
        P, Q = (x @ Wd[:f]).reshape(n, 1, d), (x @ Wd[f:]).reshape(n, 1, d)
        out, gP, gQ, ga, _ = pair_restatement(3, pairs[0], pairs[1], P, Q, ad.reshape(1, d), g, torch.float64)
        gW = torch.cat([x.t() @ gP.reshape(n, d), x.t() @ gQ.reshape(n, d)], 0)
        ga = ga.reshape(d, 1)
    elif att == 2:
        h = (x @ Wd).reshape(n, 1, d)
        out, gP, gQ, _, _ = pair_restatement(2, pairs[0], pairs[1], h, h, None, g, torch.float64)
        gW = x.t() @ (gP + gQ).reshape(n, d)
        ga = None                                      # att 2 does not use a
    else:
        h = x @ Wd
        P, Q = h @ ad[:d], h @ ad[d:]
        out, gP, gQ, _, _ = pair_restatement(1, pairs[0], pairs[1], P, Q, None, g, torch.float64)
        gW = x.t() @ (gP @ ad[:d].t() + gQ @ ad[d:].t())
        ga = torch.cat([h.t() @ gP, h.t() @ gQ], 0)
    assert rel_err(out, ref.detach()) <= 1e-12
    assert rel_err(gW, W.grad) <= 1e-12
    assert (ga is None and a.grad is None) or rel_err(ga, a.grad) <= 1e-12


def test_exact_cancellation_takes_the_lower_slope_in_torch():
    """z = P + Q = +0 from nonzero P, Q: torch's leaky_relu backward (like the kernels' sign record, where
    w = -P - Q = +0 has its sign bit clear) takes the 0.01 side."""
    P = torch.tensor([0.5, -0.375], dtype=torch.float64)
    Q = torch.tensor([-0.5, 0.375], dtype=torch.float64, requires_grad=True)
    z = P + Q
    assert bool((z == 0).all()) and not bool(torch.signbit(z).any())
    torch.nn.functional.leaky_relu(z).sum().backward()
    assert torch.equal(Q.grad, torch.full((2,), 0.01, dtype=torch.float64))
    w = (-P.float()) - Q.detach().float()
    assert not bool(torch.signbit(w).any())
