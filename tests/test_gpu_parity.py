"""GPU parity tests (run on the B200 box: `pytest -m gpu`).

Everything here goes through the C ABI (ctypes -> libedis.so) and is compared with
  (i) golden vectors produced by the unmodified reference (tests/golden/*.npz), and
  (ii) the CPU oracle (oracle/) on seeded random graphs with hubs, split rows, ragged shapes.
Tolerance: 1e-5 relative to the tensor's scale for fp32 results (north_star); bit-exact for
graph structure.
"""
import numpy as np
import pytest
import torch

import edgedisentangle_ssl_b200 as edis
from edgedisentangle_ssl_b200 import functional as Fn
from edgedisentangle_ssl_b200.layers import run_channels
from oracle import disgat as od
from oracle import graph as og
from helpers import load, t, assert_close, params_from, group_floor

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(autouse=True, params=["agg", "proj"])
def at_plan(request, monkeypatch):
    """Run every test under both execution plans of gnn_type AT / GCN (layers.run_channels):
    aggregate-then-project (shared-operand kernels) and project-then-aggregate (DisGAFused)."""
    monkeypatch.setenv("EDIS_AT_PLAN", request.param)
    return request.param
RT = 1e-5
RT_GRAD = 2e-5   # gradients: long reassociated sums over edges / nodes (see grad_tol)


def cuda_adj(n, indices):
    idx = torch.as_tensor(indices, dtype=torch.int64)
    return torch.sparse_coo_tensor(idx, torch.ones(idx.shape[1]), (n, n)).to(DEV)


def hub_graph(n, m, seed, hub_deg=None):
    rng = np.random.RandomState(seed)
    src = rng.randint(0, n, size=m)
    dst = rng.randint(0, n, size=m)
    hub_deg = hub_deg or n // 2
    dst[:hub_deg] = 1                      # a hub destination (long CSR row)
    src[:hub_deg] = rng.permutation(n)[:hub_deg]
    idx, _ = og.build_adjacency(n, dst, src)
    return idx


# ------------------------------------------------------------------ graph handle
def test_graph_handle_csr_csc():
    g = load("layer_s64")
    n, idx = int(g["n"]), g["indices"]
    gr = edis.Graph(n, idx[0], idx[1], device=DEV, max_chunk=8)
    ex = gr.export()
    assert gr.e == idx.shape[1] and gr.info["was_sorted"]
    assert np.array_equal(ex["rowptr"], np.concatenate([[0], np.cumsum(np.bincount(idx[0], minlength=n))]))
    assert np.array_equal(ex["col"], idx[1].astype(np.int32))
    assert np.array_equal(ex["perm"], np.arange(gr.e))
    assert np.array_equal(gr.indices.cpu().numpy(), idx)
    # CSC: slot k of column j holds (row, csr slot) sorted by row
    eid = ex["csceid"]
    assert np.array_equal(np.sort(eid), np.arange(gr.e))
    assert np.array_equal(idx[0][eid], ex["cscrow"])
    assert np.array_equal(np.repeat(np.arange(n), np.diff(ex["cscptr"])), idx[1][eid])
    assert gr.info["dst_slots"] > 0 and gr.info["max_in"] > 8   # hub row got split


def test_graph_handle_unsorted_duplicates():
    rng = np.random.RandomState(0)
    n = 50
    r, c = rng.randint(0, n, 400), rng.randint(0, n, 400)
    gr = edis.Graph(n, r, c, device=DEV)
    key = np.unique(r * n + c)
    ex = gr.export()
    assert gr.e == key.shape[0] and not gr.info["was_sorted"]
    rows = np.repeat(np.arange(n), np.diff(ex["rowptr"]))
    assert np.array_equal(rows * n + ex["col"], key)
    assert np.array_equal(key[ex["perm"]], r * n + c)   # every input entry maps to its slot


# ------------------------------------------------------------------ one channel vs reference golden
def make_layer(g, k, fin, dd, att, gnn):
    lay = edis.DisGALayer(fin, dd, dropout=0.3, alpha=0.1, concat=True, att_type=att, gnn_type=gnn)
    sd = {name: v for name, v in params_from(g, k + "p.").items()}
    lay.load_state_dict(sd, strict=True)
    return lay.to(DEV).eval()


@pytest.mark.parametrize("tag", ["s8", "s64"])
@pytest.mark.parametrize("att", [1, 2, 3])
@pytest.mark.parametrize("gnn", ["AT", "SAGE", "GCN"])
def test_layer_vs_reference_golden(tag, att, gnn):
    g = load("layer_" + tag)
    k = "a%d_%s_" % (att, gnn)
    x = t(g["x"]).to(DEV).requires_grad_(True)
    n, fin = x.shape
    dd = g[k + "out"].shape[1]
    lay = make_layer(g, k, fin, dd, att, gnn)
    adj = cuda_adj(n, g["indices"])
    aux = [t(g["aux0"]).to(DEV), t(g["aux1"]).to(DEV)]
    out, e, au = lay(x, adj, aux)
    assert_close(out.cpu(), g[k + "out"], RT, "out")
    assert_close(e.cpu(), g[k + "edge_e"], RT, "edge_e")
    assert_close(au[0].cpu(), g[k + "aux0"], RT, "aux0")
    assert_close(au[1].cpu(), g[k + "aux1"], RT, "aux1")
    loss = (out * t(g["r_out"]).to(DEV)).sum() + (e * t(g["r_e"]).to(DEV)).sum() \
        + (au[0] * t(g["r_aux0"]).to(DEV)).sum() + (au[1] * t(g["r_aux1"]).to(DEV)).sum()
    loss.backward()
    assert_close(x.grad.cpu(), g[k + "gx"], RT_GRAD, "gx")
    floor = group_floor([v for kk, v in g.items() if kk.startswith(k + "g.")])
    for name, prm in lay.named_parameters():
        if k + "g." + name in g:
            assert_close(prm.grad.cpu(), g[k + "g." + name], RT_GRAD, "g." + name, floor)
        else:
            assert prm.grad is None or float(prm.grad.abs().max()) == 0.0


# ------------------------------------------------------------------ model vs reference golden
MODEL_TAGS = ["model_a3_AT", "model_a1_SAGE", "model_a2_GCN", "model_a3_AT_res"]


def model_from_golden(tag):
    from edgedisentangle_ssl_b200.utils import get_parser
    g = load(tag)
    args = get_parser().parse_args([str(a) for a in g["argv"]])
    args.cuda, args.hetero = True, True
    args.size = g["x"].shape[1]
    enc = edis.DISGAT(args, nfeat=args.size, nhid=args.nhid, nclass=args.nhid, nheads=args.nhead,
                      dropout=args.dropout)
    enc.load_state_dict(params_from(g, "enc0."), strict=True)
    fus = []
    for i, res in ((1, args.size), (2, args.nhid)):
        f = edis.FuseLayer(args, args.nhead, nfeat=args.nhid, residue=res if args.residue else 0)
        f.load_state_dict(params_from(g, "cls0.fuse%d." % i), strict=True)
        fus.append(f.to(DEV))
    return g, args, enc.to(DEV), fus


@pytest.mark.parametrize("tag", MODEL_TAGS)
def test_model_traversal_vs_reference_golden(tag):
    g, args, enc, fus = model_from_golden(tag)
    enc.eval()
    x = t(g["x"]).to(DEV)
    adj = cuda_adj(int(g["n"]), g["indices"])
    aux = [t(g["aux0"]).to(DEV), t(g["aux1"]).to(DEV)]
    with torch.no_grad():
        em = enc.get_em(x, adj, fus)
        assert_close(em[0].cpu(), g["get_em_1"], RT, "get_em[0]")
        assert_close(em[1].cpu(), g["get_em_2"], RT, "get_em[1]")
        assert_close(enc(x, adj, fus).cpu(), g["forward"], RT, "forward")
        ga = enc.get_adjs(x, adj, fus)
        pa = enc.predict_adjs_sparse(x, adj, fus, aux)
        ge = enc.get_edge_em(x, adj, fus)
    for layer in range(2):
        assert_close(torch.stack(ga[layer]).cpu(), g["get_adjs"][layer], RT, "get_adjs")
        assert_close(torch.stack([h[0] for h in pa[layer]]).cpu(), g["pred_aux0"][layer], RT, "aux0")
        assert_close(torch.stack([h[1] for h in pa[layer]]).cpu(), g["pred_aux1"][layer], RT, "aux1")
        assert_close(torch.stack(ge[layer]).cpu(), g["edge_em_l%d" % layer], RT, "edge_em")


def cls_step_grads_fp64(g, args):
    """Encoder gradients of the recorded CLS step evaluated in float64 by the oracle."""
    dd = torch.float64
    p = {k: v.to(dd).requires_grad_(True) for k, v in params_from(g, "enc0.").items()}
    fus = [{k: v.to(dd) for k, v in params_from(g, "cls0.fuse%d." % i).items()} for i in (1, 2)]
    mp = {k: v.to(dd) for k, v in params_from(g, "cls0.classifier.").items()}
    r = od.disgat_traverse(p, fus, t(g["x"]).to(dd), t(g["indices"]), args.nhead, args.att, args.gnn_type,
                           residue=args.residue, residue_type=args.residue_type)
    tr = t(g["cls_idx_train"])
    torch.nn.functional.nll_loss(od.mlp(mp, r["feats"][-1], cls=True)[tr], t(g["labels"])[tr]).backward()
    return {k: v.grad for k, v in p.items()}


@pytest.mark.parametrize("tag", MODEL_TAGS)
def test_model_cls_step_grads_vs_reference_golden(tag):
    """First recorded train step (CLS, dropout 0): loss and encoder / fuser gradients."""
    g, args, enc, fus = model_from_golden(tag)
    enc.train()
    clf = edis.MLP(in_feat=args.nhid, hidden_size=args.nhid, out_size=int(g["labels"].max()) + 1, layers=2)
    clf.load_state_dict(params_from(g, "cls0.classifier."), strict=True)
    clf.to(DEV)
    x, labels = t(g["x"]).to(DEV), t(g["labels"]).to(DEV)
    adj = cuda_adj(int(g["n"]), g["indices"])
    out = clf(enc.get_em(x, adj, fus)[-1], cls=True)
    tr = t(g["cls_idx_train"]).to(DEV)
    loss = torch.nn.functional.nll_loss(out[tr], labels[tr])
    assert_close(loss.item(), g["cls.log.loss_train"], RT, "loss_train")
    loss.backward()
    checked = 0
    floor = group_floor([v for k, v in g.items() if k.startswith("cls.encgrad.")])
    truth = cls_step_grads_fp64(g, args)
    for name, prm in enc.named_parameters():
        key = "cls.encgrad." + name
        if key in g:
            assert_close(prm.grad.cpu(), g[key], grad_tol(g[key], truth[name]), key, floor)
            checked += 1
    assert checked >= 8
    for name, prm in fus[0].named_parameters():
        assert_close(prm.grad.cpu(), g["cls.fuse1grad." + name], RT_GRAD, "fuse1." + name)


# ------------------------------------------------------------------ fused channels vs CPU oracle
def grad_tol(ref32, ref64):
    """Gradient tolerance: 2e-5, or 16x the error the reference's own fp32 arithmetic makes
    against a float64 evaluation of the same formula.  Softmax-backward gradients are differences of
    nearly equal terms (d alpha - sum_k alpha_k d alpha_k), so every fp32 evaluation order -- the
    reference's included -- carries cancellation noise well above 1e-5 of the result on some tensors."""
    from helpers import rel_err
    return max(RT_GRAD, 16.0 * rel_err(ref32, ref64))


def oracle_layer_all(chs, x_cpu, idx, att, gnn, aux, r_out, r_e, r_aux, dtype=torch.float32, keep=None):
    """Run the oracle per channel; returns outputs and grads in the fused layout.
    keep: [E, C] dropout multipliers (the kernels' own mask, helpers.edge_keep) or None (no dropout).
    r_e None: the loss has no edge_e term.  Output rows past r_out's (the halo sources of a rectangular
    slice) are not destinations and are dropped."""
    p = {}
    for c, l in enumerate(chs):
        for name, prm in l.named_parameters():
            p["c%d.%s" % (c, name)] = prm.detach().cpu().clone().to(dtype).requires_grad_(True)
    x = x_cpu.clone().to(dtype).requires_grad_(True)
    r_out, r_aux = r_out.to(dtype), [r.to(dtype) for r in r_aux]
    outs, es, auxs = [], [], []
    for c in range(len(chs)):
        o, e, au = od.disga_layer(p, "c%d." % c, x, idx, att, gnn, aux=aux,
                                  keep=None if keep is None else keep[:, c:c + 1])
        outs.append(o)
        es.append(e)
        auxs.append(au)
    out = torch.cat(outs, 1)[:r_out.shape[0]]
    e = torch.cat(es, 1)
    au = [torch.cat([a_[k] for a_ in auxs], 1) for k in range(len(aux))]
    loss = (out * r_out).sum() + sum((a_ * r).sum() for a_, r in zip(au, r_aux))
    if r_e is not None:
        loss = loss + (e * r_e.to(dtype)).sum()
    loss.backward()
    return out, e, au, x.grad, p


CASES = [
    # (n, m, C, D, F, max_chunk[, kind])
    (300, 2500, 4, 64, 24, 16),     # VecT<2,16>, split rows
    (257, 1800, 8, 64, 100, 32),    # C=8 (config A shape), F=100
    (200, 1500, 2, 64, 16, 0),      # VecT<1,16>
    (150, 900, 3, 20, 10, 8),       # scalar path, odd C, D not multiple of 4... (20 is), ragged
    (120, 700, 2, 13, 7, 0),        # scalar path, D % 4 != 0
    (90, 500, 4, 32, 12, 4),        # VecT<1,8>
    (80, 400, 1, 128, 9, 0),        # VecT<1,32>
    (260, 2200, 8, 64, 64, 16),     # F == D == 64: shared operand on the 128-bit layout (layer-2 shape), split rows
    (180, 1400, 4, 64, 64, 0),      # same, VecT<2,16>
    (150, 1000, 2, 64, 64, 8),      # same, VecT<1,16>
    (200, 150, 4, 64, 16, 0, "sparse"),   # low degree; train mode at p = 0.9 drops every in-edge of some rows
    (400, 3500, 8, 64, 20, 16, "slice"),  # middle destination range of a partition: rectangular, n_cols > n
]

# (att, mode): train mode draws the dropout mask in the kernels (seed fixed below); "train-no-e" leaves
# edge_e out of the loss, so the backward runs without a logit gradient (the benchmark's combination)
ATT_MODES = [pytest.param(att, mode, id=str(att) if mode == "eval" else "%d-%s" % (att, mode))
             for att, mode in [(1, "eval"), (1, "train"), (2, "eval"), (2, "train"), (3, "eval"), (3, "train"),
                               (3, "train-no-e")]]
SEED = 0xD1B54A32D192ED03     # both 32-bit halves of the seed enter the mask
P_TRAIN = 0.3


def slice_of(idx_np, n):
    """Middle third of the destination rows of a square graph in a partition's local indexing
    (own columns first, then halo), row-major sorted.  -> (indices, rows, columns)."""
    from edgedisentangle_ssl_b200 import parallel as par
    lo, hi = n // 3, 2 * n // 3
    sel = (idx_np[0] >= lo) & (idx_np[0] < hi)
    row_l, col_l, halo = par.compact_columns(lo, hi, idx_np[0][sel], idx_np[1][sel])
    order = np.lexsort((col_l, row_l))
    return np.stack([row_l[order], col_l[order]]), hi - lo, hi - lo + len(halo)


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("att,mode", ATT_MODES)
@pytest.mark.parametrize("gnn", ["AT", "GCN", "SAGE"])
def test_fused_channels_vs_oracle(case, att, mode, gnn, monkeypatch):
    from edgedisentangle_ssl_b200 import layers
    from helpers import edge_keep
    n, m, C, D, Fin, max_chunk = case[:6]
    kind = case[6] if len(case) > 6 else None
    train = mode != "eval"
    p = (0.9 if kind == "sparse" else P_TRAIN) if train else 0.2
    torch.manual_seed(1000 + n + att)
    idx_np = hub_graph(n, m, seed=n)
    n_cols = n
    if kind == "slice":
        idx_np, n, n_cols = slice_of(idx_np, n)
    idx = torch.from_numpy(idx_np)
    e_cnt = idx.shape[1]
    chs = [edis.DisGALayer(Fin, D, dropout=p, alpha=0.1, att_type=att, gnn_type=gnn) for _ in range(C)]
    x_cpu = torch.randn(n_cols, Fin)
    rng = np.random.RandomState(7)
    aux = [torch.from_numpy(np.sort(rng.randint(0, n * n, 333))).long()]
    aux = [torch.stack([a_ // n, a_ % n]) for a_ in aux] + [torch.from_numpy(rng.randint(0, n, (2, 65))).long()]
    r_out, r_e = torch.randn(n, C * D), torch.randn(e_cnt, C)
    r_aux = [torch.randn(a_.shape[1], C) for a_ in aux]
    if mode == "train-no-e":
        r_e = None
    keep = None
    if train:
        keep = edge_keep(SEED, e_cnt, C, p)
        if kind == "sparse":
            kept = np.zeros((n, C))
            np.add.at(kept, idx_np[0], keep > 0)
            assert (kept == 0).any(), "no (row, channel) pair with every in-edge dropped"
        keep = torch.from_numpy(keep)
    o_ref, e_ref, au_ref, gx_ref, p_ref = oracle_layer_all(chs, x_cpu, idx, att, gnn, aux, r_out, r_e, r_aux,
                                                           keep=keep)
    _, _, _, gx_64, p_64 = oracle_layer_all(chs, x_cpu, idx, att, gnn, aux, r_out, r_e, r_aux, torch.float64,
                                            keep=keep)

    monkeypatch.setattr(layers, "_next_seed", lambda: SEED)
    for l in chs:
        l.to(DEV).train(train)
    graph = edis.Graph(n, idx_np[0], idx_np[1], device=DEV, max_chunk=max_chunk, n_cols=n_cols)
    assert graph.info["was_sorted"]
    x = x_cpu.to(DEV).requires_grad_(True)
    out, e, au = run_channels(chs, x, graph, [a_.to(DEV) for a_ in aux])
    assert_close(out.cpu(), o_ref, RT, "out")
    assert_close(e.cpu(), e_ref, RT, "edge_e")
    for k in range(2):
        assert_close(au[k].cpu(), au_ref[k], RT, "aux%d" % k)
    loss = (out * r_out.to(DEV)).sum() + sum((a_ * r.to(DEV)).sum() for a_, r in zip(au, r_aux))
    if r_e is not None:
        loss = loss + (e * r_e.to(DEV)).sum()
    loss.backward()
    assert_close(x.grad.cpu(), gx_ref, grad_tol(gx_ref, gx_64), "gx")
    floor = group_floor([v.grad for v in p_ref.values() if v.grad is not None])
    for c, l in enumerate(chs):
        for name, prm in l.named_parameters():
            key = "c%d.%s" % (c, name)
            ref = p_ref[key].grad
            if ref is None:
                assert prm.grad is None or float(prm.grad.abs().max()) == 0.0
            else:
                assert_close(prm.grad.cpu(), ref, grad_tol(ref, p_64[key].grad), key, floor)


@pytest.mark.parametrize("C", [2, 8, 16])
@pytest.mark.parametrize("p", [0.1, 0.5, 0.9])
@pytest.mark.parametrize("seed", [12345, SEED])
def test_dropout_mask_matches_port(C, p, seed, monkeypatch):
    """Every row has exactly one in-edge (CSR slot e = row e) and every V row is all-ones, so the
    train-mode output is the mask itself: zero exactly where helpers.keep_scale drops, 1/(1-p) elsewhere.
    C = 16 runs the LDG kernels with two channel groups; the agg plan runs the shared-operand kernels."""
    from edgedisentangle_ssl_b200 import layers
    from helpers import edge_keep
    n, D, Fin = 4096, 64, 64
    perm = np.random.RandomState(C).permutation(n)
    graph = edis.Graph(n, np.arange(n), perm, device=DEV)
    torch.manual_seed(C)
    chs = [edis.DisGALayer(Fin, D, dropout=p, alpha=0.1, att_type=3, gnn_type="AT") for _ in range(C)]
    for l in chs:
        l.W_em.data.fill_(1.0 / Fin)
        l.to(DEV).train()
    monkeypatch.setattr(layers, "_next_seed", lambda: seed)
    with torch.no_grad():
        out, _, _ = run_channels(chs, torch.ones(n, Fin, device=DEV), graph)
    out = out.reshape(n, C, D).cpu().numpy()
    keep = edge_keep(seed, n, C, p)
    assert np.array_equal(out == 0, np.broadcast_to((keep == 0)[:, :, None], out.shape))
    kept = keep > 0
    assert kept.any() and (~kept).any()
    ref = np.broadcast_to(keep[:, :, None], out.shape)[kept]
    assert np.abs(out[kept] - ref).max() <= 1e-6 * ref.max()


def test_isolated_rows_and_empty_pairs():
    """Rows without in-edges aggregate to 0 (elu(0) = 0); an empty pair list is legal."""
    n, C, D, Fin = 40, 2, 64, 8
    rows = np.array([0, 0, 3, 5, 5, 5], dtype=np.int64)
    cols = np.array([1, 2, 3, 0, 5, 7], dtype=np.int64)
    graph = edis.Graph(n, rows, cols, device=DEV)
    chs = [edis.DisGALayer(Fin, D, 0.0, 0.1, att_type=3, gnn_type="AT").to(DEV).eval() for _ in range(C)]
    x = torch.randn(n, Fin, device=DEV, requires_grad=True)
    empty = torch.zeros(2, 0, dtype=torch.int64, device=DEV)
    out, e, au = run_channels(chs, x, graph, [empty])
    assert au[0].shape == (0, C) and e.shape == (6, C)
    mask = torch.ones(n, dtype=torch.bool)
    mask[[0, 3, 5]] = False
    assert float(out[mask.to(DEV)].abs().max()) == 0.0
    out.sum().backward()
    assert torch.isfinite(x.grad).all()


# ------------------------------------------------------------------ 3xTF32 projection
def test_proj3x_tf32_is_fp32_accurate():
    torch.manual_seed(0)
    x = (torch.randn(20000, 100, device=DEV) * torch.logspace(-3, 3, 100, device=DEV)).requires_grad_(True)
    w = torch.randn(100, 1536, device=DEV, requires_grad=True)
    ref = x.double() @ w.double()
    got = Fn.Proj3xTF32.apply(x, w)
    plain = x @ w
    e3, e1 = ((got.double() - ref).abs().max() / ref.abs().max()).item(), \
        ((plain.double() - ref).abs().max() / ref.abs().max()).item()
    assert e3 < 2e-6 and e3 < 8 * max(e1, 1e-7), (e3, e1)
    r = torch.randn_like(got)
    gx, gw = torch.autograd.grad((got * r).sum(), (x, w))
    gx2, gw2 = torch.autograd.grad((plain * r).sum(), (x, w))
    assert torch.equal(gx, gx2) and torch.equal(gw, gw2)     # backward is the plain fp32 one


# ------------------------------------------------------------------ destination-range partition
@pytest.mark.parametrize("att,gnn", [(3, "AT"), (1, "GCN"), (2, "SAGE")])
def test_partitioned_matches_full_graph(att, gnn):
    """Rectangular (own rows x own+halo columns) graphs: running each destination range on its own
    compact slice and summing the weight / input gradients reproduces the full-graph result."""
    from edgedisentangle_ssl_b200 import parallel as par
    n, C, D, Fin = 400, 4, 64, 20
    idx_np = hub_graph(n, 3500, seed=11)
    torch.manual_seed(5)
    chs = [edis.DisGALayer(Fin, D, 0.0, 0.1, att_type=att, gnn_type=gnn).to(DEV).eval() for _ in range(C)]
    x = torch.randn(n, Fin, device=DEV, requires_grad=True)
    R = torch.randn(n, C * D, device=DEV)
    full = edis.Graph(n, idx_np[0], idx_np[1], device=DEV, max_chunk=32)
    out_full, _, _ = run_channels(chs, x, full)
    (out_full * R).sum().backward()
    ref = {"x": x.grad.clone()}
    for c, l in enumerate(chs):
        for name, prm in l.named_parameters():
            if prm.grad is not None:
                ref["c%d.%s" % (c, name)] = prm.grad.clone()
                prm.grad = None
    x.grad = None
    rowptr = np.concatenate([[0], np.cumsum(np.bincount(idx_np[0], minlength=n))])
    bounds = par.row_ranges(rowptr, 3)
    outs = []
    for r in range(3):
        lo, hi = int(bounds[r]), int(bounds[r + 1])
        sel = (idx_np[0] >= lo) & (idx_np[0] < hi)
        row_l, col_l, halo = par.compact_columns(lo, hi, idx_np[0][sel], idx_np[1][sel])
        g = edis.Graph(hi - lo, row_l, col_l, device=DEV, max_chunk=32, n_cols=hi - lo + len(halo))
        assert g.n_cols > g.n
        x_need = torch.cat([x[lo:hi], x[torch.from_numpy(halo).to(DEV)]], 0)
        o, _, _ = run_channels(chs, x_need, g)
        (o * R[lo:hi]).sum().backward()
        outs.append(o.detach())
    assert_close(torch.cat(outs, 0).cpu(), out_full.detach().cpu(), RT, "partitioned out")
    floor = group_floor([v.cpu() for v in ref.values()])
    assert_close(x.grad.cpu(), ref["x"].cpu(), RT_GRAD, "gx", floor)
    for c, l in enumerate(chs):
        for name, prm in l.named_parameters():
            if prm.grad is not None:
                assert_close(prm.grad.cpu(), ref["c%d.%s" % (c, name)].cpu(), 5e-5, "c%d.%s" % (c, name), floor)


# ------------------------------------------------------------------ dropout (train mode)
def fused(graph, att, C, D, P, Q, a, V, training=False, p=0.0, seed=0):
    """DisGAFused on explicit operands (builds the [N, W] projection block the op expects)."""
    CD = C * D
    if att == 3:
        proj, offs = torch.cat([P, Q, V], 1), (0, CD, 2 * CD)
    else:
        proj, offs = torch.cat([P, V], 1), (0, 0, CD)
    return Fn.DisGAFused.apply(graph, att, C, D, proj, offs[0], offs[1], offs[2], None, None, a, None,
                               training, p, seed)


def test_dropout_is_reproducible_and_consistent_between_fwd_and_bwd():
    n, m, C, D = 300, 3000, 4, 64
    idx_np = hub_graph(n, m, seed=3)
    graph = edis.Graph(n, idx_np[0], idx_np[1], device=DEV, max_chunk=32)
    torch.manual_seed(0)
    P, Q, V = (torch.randn(n, C * D, device=DEV) for _ in range(3))
    a = torch.randn(C, D, device=DEV)
    V = V.requires_grad_(True)
    o1, _ = fused(graph, 3, C, D, P, Q, a, V, True, 0.5, 1234)
    o2, _ = fused(graph, 3, C, D, P, Q, a, V, True, 0.5, 1234)
    o3, _ = fused(graph, 3, C, D, P, Q, a, V, True, 0.5, 99)
    o_eval, _ = fused(graph, 3, C, D, P, Q, a, V, False, 0.5, 0)
    assert torch.equal(o1, o2) and not torch.equal(o1, o3) and not torch.equal(o1, o_eval)
    # same mask in fwd and bwd: directional derivative wrt V (finite differences, fixed seed)
    r = torch.randn(n, C * D, device=DEV)
    (gV,) = torch.autograd.grad((o1 * r).sum(), V)
    dV = torch.randn_like(V)
    eps = 1e-3
    op, _ = fused(graph, 3, C, D, P, Q, a, (V + eps * dV).detach(), True, 0.5, 1234)
    om, _ = fused(graph, 3, C, D, P, Q, a, (V - eps * dV).detach(), True, 0.5, 1234)
    fd = (((op - om) * r).sum() / (2 * eps)).item()
    an = (gV * dV).sum().item()
    assert abs(fd - an) <= 5e-3 * max(1.0, abs(an)), (fd, an)
    # keep rate: E[alpha_drop] = alpha  ->  the train-mode aggregate is an unbiased estimate
    ones = torch.ones(n, C * D, device=DEV)
    outs = torch.stack([fused(graph, 2, C, D, P, P, None, ones, True, 0.5, s)[0] for s in range(24)]).mean(0)
    assert abs(outs.mean().item() - 1.0) < 0.02     # elu(1) = 1 when every V row is all-ones


# ------------------------------------------------------------------ SSL ops
@pytest.mark.parametrize("cs", [1, 4, 8])
def test_ssl_wmse_vs_oracle(cs):
    torch.manual_seed(cs)
    m = 5000
    s = torch.randn(m, cs)
    tgt = (torch.rand(m) < 0.11).float()
    s_ref = s.clone().requires_grad_(True)
    ref = od.adj_mse_loss(torch.sigmoid(s_ref.sum(1)), tgt)
    ref.backward()
    sg = s.to(DEV).requires_grad_(True)
    loss = Fn.SslWmse.apply(sg, tgt.to(DEV), int((tgt != 0).sum()))
    assert_close(loss.item(), ref.item(), RT, "wmse")
    (loss * 3.0).backward()
    assert_close(sg.grad.cpu(), 3.0 * s_ref.grad, RT, "wmse grad")


def test_ssl_wmse_vs_reference_golden():
    g = load("loss_small")
    pred = t(g["pred"])
    logit = torch.log(pred / (1 - pred)).unsqueeze(1).to(DEV)   # sigmoid^-1, one channel
    tgt = t(g["tgt"]).to(DEV)
    loss = Fn.SslWmse.apply(logit, tgt, int((tgt != 0).sum()))
    assert_close(loss.item(), float(g["loss"]), 1e-5, "adj_mse_loss golden")


@pytest.mark.parametrize("k", [4, 8])
def test_nll_const_label_vs_torch(k):
    torch.manual_seed(k)
    n = 3001
    z = torch.randn(n, k) * 3
    for label in (0, k - 1):
        z_ref = z.clone().requires_grad_(True)
        ref = torch.nn.functional.nll_loss(torch.log_softmax(z_ref, 1), torch.full((n,), label))
        ref.backward()
        zg = z.to(DEV).requires_grad_(True)
        loss = Fn.NllConstLabel.apply(zg, label)
        assert_close(loss.item(), ref.item(), RT, "nll")
        loss.backward()
        assert_close(zg.grad.cpu(), z_ref.grad, RT, "nll grad")


@pytest.mark.parametrize("tag", ["s8", "s64"])
def test_sp_ops_vs_reference_golden(tag):
    from edgedisentangle_ssl_b200 import utils as U
    g = load("layer_" + tag)
    idx = t(g["indices"]).to(DEV)
    vals = t(g["spmm_vals"]).to(DEV).requires_grad_(True)
    mat = t(g["spmm_mat"]).to(DEV).requires_grad_(True)
    n = int(g["n"])
    out = U.sp_matmul(idx, vals, mat)
    assert_close(out.cpu(), g["spmm_out"], RT, "sp_matmul")
    sm = U.sp_softmax(idx, vals, n)
    assert_close(sm.cpu(), g["spsm_out"], RT, "sp_softmax")
    # gradients vs the oracle's autograd
    r1, r2 = torch.randn(out.shape), torch.randn(sm.shape)
    ((out * r1.to(DEV)).sum() + (sm * r2.to(DEV)).sum()).backward()
    v_ref = t(g["spmm_vals"]).clone().requires_grad_(True)
    m_ref = t(g["spmm_mat"]).clone().requires_grad_(True)
    ic = t(g["indices"])
    ((od.sp_matmul(ic, v_ref, m_ref) * r1).sum() + (od.sp_softmax(ic, v_ref, n) * r2).sum()).backward()
    assert_close(vals.grad.cpu(), v_ref.grad, RT_GRAD, "g values")
    assert_close(mat.grad.cpu(), m_ref.grad, RT_GRAD, "g mat")


# ------------------------------------------------------------------ size-independent properties
@pytest.mark.parametrize("n,raw", [(100_000, 1_000_000), (2_400_000, 30_600_000)],
                         ids=["2M-edges", "configA-63M-edges"])
def test_large_graph_properties(n, raw, at_plan):
    """Power-law graph, C=8, D=64, at 2M edges and at BASELINE config[3]'s FULL size (2.4M nodes,
    63M edges): softmax rows sum to one (all-ones V -> out == 1), the aggregate is linear in V,
    and the source pass is the exact adjoint of the forward."""
    from edgedisentangle_ssl_b200.synthetic import power_law_graph
    C, D = 8, 64
    if n > 1_000_000 and at_plan != "proj":
        pytest.skip("full size once (these calls go to DisGAFused directly: the plan does not matter)")
    idx = power_law_graph(n, raw, seed=5 if n < 1_000_000 else 0)
    graph = edis.Graph(n, idx[0], idx[1], device=DEV)
    del idx
    assert graph.info["max_in"] > 1000
    torch.manual_seed(0)
    P = torch.randn(n, C * D, device=DEV) * 0.3
    Q = torch.randn(n, C * D, device=DEV) * 0.3
    a = torch.randn(C, D, device=DEV) * 0.3
    ones = torch.ones(n, C * D, device=DEV)
    out, e = fused(graph, 3, C, D, P, Q, a, ones)
    assert float((out - 1).abs().max()) < 2e-6
    V1, V2 = torch.randn(n, C * D, device=DEV), torch.randn(n, C * D, device=DEV)
    pos = lambda V: fused(graph, 3, C, D, P, Q, a, V)  # noqa: E731
    # inverse-elu makes the comparison linear: compare pre-activations via positive shifts
    big = 50.0
    o1, _ = pos(V1 + big)
    o2, _ = pos(V2 + big)
    o12, _ = pos(V1 + V2 + big)
    assert float(((o1 - big) + (o2 - big) - (o12 - big)).abs().max()) < 2e-4
    # adjoint: <A V, R> == <V, A^T R>
    Vg = V1.clone().requires_grad_(True)
    o, _ = pos(Vg + big)
    R = torch.randn_like(o)
    (gV,) = torch.autograd.grad((o * R).sum(), Vg)
    lhs = ((o - big) * R).sum().double().item()
    rhs = (gV * V1).sum().double().item()
    assert abs(lhs - rhs) <= 1e-4 * max(abs(lhs), 1.0), (lhs, rhs)


def test_node_linear_backward_matches_float64():
    """FuseLayer's Linear on a node tensor large enough for the custom backward (3xTF32 input
    gradient, slab-wise weight gradient): same numbers as the float64 evaluation to fp32 accuracy."""
    from edgedisentangle_ssl_b200.functional import node_linear
    torch.manual_seed(0)
    n, fin, fout = 300_000, 512, 64
    lin = torch.nn.Linear(fin, fout).to(DEV)
    x = torch.randn(n, fin, device=DEV, requires_grad=True)
    r = torch.randn(n, fout, device=DEV)
    (node_linear(lin, x) * r).sum().backward()
    x64 = x.detach().double().requires_grad_(True)
    w64 = lin.weight.detach().double().requires_grad_(True)
    b64 = lin.bias.detach().double().requires_grad_(True)
    ((x64 @ w64.t() + b64) * r.double()).sum().backward()
    assert_close(x.grad.cpu(), x64.grad.float().cpu(), 2e-6, "gx")
    assert_close(lin.weight.grad.cpu(), w64.grad.float().cpu(), 2e-5, "gw")
    assert_close(lin.bias.grad.cpu(), b64.grad.float().cpu(), 2e-5, "gb")


def test_recompute_projection_is_bit_identical_and_leaner(monkeypatch, at_plan):
    """EDIS_RECOMPUTE_PROJ=1: the saved projection is replaced by a marker and recomputed in the
    backward -- identical outputs, same gradients, lower peak memory across two layers."""
    if at_plan != "proj":
        pytest.skip("the projection is only saved by the project-then-aggregate plan")
    from edgedisentangle_ssl_b200.synthetic import power_law_graph
    n, C, D, Fin = 60_000, 8, 64, 100
    idx = power_law_graph(n, 300_000, seed=2)
    graph = edis.Graph(n, idx[0], idx[1], device=DEV)
    torch.manual_seed(1)
    l1 = [edis.DisGALayer(Fin, D, 0.0, 0.1, att_type=3, gnn_type="AT").to(DEV).eval() for _ in range(C)]
    l2 = [edis.DisGALayer(C * D, D, 0.0, 0.1, att_type=3, gnn_type="AT").to(DEV).eval() for _ in range(C)]
    x0 = torch.randn(n, Fin, device=DEV)
    R = torch.randn(n, C * D, device=DEV)

    def run(mode):
        monkeypatch.setenv("EDIS_RECOMPUTE_PROJ", mode)
        for l in l1 + l2:
            l.zero_grad(set_to_none=True)
        x = x0.clone().requires_grad_(True)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        h, _, _ = run_channels(l1, x, graph)
        o, _, _ = run_channels(l2, h, graph)
        (o * R).sum().backward()
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        grads = [x.grad.clone()] + [p.grad.clone() for l in l1 + l2 for p in l.parameters() if p.grad is not None]
        return o.detach().clone(), grads, peak

    o_a, g_a, peak_a = run("0")
    o_b, g_b, peak_b = run("1")
    assert torch.equal(o_a, o_b)
    assert len(g_a) == len(g_b)
    for k, (a_, b_) in enumerate(zip(g_a, g_b)):
        # same operands bit for bit; only the atomically accumulated `a` gradients may differ in
        # the order of their float additions between any two runs
        assert_close(b_.cpu(), a_.cpu(), 1e-5, "grad %d" % k)
    assert peak_b < peak_a - n * 3 * C * D * 4 * 0.5, (peak_a, peak_b)     # at least half a projection saved
