"""Pin the CPU oracle against golden vectors produced by the unmodified reference.

(CPU only.)  The goldens come from tests/golden/make_golden.py.
"""
import hashlib
import os
import random

import numpy as np
import pytest
import torch

from oracle import disgat as od
from oracle import graph as og
from helpers import load, t, assert_close, params_from, rel_err, GOLDEN

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


# ------------------------------------------------------------------ graph construction
def test_graph_edge_list_bit_exact():
    g = load("graph_small")
    n, r, c = og.edge_list_to_coo(g["el_edges"])
    assert n == int(g["el_n"])
    idx, val = og.build_adjacency(n, r, c)
    assert np.array_equal(idx, g["el_indices"])
    assert np.array_equal(val, g["el_values"])
    assert np.array_equal(og.features_row_normalize(g["el_feat"]).astype(np.float32), g["el_features"])


def test_graph_weighted_csr_bit_exact():
    g = load("graph_small")
    idx, val = og.build_adjacency(int(g["csr_n"]), g["csr_row"], g["csr_col"], g["csr_val"])
    assert np.array_equal(idx, g["csr_indices"])
    assert np.array_equal(val, g["csr_values"])


@pytest.mark.parametrize("ds", ["cora", "chameleon", "cora_full"])
def test_graph_bundled_hash(ds):
    import scipy.sparse as sp
    g = load("graph_bundled")
    d = os.path.join(ROOT, "data", ds)
    if os.path.exists(os.path.join(d, "adj_1.npy")):
        n, r, c = og.edge_list_to_coo(np.load(os.path.join(d, "adj_1.npy")))
        v = None
    else:
        m = sp.load_npz(os.path.join(d, "adj_1_sp.npz")).tocoo()
        n, r, c, v = m.shape[0], m.row, m.col, m.data
    idx, val = og.build_adjacency(n, r, c, v)
    assert n == int(g[ds + "_n"]) and idx.shape[1] == int(g[ds + "_e"])
    assert sha(idx) == str(g[ds + "_idx_sha"])
    assert sha(val) == str(g[ds + "_val_sha"])


def test_sampler_cora_bit_exact():
    import scipy.sparse as sp
    g = load("graph_bundled")
    m = sp.load_npz(os.path.join(ROOT, "data", "cora", "adj_1_sp.npz")).tocoo()
    idx, _ = og.build_adjacency(m.shape[0], m.row, m.col, m.data)
    torch.manual_seed(4)
    np.random.seed(4)
    pairs, lab = og.sample_pairs(m.shape[0], idx, chunk_rows=677)
    assert pairs.shape[1] == int(g["cora_sample_m"])
    assert sha(pairs) == str(g["cora_sample_idx_sha"])
    assert sha(lab) == str(g["cora_sample_lab_sha"])


# ------------------------------------------------------------------ sparse ops / loss
@pytest.mark.parametrize("tag", ["s8", "s64"])
def test_sp_ops(tag):
    g = load("layer_" + tag)
    idx = t(g["indices"])
    assert_close(od.sp_matmul(idx, t(g["spmm_vals"]), t(g["spmm_mat"])), g["spmm_out"], what="sp_matmul")
    assert_close(od.sp_softmax(idx, t(g["spmm_vals"]), int(g["n"])), g["spsm_out"], what="sp_softmax")


def test_adj_mse_loss():
    g = load("loss_small")
    assert_close(od.adj_mse_loss(t(g["pred"]), t(g["tgt"])), g["loss"], what="adj_mse_loss")


# ------------------------------------------------------------------ one channel
@pytest.mark.parametrize("tag", ["s8", "s64"])
@pytest.mark.parametrize("att", [1, 2, 3])
@pytest.mark.parametrize("gnn", ["AT", "SAGE", "GCN"])
def test_layer_fwd_bwd(tag, att, gnn):
    g = load("layer_" + tag)
    k = "a%d_%s_" % (att, gnn)
    p = {n_: v.clone().requires_grad_(True) for n_, v in params_from(g, k + "p.").items()}
    x = t(g["x"]).clone().requires_grad_(True)
    idx = t(g["indices"])
    aux = [t(g["aux0"]), t(g["aux1"])]
    out, e, au = od.disga_layer(p, "", x, idx, att, gnn, aux=aux)
    assert_close(out, g[k + "out"], what="out")
    assert_close(e, g[k + "edge_e"], what="edge_e")
    assert_close(au[0], g[k + "aux0"], what="aux0")
    assert_close(au[1], g[k + "aux1"], what="aux1")
    loss = (out * t(g["r_out"])).sum() + (e * t(g["r_e"])).sum() \
        + (au[0] * t(g["r_aux0"])).sum() + (au[1] * t(g["r_aux1"])).sum()
    loss.backward()
    assert_close(x.grad, g[k + "gx"], what="gx")
    for name, prm in p.items():
        if k + "g." + name in g:
            assert_close(prm.grad, g[k + "g." + name], what="g." + name)
        else:  # att=2: `a` receives no gradient in the reference
            assert prm.grad is None or float(prm.grad.abs().max()) == 0.0


# ------------------------------------------------------------------ model traversal + losses
MODEL_TAGS = ["model_a3_AT", "model_a1_SAGE", "model_a2_GCN", "model_a3_AT_res"]


def model_setup(tag):
    g = load(tag)
    argv = [str(a) for a in g["argv"]]
    att = int([a for a in argv if a.startswith("--att=")][0].split("=")[1])
    gnn = [a for a in argv if a.startswith("--gnn_type=")][0].split("=")[1]
    cfg = dict(nheads=4, att=att, gnn=gnn, residue="--residue" in argv,
               residue_type=2 if "--residue_type=2" in argv else 0,
               constrain_layer=1 if "--constrain_layer=1" in argv else 0)
    return g, cfg


def fusers_of(g, who):
    return [params_from(g, "%s0.fuse1." % who), params_from(g, "%s0.fuse2." % who)]


@pytest.mark.parametrize("tag", MODEL_TAGS)
def test_model_traversal(tag):
    g, cfg = model_setup(tag)
    p = params_from(g, "enc0.")
    x, idx = t(g["x"]), t(g["indices"])
    aux = [t(g["aux0"]), t(g["aux1"])]
    with torch.no_grad():
        r = od.disgat_traverse(p, fusers_of(g, "cls"), x, idx, cfg["nheads"], cfg["att"], cfg["gnn"],
                               aux=aux, residue=cfg["residue"], residue_type=cfg["residue_type"])
    assert_close(r["feats"][0], g["get_em_1"], what="get_em[0]")
    assert_close(r["feats"][1], g["get_em_2"], what="get_em[1]")
    assert_close(r["logp"], g["forward"], what="forward")
    for layer in range(2):
        assert_close(torch.stack(r["edge_e"][layer]), g["get_adjs"][layer], what="get_adjs")
        assert_close(torch.stack([h[0] for h in r["aux"][layer]]), g["pred_aux0"][layer], what="aux0")
        assert_close(torch.stack([h[1] for h in r["aux"][layer]]), g["pred_aux1"][layer], what="aux1")
        assert_close(torch.stack(r["edge_em"][layer]), g["edge_em_l%d" % layer], what="edge_em")


def seed_all(s):
    random.seed(s)
    np.random.seed(s)
    torch.manual_seed(s)


@pytest.mark.parametrize("tag", MODEL_TAGS)
def test_sampler_small_bit_exact(tag):
    g, cfg = model_setup(tag)
    n, idx = int(g["n"]), g["indices"]
    seed_all(8)
    pairs, lab = og.sample_pairs(n, idx, chunk_rows=16)
    assert np.array_equal(pairs, g["sup.sample_idx"])
    assert np.array_equal(lab, g["sup.sample_lab"])
    homo, het = og.homo_hetero_split(idx, g["labels"])
    seed_all(9)
    p0, l0 = og.sample_pairs(n, homo, chunk_rows=32)
    p1, l1 = og.sample_pairs(n, het, chunk_rows=48)
    assert np.array_equal(p0, g["dis.sample_idx0"]) and np.array_equal(l0, g["dis.sample_lab0"])
    assert np.array_equal(p1, g["dis.sample_idx1"]) and np.array_equal(l1, g["dis.sample_lab1"])


@pytest.mark.parametrize("tag", MODEL_TAGS[:1] + MODEL_TAGS[3:])
def test_first_step_losses_and_grads(tag):
    """CLS step (first in the recorded sequence, so the encoder is still enc0)."""
    g, cfg = model_setup(tag)
    p = {k: v.clone().requires_grad_(True) for k, v in params_from(g, "enc0.").items()}
    fus = [{k: v.clone().requires_grad_(True) for k, v in f.items()} for f in fusers_of(g, "cls")]
    mp = params_from(g, "cls0.classifier.")
    x, idx, labels = t(g["x"]), t(g["indices"]), t(g["labels"])
    r = od.disgat_traverse(p, fus, x, idx, cfg["nheads"], cfg["att"], cfg["gnn"],
                           residue=cfg["residue"], residue_type=cfg["residue_type"])
    logp = od.mlp(mp, r["feats"][-1], cls=True)
    tr = t(g["cls_idx_train"])
    loss = torch.nn.functional.nll_loss(logp[tr], labels[tr])
    assert_close(loss, g["cls.log.loss_train"], rtol=1e-5, what="cls loss")
    loss.backward()
    for k, prm in p.items():
        key = "cls.encgrad." + k
        if key in g:
            assert_close(prm.grad, g[key], rtol=2e-5, what=key)
    for k, prm in fus[0].items():
        assert_close(prm.grad, g["cls.fuse1grad." + k], rtol=2e-5, what="fuse1 " + k)


# ------------------------------------------------------------------ bundled graphs (BASELINE configs)
@pytest.mark.parametrize("ds,att,gnn", [("cora", 3, "AT"), ("chameleon", 3, "AT"), ("chameleon", 1, "SAGE"),
                                        ("chameleon", 2, "GCN")])
def test_oracle_on_bundled_graphs_vs_reference_samples(ds, att, gnn):
    """The oracle against what the UNMODIFIED reference produced on the bundled graphs with the same
    seeded weights (tests/golden/bundled_ref.npz): logits / alpha at 512 fixed edges, elu(h') and
    feature_2 at 64 fixed nodes.  (The CUDA path is checked against both in tests/test_gpu_bundled.py.)"""
    import test_gpu_bundled as tb
    g = load("bundled_ref")
    k = "%s.a%d_%s." % (ds, att, gnn)
    adj, x, labels = tb.dataset(ds)
    idx = adj.indices().numpy()
    n = adj.shape[0]
    args, enc, fus, clf = tb.build_edis(att, gnn, x.shape[1])
    assert abs(tb.state_checksum([enc] + fus + clf) - float(g[k + "state_checksum"])) < 1e-6 * float(g[k + "state_checksum"])
    p = {kk: v.detach().clone() for kk, v in enc.state_dict().items() if kk.startswith("attention")}
    fp = [{kk: v.detach().clone() for kk, v in f.state_dict().items()} for f in fus]
    with torch.no_grad():
        r = od.disgat_traverse(p, fp, x, torch.from_numpy(idx), tb.C, att, gnn)
    sel_e, sel_n = g[ds + ".sel_e"], g[ds + ".sel_n"]
    for l in range(2):
        e = torch.cat(r["edge_e"][l], 1)
        assert rel_err(e[sel_e], g[k + "e%d" % l], floor=float(g[k + "e%d_absmax" % l])) <= 1e-5
        al = torch.cat([od.sp_softmax(torch.from_numpy(idx), torch.sigmoid(ec), n) for ec in r["edge_e"][l]], 1)
        assert rel_err(al[sel_e], g[k + "alpha%d" % l], floor=1.0) <= 1e-5
        out = torch.cat([em[:, -tb.D:] for em in r["edge_em"][l]], 1)
        assert rel_err(out[sel_n], g[k + "out%d" % l], floor=float(g[k + "out%d_absmax" % l])) <= 1e-5
    assert rel_err(r["feats"][-1][sel_n], g[k + "feat2"], floor=float(g[k + "feat2_absmax"])) <= 1e-5


def test_single_pass_softmax_backward_conditioning():
    """Why the `a` gradients get 1e-4 (not 2e-5) against the float64 arbiter in tests/test_gpu_trainers.py.

    The kernels compute the softmax backward d logit_ij = alpha_ij (dalpha_ij - t_i) s'(e_ij) in ONE pass over
    a row, with t_i = <gh_i, agg_i> taken from the stored aggregate instead of a second reduction
    sum_k alpha_ik dalpha_ik.  Both are the same number in exact arithmetic; in fp32 the stored aggregate is
    rounded independently of the dalpha_ik, so the cancellation dalpha - t sees an extra ~1e-7 |dalpha| error.
    On layer 2 of the toy models (near-constant messages: dalpha - t is ~1e-3 of dalpha) that shows up on the
    tiny `a` gradients.  This test reproduces both forms in plain fp32 torch on the CPU -- no kernel involved --
    against float64: the two-reduction (reference) form stays below 2e-5, the single-pass form below 1e-4."""
    import torch.nn.functional as F
    from edgedisentangle_ssl_b200.utils import get_parser
    from helpers import group_floor
    g = load("model_a3_AT_res")
    args = get_parser().parse_args([str(a) for a in g["argv"]])
    n, idx, labels, it = int(g["n"]), torch.as_tensor(g["indices"]), t(g["labels"]), t(g["cls_idx_train"])
    kw = dict(residue=bool(args.residue), residue_type=args.residue_type, no_relu=bool(args.fuse_no_relu))

    def run(dt):
        p = {k: v.to(dt).requires_grad_(True) for k, v in params_from(g, "enc0.").items() if k.startswith("attention")}
        fus = [{k: v.to(dt) for k, v in params_from(g, "cls0.fuse%d." % i).items()} for i in (1, 2)]
        clf = {k: v.to(dt) for k, v in params_from(g, "cls0.classifier.").items()}
        r = od.disgat_traverse(p, fus, t(g["x"]).to(dt), idx, args.nhead, args.att, args.gnn_type, **kw)
        F.nll_loss(od.mlp(clf, r["feats"][-1], cls=True)[it], labels[it]).backward()
        return {k: v.grad for k, v in p.items() if v.grad is not None}

    class SinglePass(torch.autograd.Function):
        @staticmethod
        def forward(ctx, e, V, row, col, n_):
            w = torch.exp(torch.sigmoid(e))
            den = torch.zeros(n_, 1, dtype=e.dtype).index_add_(0, row, w)
            alpha = w / den[row]
            agg = torch.zeros(n_, V.shape[1], dtype=e.dtype).index_add_(0, row, alpha * V[col])
            ctx.save_for_backward(e, V, row, col, alpha, agg)
            return agg

        @staticmethod
        def backward(ctx, gh):
            e, V, row, col, alpha, agg = ctx.saved_tensors
            tc = (gh * agg).sum(1, keepdim=True)                      # t_i from the stored aggregate
            gdot = (gh[row] * V[col]).sum(1, keepdim=True)
            s = torch.sigmoid(e)
            de = alpha * (gdot - tc[row]) * s * (1 - s)
            return de, torch.zeros_like(V).index_add_(0, col, alpha * gh[row]), None, None, None

    def single_pass_layer(p, prefix, x, indices, att, gnn, dropout=0.0, training=False, aux=None):
        e = od.pair_logits(x, p[prefix + "W"], p[prefix + "a"], indices, att)
        h = SinglePass.apply(e, x @ p[prefix + "W_em"], indices[0], indices[1], x.size(0))
        return F.elu(h), e

    g64, g32 = run(torch.float64), run(torch.float32)
    orig = od.disga_layer
    od.disga_layer = single_pass_layer
    try:
        s32 = run(torch.float32)
    finally:
        od.disga_layer = orig
    floor = group_floor(g64.values())
    two = max(rel_err(g32[k], g64[k], floor) for k in g64)
    one = max(rel_err(s32[k], g64[k], floor) for k in g64)
    print("fp32 vs float64, worst tensor: two-reduction form %.2e, single-pass form %.2e" % (two, one))
    assert two < 2e-5 and one < 1e-4


# ------------------------------------------------------------------ the kernels' dropout mask, restated
def test_dropout_mask_port_keep_rate_and_high_words():
    """helpers.keep_scale (the numpy restatement the train-mode GPU tests build their oracle mask with):
    keep rate 1 - p, multiplier float32 1 / (1 - p), and both 32-bit halves of the seed and of the
    element index change the mask."""
    from helpers import keep_scale
    idx = np.arange(1 << 20, dtype=np.uint64)
    seed = 0xD1B54A32D192ED03
    for p in (0.1, 0.5, 0.9):
        k = keep_scale(seed, idx, p)
        assert k.dtype == np.float32
        assert set(np.unique(k)) == {np.float32(0), np.float32(1) / (np.float32(1) - np.float32(p))}
        assert abs((k > 0).mean() - (1 - p)) < 3e-3, p
    base = keep_scale(seed, idx[:4096], 0.5) > 0
    for other in (keep_scale(seed ^ (1 << 40), idx[:4096], 0.5), keep_scale(seed, idx[:4096] + np.uint64(1 << 33), 0.5),
                  keep_scale(seed ^ 1, idx[:4096], 0.5)):
        assert 0.4 < ((other > 0) != base).mean() < 0.6
    assert np.array_equal(keep_scale(seed, idx[:4096], 0.5), keep_scale(seed, idx[:4096], 0.5))


def test_oracle_keep_replaces_dropout():
    """disga_layer(keep=...) multiplies alpha by the given mask: an all-kept mask of ones is the eval
    result, and a mask that drops every in-edge of a row zeroes that row's AT output."""
    torch.manual_seed(0)
    n, fin, d = 30, 5, 4
    idx = torch.from_numpy(og.build_adjacency(n, np.arange(n), (np.arange(n) + 1) % n)[0])
    p = {"W": torch.randn(2 * fin, d), "a": torch.randn(d, 1), "W_em": torch.randn(fin, d)}
    x = torch.randn(n, fin)
    o0, e0 = od.disga_layer(p, "", x, idx, 3, "AT")
    o1, e1 = od.disga_layer(p, "", x, idx, 3, "AT", keep=torch.ones(idx.shape[1], 1))
    assert torch.equal(o0, o1) and torch.equal(e0, e1)
    keep = torch.full((idx.shape[1], 1), 2.0)
    keep[idx[0] == 3] = 0.0
    o2, _ = od.disga_layer(p, "", x, idx, 3, "AT", keep=keep)
    assert float(o2[3].abs().max()) == 0.0
    rest = torch.arange(n) != 3
    h0 = torch.where(o0 > 0, o0, torch.log1p(o0))     # inverse elu
    h2 = torch.where(o2 > 0, o2, torch.log1p(o2))
    assert torch.allclose(h2[rest], 2 * h0[rest], rtol=1e-5, atol=1e-6)
