"""Oracle (CPU, torch eager) for the DISGAT layers, traversal and SSL losses.

TEST INFRASTRUCTURE ONLY -- see oracle/__init__.py.  This restates the reference's
algorithm op for op (per-channel Python loop, [E, 2F] gathers, scatter_add) so that
(i) autograd supplies reference gradients and (ii) timing it is a fair "port" of the
reference's CPU path.  Parameters are passed as a flat dict keyed by the reference's
state_dict names (`attention1_0.W`, ...), so a reference state_dict loads unchanged.
"""
import torch
import torch.nn.functional as F


# --------------------------------------------------------------------------- sparse ops
def sp_softmax(indices, values, n):
    """Per-row softmax of edge values.  Follows utils.py:192-200.

    Shift is the GLOBAL max over all edges, groups are rows (indices[0]),
    denominator gets +1e-10.
    """
    row = indices[0]
    shifted = torch.exp(values - values.max())
    denom = torch.zeros(n, 1, dtype=values.dtype)
    denom.scatter_add_(0, row.unsqueeze(1), shifted)
    denom = denom + 1e-10
    return shifted / denom[row]


def sp_matmul(indices, values, mat):
    """out[i] = sum_{(i,j)} values_ij * mat[j].  Follows utils.py:203-207 (square adj)."""
    row, col = indices[0], indices[1]
    out = torch.zeros_like(mat)
    out.scatter_add_(0, row.unsqueeze(1).expand(-1, mat.size(1)), values * mat[col])
    return out


# --------------------------------------------------------------------------- one channel
def pair_logits(x, W, a, pairs, att):
    """Raw (pre-sigmoid) attention logit on arbitrary (i, j) pairs.

    Follows layers.py:349-389: att=1 `[hW_i || hW_j] a`; att=2 `<hW_i, hW_j>`;
    att=3 `lrelu_0.01([x_i || x_j] W) a`.  pairs[0] = i (row/dst), pairs[1] = j (col/src).
    """
    i, j = pairs[0], pairs[1]
    if att == 1:
        h = x @ W
        return torch.cat((h[i], h[j]), dim=1) @ a
    if att == 2:
        h = x @ W
        return (h[i] * h[j]).sum(-1, keepdim=True)
    if att == 3:
        z = torch.cat((x[i], x[j]), dim=1) @ W
        return F.leaky_relu(z) @ a
    raise ValueError(att)


def disga_layer(p, prefix, x, indices, att, gnn, dropout=0.0, training=False, aux=None, keep=None):
    """One DisGALayer channel, sparse branch, incl. the ELU of `forward`.

    Follows layers.py:340-416 and 493-511.  `p[prefix + 'W']` etc. are the parameters.
    `keep` ([E,1] multipliers: 0 or 1/(1-p)) replaces the dropout of alpha by a given mask, e.g. the
    one a kernel drew, so that a train-mode result can be compared element for element.
    Returns (elu(h'), edge_e[E,1] raw logits, [aux logits]) -- aux list only if given.
    """
    n = x.size(0)
    W, a = p[prefix + "W"], p[prefix + "a"]
    edge_e = pair_logits(x, W, a, indices, att)
    aux_out = None
    if aux is not None:
        if not isinstance(aux, (list, tuple)):
            aux = [aux]
        aux_out = [pair_logits(x, W, a, q, att) for q in aux]
    alpha = sp_softmax(indices, torch.sigmoid(edge_e), n)
    if keep is None:
        alpha = F.dropout(alpha, dropout, training=training)
    else:
        alpha = alpha * keep.to(alpha.dtype)
    if gnn == "AT":
        h = sp_matmul(indices, alpha, x @ p[prefix + "W_em"])
    elif gnn == "GCN":
        # layers.py:38-54: A (x W) + b, A's values are alpha (after coalesce: same order)
        h = sp_matmul(indices, alpha, x @ p[prefix + "ag_layer.weight"]) + p[prefix + "ag_layer.bias"]
    elif gnn == "SAGE":
        # layers.py:96-110: divisor = detached dense row sum of alpha, +1
        div = torch.zeros(n, 1, dtype=x.dtype)
        div.scatter_add_(0, indices[0].unsqueeze(1), alpha.detach())
        neigh = sp_matmul(indices, alpha, x) / (div + 1)
        h = torch.cat([x, neigh], dim=-1) @ p[prefix + "ag_layer.proj.weight"].t()
    else:
        raise ValueError(gnn)
    out = F.elu(h)
    if aux_out is not None:
        return out, edge_e, aux_out
    return out, edge_e


def fuse_layer(fp, feats, residue=None, residue_type=0, residue_dim=0, no_relu=False):
    """FuseLayer.forward, layers.py:896-921.  fp = {'fuse.weight', 'fuse.bias'[, 'fuse2.*']}."""
    z = torch.cat(feats, dim=-1)
    use_res = residue_dim != 0 and residue is not None
    if residue_type == 0:
        if use_res:
            z = torch.cat([z, residue], dim=-1)
        z = F.linear(z, fp["fuse.weight"], fp["fuse.bias"])
    elif residue_type == 1:
        if use_res:
            z = torch.cat([z, residue], dim=-1)
        z = F.leaky_relu(F.linear(z, fp["fuse.weight"], fp["fuse.bias"]))
        z = F.linear(z, fp["fuse2.weight"], fp["fuse2.bias"])
    elif residue_type == 2:
        z = F.linear(z, fp["fuse.weight"], fp["fuse.bias"])
        if use_res:
            z = z + F.linear(residue, fp["fuse2.weight"], fp["fuse2.bias"])
    return z if no_relu else F.leaky_relu(z)


# --------------------------------------------------------------------------- traversal
def disgat_traverse(p, fusers, x, indices, nheads, att, gnn, dropout=0.0, training=False,
                    aux=None, residue=False, residue_type=0, no_relu=False):
    """The shared 2-layer x C-channel traversal of DISGAT (models.py:181-373).

    Returns a dict with what the five reference methods return:
      'feats'   -> get_em            [feature_1, feature_2]          (models.py:217-252)
      'logp'    -> forward           log_softmax(fuser2 output)      (models.py:181-214)
      'edge_e'  -> get_adjs          [[e_c]_c]_layer                  (models.py:254-288)
      'aux'     -> predict_adjs_sparse [[aux_c]_c]_layer (if aux)    (models.py:290-330)
      'edge_em' -> get_edge_em       [[cat(x_in, elu(h'_c))]_c]_layer (models.py:333-373)
    """
    res = {"edge_e": [], "aux": [], "edge_em": []}
    x_in = F.dropout(x, dropout, training=training)
    feats = []
    for layer in (1, 2):
        outs, es, auxs, ems = [], [], [], []
        for c in range(nheads):
            r = disga_layer(p, "attention%d_%d." % (layer, c), x_in, indices, att, gnn,
                            dropout, training, aux)
            outs.append(r[0])
            es.append(r[1])
            if aux is not None:
                auxs.append(r[2])
            ems.append(torch.cat((x_in, r[0]), dim=-1))
        res["edge_e"].append(es)
        res["aux"].append(auxs)
        res["edge_em"].append(ems)
        fdim = x_in.size(1) if residue else 0
        fused = fuse_layer(fusers[layer - 1], outs, x_in, residue_type, fdim, no_relu)
        if layer == 2:
            res["logp"] = F.log_softmax(fused, dim=1)
        x_in = F.dropout(fused, dropout, training=training)
        feats.append(x_in)
    res["feats"] = feats
    return res


# --------------------------------------------------------------------------- losses
def adj_mse_loss(pred, tgt):
    """Class-balanced MSE.  Follows utils.py:287-298 incl. the `shape[0]**2` total."""
    n_pos = int((tgt != 0).sum())
    total = tgt.shape[0] ** 2
    w_neg = n_pos / (total - n_pos)
    w = torch.ones_like(tgt)
    w[tgt == 0] = w_neg
    return torch.mean(w * (pred - tgt) ** 2)


def mlp(mp, z, cls=False):
    """models.MLP with layers=2 (models.py:523-543): Linear -> LeakyReLU(0.1) -> Linear."""
    z = F.leaky_relu(F.linear(z, mp["model.0.weight"], mp["model.0.bias"]), 0.1)
    z = F.linear(z, mp["model.2.weight"], mp["model.2.bias"])
    return F.log_softmax(z, dim=1) if cls else z


def supedge_loss(aux_by_layer, labels, constrain_layer=0):
    """SupEdgeTrainer.train_step loss, pretrainer.py:726-747 (sparse branch)."""
    loss = None
    for layer, per_head in enumerate(aux_by_layer):
        if constrain_layer == 0 or constrain_layer == layer:
            pred = torch.sigmoid(torch.stack([h[0] for h in per_head]).sum(0))
            term = adj_mse_loss(pred.squeeze(), labels)
            loss = term if loss is None else loss + term
    return loss


def disedge_loss(aux_by_layer, labels2, constrain_layer=0):
    """GeneratedEdgeTrainer.train_step loss, pretrainer.py:596-627 (sparse branch)."""
    loss = None
    for layer, per_head in enumerate(aux_by_layer):
        if constrain_layer == 0 or constrain_layer == layer:
            c = len(per_head)
            homo = torch.sigmoid(torch.stack([h[0] for h in per_head][: int(c / 2)]).sum(0))
            het = torch.sigmoid(torch.stack([h[1] for h in per_head][int(c / 2):]).sum(0))
            term = adj_mse_loss(homo.squeeze(), labels2[0]) + adj_mse_loss(het.squeeze(), labels2[1])
            loss = term if loss is None else loss + term
    return loss


def difhead_loss(edge_em_by_layer, classifiers):
    """DifHeadTrainer.train_step loss, pretrainer.py:819-832: NLL(label == channel id)."""
    loss = None
    for layer, per_head in enumerate(edge_em_by_layer):
        mp = classifiers[0] if layer == 0 else classifiers[1]
        for c, em in enumerate(per_head):
            lab = torch.full((em.shape[0],), c, dtype=torch.long)
            term = F.nll_loss(mlp(mp, em, cls=True), lab)
            loss = term if loss is None else loss + term
    return loss
