"""torch.autograd.Function wrappers over the C ABI (include/edis.h).

PyTorch is plumbing here: it owns device memory, streams and the dense GEMMs; every sparse /
segment / reduction step runs in libedis.so on the caller's current CUDA stream.
"""
import ctypes

import torch

from . import _lib
from ._lib import LayerDesc, check, lib


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _off(t, col):
    """Device pointer of column `col` of a 2-D fp32 tensor."""
    return ctypes.c_void_p(t.data_ptr() + 4 * int(col))


def _rows(t, what):
    """(tensor, leading stride) of a 2-D fp32 CUDA tensor with unit inner stride."""
    if t.dtype != torch.float32 or not t.is_cuda:
        raise _lib.EdisError("%s must be a float32 CUDA tensor (got %s on %s)" % (what, t.dtype, t.device))
    if t.dim() != 2 or t.stride(1) != 1:
        t = t.contiguous()
    return t, t.stride(0)


class KernelTimer:
    """Optional per-call CUDA-event timing + launch counting (bench.py switches it on).

    Events are recorded on the stream the kernels are launched on; durations are read after
    the caller synchronises.  Off by default: zero overhead on the product path."""

    def __init__(self):
        self.enabled = False
        self.records = {}     # name -> list of (start_event, end_event, bytes dict)
        self.launches = 0

    def reset(self):
        self.records = {}
        self.launches = 0

    def durations_ms(self):
        return {k: [a.elapsed_time(b) for a, b, _ in v] for k, v in self.records.items()}

    def bytes(self):
        return {k: [m for _, _, m in v] for k, v in self.records.items()}


TIMER = KernelTimer()


def kernel_bytes(kind, n, nc, e, att, C, D, Fin=None, sage=False):
    """Bytes of one layer kernel launch, fp32: {"alg": ..., "moved": ...}.

    alg   = SURVEY 8(d)'s gather model of the REFERENCE's layer (every gathered row is DRAM traffic):
            fwd E(score + agg + 4C + 4) + 8CD N; bwd split as dst pass E(score + agg + 4C + 4) + 8CD N
            and src pass E(score + agg) + 4CD N, with score = 4CD (att 2/3) or 4C (att 1) and
            agg = 4CD (gnn AT / GCN, whatever plan executes it) or 4F (SAGE).
    moved = what THIS implementation has to move if nothing hits in L2 (att-3 sign record instead of
            re-gathering Q_j / P_i in the backward; F floats instead of C*D for a shared operand)."""
    CD = C * D
    score = 4 * C if att == 1 else 4 * CD
    agg_ref = 4 * Fin if sage else 4 * CD                 # the reference layer's aggregated operand
    agg_own = 4 * CD if Fin is None else 4 * Fin          # what this kernel gathers per edge
    wout = CD if Fin is None else C * Fin                 # node-tensor width of the aggregate
    sign = CD // 8 if att == 3 else 0
    if kind == "fwd":
        alg = e * (score + agg_ref + 4 * C + 4) + 8 * CD * n
        moved = e * (score + agg_own + 4 * C + sign + 4) + n * (score + 4 * wout * (1 if Fin else 2) + 8 * C)
    elif kind == "bwd_dst":
        alg = e * (score + agg_ref + 4 * C + 4) + 8 * CD * n
        moved = (e * ((score if att == 2 else 0) + agg_own + 4 * C + 8 * C + sign + 4)
                 + n * (12 * wout + 2 * score + 8 * C))
    elif kind == "bwd_src":
        alg = e * (score + agg_ref) + 4 * CD * n
        moved = (e * ((score if att == 2 else 0) + 4 * wout + 8 * C + sign + 8)
                 + nc * (score + (4 * CD if Fin is None else 4 * Fin)))
    elif kind == "bwd_src_score":                         # lane-strided shared operand: score side only
        alg = e * score + 4 * CD * n
        moved = e * ((score if att == 2 else 0) + 8 * C + sign + 8) + nc * score
    else:                                                 # "bwd_gx": separate dX kernel of that path
        alg = e * agg_ref
        moved = e * (4 * wout + 4 * C + 8) + nc * 4 * Fin
    return {"alg": int(alg), "moved": int(moved)}


class _timed:
    def __init__(self, name, graph, launches, nbytes=None):
        self.name, self.launches, self.nbytes = name, launches, nbytes

    def __enter__(self):
        if TIMER.enabled:
            self.start = torch.cuda.Event(enable_timing=True)
            self.end = torch.cuda.Event(enable_timing=True)
            self.start.record(torch.cuda.current_stream())
        return self

    def __exit__(self, *exc):
        if TIMER.enabled:
            self.end.record(torch.cuda.current_stream())
            TIMER.records.setdefault(self.name, []).append((self.start, self.end, self.nbytes))
            TIMER.launches += self.launches
        return False


def phase(name):
    """Time a host-orchestrated phase (GEMMs, exposed collective waits) with CUDA events on the current
    stream when bench.py has switched the timer on; counts no launches and carries no byte model."""
    return _timed("phase:" + name, None, 0, None)


def _desc(att, C, D, training=False, p=0.0, seed=0):
    return LayerDesc(att=att, C=C, D=D, Dv=D, training=1 if (training and p > 0) else 0, p=float(p),
                     seed=int(seed) & 0xFFFFFFFFFFFFFFFF)


def _edge_rec(graph, d, device):
    nbytes = check(lib.edis_disga_rec_bytes(graph.handle, ctypes.byref(d)), "edis_disga_rec_bytes")
    return torch.empty(int(nbytes), dtype=torch.uint8, device=device)


def _sign_rec(graph, d, device, wanted):
    """att 3: the forward's 1-bit-per-element record of sign(P_i + Q_j), kept for the backward."""
    if d.att != 3 or not wanted:
        return None
    nbytes = check(lib.edis_disga_sign_bytes(graph.handle, ctypes.byref(d)), "edis_disga_sign_bytes")
    return torch.empty(int(nbytes), dtype=torch.uint8, device=device)


def _workspace(graph, width, like):
    nbytes = graph.workspace_bytes(width)
    return torch.empty(nbytes, dtype=torch.uint8, device=like.device), nbytes


def disga_forward_raw(graph, d, P, ldp, Q, ldq, V, ldv, a, bias, device, want_sign):
    """One edis_disga_fwd launch on raw operands (ctypes pointers + row strides).  Allocates and
    returns (out, hpre, edge_e, stats, esign).  Shared by DisGAFused and parallel.PartitionedLayer."""
    C, D = d.C, d.D
    CD = C * D
    n, e = graph.n, graph.e
    out = torch.empty(n, CD, dtype=torch.float32, device=device)
    hpre = torch.empty_like(out)
    edge_e = torch.empty(e, C, dtype=torch.float32, device=device)
    stats = torch.empty(n, 2 * C, dtype=torch.float32, device=device)
    ws, nbytes = _workspace(graph, CD + 2 * C, out)
    esign = _sign_rec(graph, d, device, want_sign)
    with _timed("disga_fwd", graph, 1 + (1 if graph.info["dst_slots"] else 0),
                kernel_bytes("fwd", n, graph.n_cols, e, d.att, C, D)):
        check(lib.edis_disga_fwd(graph.handle, ctypes.byref(d), P, ldp, Q, ldq, _ptr(a), V, ldv, _ptr(bias),
                                 _ptr(out), _ptr(hpre), _ptr(edge_e), _ptr(stats), _ptr(esign), _ptr(ws), nbytes,
                                 _stream()), "edis_disga_fwd")
    return out, hpre, edge_e, stats, esign


def disga_backward_raw(graph, d, P, ldp, Q, ldq, V, ldv, a, bias, hpre, edge_e, stats, esign, g_out, g_edge_e,
                       gP, ldgp, gQ, ldgq, ga, gV, ldgv, device):
    """edis_disga_bwd_dst + edis_disga_bwd_src on raw operands; the caller owns gP / gQ / gV / ga.
    Returns gh[n, C*D] (gradient wrt the pre-ELU aggregate; its column sum is the bias gradient)."""
    C, D, att = d.C, d.D, d.att
    CD = C * D
    n, e, nc = graph.n, graph.e, graph.n_cols
    edge_rec = _edge_rec(graph, d, device)
    gh = torch.empty(n, CD, dtype=torch.float32, device=device)
    ws, nbytes = _workspace(graph, 2 * CD + 2 * C, gh)
    args = (graph.handle, ctypes.byref(d), P, ldp, Q, ldq, _ptr(a), V, ldv, _ptr(bias),
            _ptr(hpre), _ptr(edge_e), _ptr(stats), _ptr(esign), _ptr(g_out), _ptr(g_edge_e), gP, ldgp, gQ, ldgq,
            _ptr(ga), gV, ldgv, _ptr(edge_rec), _ptr(gh), _ptr(ws), nbytes, _stream())
    with _timed("disga_bwd_dst", graph, 1 + (1 if graph.info["dst_slots"] else 0),
                kernel_bytes("bwd_dst", n, nc, e, att, C, D)):
        check(lib.edis_disga_bwd_dst(*args), "edis_disga_bwd_dst")
    with _timed("disga_bwd_src", graph, 1 + (2 if graph.info["src_slots"] else 0),
                kernel_bytes("bwd_src", n, nc, e, att, C, D)):
        check(lib.edis_disga_bwd_src(*args), "edis_disga_bwd_src")
    return gh


class DisGAFused(torch.autograd.Function):
    """All C channels of one DisGALayer: scoring -> sigmoid -> segment softmax -> dropout ->
    aggregation -> (+bias) -> ELU.  Replaces layers.py:349-416 + 500/509 per channel.

    forward(graph, att, C, D, proj, off_p, off_q, off_v, sdst, ssrc, a, bias, training, p, seed)
        -> (out[N, C*D], edge_e[E, C])
    `proj` is the output of the layer's single projection GEMM, [N, W]; the operands are column
    blocks of it (no copies): V = proj[:, off_v:off_v+C*D] and, for att 2/3,
    P = proj[:, off_p:...], Q = proj[:, off_q:...] (att 2: off_p == off_q).  For att 1 the
    per-node scalars sdst/ssrc [N, C] are passed instead.  The backward writes gP/gQ/gV
    straight into one [N, W] gradient buffer for the GEMM's backward.
    """

    @staticmethod
    def forward(ctx, graph, att, C, D, proj, off_p, off_q, off_v, sdst, ssrc, a, bias, training, p, seed):
        proj, ld = _rows(proj, "proj")
        if att == 1:
            sdst, ssrc = sdst.contiguous(), ssrc.contiguous()
            P, Q, ldp, ldq = _ptr(sdst), _ptr(ssrc), C, C
        else:
            P, Q, ldp, ldq = _off(proj, off_p), _off(proj, off_q), ld, ld
        a = a.contiguous() if a is not None else None
        bias = bias.contiguous() if bias is not None else None
        if proj.shape[0] != graph.n_cols:
            raise _lib.EdisError("projection has %d rows, graph has %d source nodes" % (proj.shape[0], graph.n_cols))
        d = _desc(att, C, D, training, p, seed)
        out, hpre, edge_e, stats, esign = disga_forward_raw(graph, d, P, ldp, Q, ldq, _off(proj, off_v), ld, a, bias,
                                                            proj.device, any(ctx.needs_input_grad))
        ctx.graph, ctx.d, ctx.offs = graph, d, (off_p, off_q, off_v)
        ctx.has_a, ctx.has_bias = a is not None, bias is not None
        ctx.save_for_backward(proj, sdst, ssrc, a, bias, hpre, edge_e, stats, esign)
        ctx.set_materialize_grads(False)
        return out, edge_e

    @staticmethod
    def backward(ctx, g_out, g_edge_e):
        proj, sdst, ssrc, a, bias, hpre, edge_e, stats, esign = ctx.saved_tensors
        graph, d = ctx.graph, ctx.d
        C, D, att = d.C, d.D, d.att
        CD = C * D
        n, e, nc = graph.n, graph.e, graph.n_cols
        rect = nc > n          # destination-range partition: rows >= n are halo sources only
        off_p, off_q, off_v = ctx.offs
        ld, W, dev = proj.stride(0), proj.shape[1], proj.device
        if g_out is None:
            g_out = torch.zeros(n, CD, dtype=torch.float32, device=dev)
        g_out = g_out.contiguous()
        if g_edge_e is not None:
            g_edge_e = g_edge_e.contiguous()
        g_sd = g_ss = gq_sep = None
        if att == 1:
            # the score columns of proj get their gradient through sdst/ssrc in torch
            g_proj = torch.zeros(nc, W, dtype=torch.float32, device=dev)
            g_sd = (torch.zeros if rect else torch.empty)(nc, C, dtype=torch.float32, device=dev)
            g_ss = torch.empty(nc, C, dtype=torch.float32, device=dev)
            P, Q, ldp, ldq = _ptr(sdst), _ptr(ssrc), C, C
            gP, gQ, ldgp, ldgq = _ptr(g_sd), _ptr(g_ss), C, C
        else:
            covered = CD * (3 if att == 3 else 2)
            g_proj = (torch.empty if W == covered and not rect else torch.zeros)(nc, W, dtype=torch.float32,
                                                                                 device=dev)
            P, Q, ldp, ldq = _off(proj, off_p), _off(proj, off_q), ld, ld
            gP, ldgp = _off(g_proj, off_p), W
            if off_q == off_p:      # att 2: P and Q are the same columns; sum the two grads
                gq_sep = torch.empty(nc, CD, dtype=torch.float32, device=dev)
                gQ, ldgq = _ptr(gq_sep), CD
            else:
                gQ, ldgq = _off(g_proj, off_q), W
        ga = torch.zeros(C, D, dtype=torch.float32, device=dev) if att == 3 else None
        gh = disga_backward_raw(graph, d, P, ldp, Q, ldq, _off(proj, off_v), ld, a, bias, hpre, edge_e, stats, esign,
                                g_out, g_edge_e, gP, ldgp, gQ, ldgq, ga, _off(g_proj, off_v), W, dev)
        if gq_sep is not None:
            g_proj[:, off_p:off_p + CD] += gq_sep
        gbias = gh.sum(0) if ctx.has_bias else None
        return (None, None, None, None, g_proj, None, None, None, g_sd, g_ss,
                ga if ctx.has_a else None, gbias, None, None, None)


def sage_forward_raw(graph, d, P, ldp, Q, ldq, X, a, want_sign):
    """One edis_disga_sage_fwd launch on raw score operands (ctypes pointers + row strides) and the shared
    operand X[n_cols, F] (tensor).  d.Dv / d.flags must be set.  -> (agg[n, C*F], edge_e, stats, esign)."""
    n, e, Fin, C = graph.n, graph.e, X.shape[1], d.C
    if X.shape[0] != graph.n_cols:
        raise _lib.EdisError("X has %d rows, graph has %d source nodes" % (X.shape[0], graph.n_cols))
    agg = torch.empty(n, C * Fin, dtype=torch.float32, device=X.device)
    edge_e = torch.empty(e, C, dtype=torch.float32, device=X.device)
    stats = torch.empty(n, 2 * C, dtype=torch.float32, device=X.device)
    ws, nbytes = _workspace(graph, C * Fin + 2 * C, X)
    esign = _sign_rec(graph, d, X.device, want_sign)
    plain = bool(d.flags & _lib.FLAG_PLAIN_MEAN)
    with _timed("disga_sage_fwd", graph, 1 + (1 if graph.info["dst_slots"] else 0),
                kernel_bytes("fwd", n, graph.n_cols, e, d.att, C, d.D, Fin, sage=not plain)):
        check(lib.edis_disga_sage_fwd(graph.handle, ctypes.byref(d), P, ldp, Q, ldq, _ptr(a), _ptr(X), X.stride(0),
                                      _ptr(agg), _ptr(edge_e), _ptr(stats), _ptr(esign), _ptr(ws), nbytes,
                                      _stream()),
              "edis_disga_sage_fwd")
    return agg, edge_e, stats, esign


def sage_backward_raw(graph, d, P, ldp, Q, ldq, X, a, agg, edge_e, stats, esign, g_agg, g_edge_e, gP, ldgp, gQ, ldgq,
                      ga, need_gx):
    """The passes of edis_disga_sage_bwd on raw operands; the caller owns gP / gQ / ga.  -> gX[n_cols, F] or None."""
    C, D, att, Fin = d.C, d.D, d.att, d.Dv
    CD = C * D
    n, e, nc = graph.n, graph.e, graph.n_cols
    dev = X.device
    gX = torch.empty(nc, Fin, dtype=torch.float32, device=dev) if need_gx else None
    edge_rec = _edge_rec(graph, d, dev)
    gh = torch.empty(n, C * Fin, dtype=torch.float32, device=dev)
    ws, nbytes = _workspace(graph, (2 * CD + 2 * C + Fin + 3) // 4 * 4, X)   # 16-byte aligned partial rows
    base = d.flags
    plain = bool(base & _lib.FLAG_PLAIN_MEAN)
    fused_gx = bool(lib.edis_disga_sage_fused_gx(ctypes.byref(d)))
    kb = lambda kind: kernel_bytes(kind, n, nc, e, att, C, D, Fin, sage=not plain)
    phases = [("disga_sage_bwd_dst", _lib.FLAG_PHASE_DST, 1 + (1 if graph.info["dst_slots"] else 0), kb("bwd_dst")),
              ("disga_sage_bwd_src", _lib.FLAG_PHASE_SRC, 1 + (1 if graph.info["src_slots"] else 0),
               kb("bwd_src" if (fused_gx and need_gx) else "bwd_src_score"))]
    if need_gx and not fused_gx:
        phases.append(("disga_sage_bwd_gx", _lib.FLAG_PHASE_GX, 1 + (1 if graph.info["src_slots"] else 0),
                       kb("bwd_gx")))
    for name, bit, nl, nb in phases:
        d.flags = base | bit
        with _timed(name, graph, nl, nb):
            check(lib.edis_disga_sage_bwd(graph.handle, ctypes.byref(d), P, ldp, Q, ldq, _ptr(a), _ptr(X),
                                          X.stride(0), _ptr(agg), _ptr(edge_e), _ptr(stats), _ptr(esign), _ptr(g_agg),
                                          _ptr(g_edge_e), gP, ldgp, gQ, ldgq, _ptr(ga), _ptr(gX),
                                          _ptr(edge_rec), _ptr(gh), _ptr(ws), nbytes, _stream()),
                  "edis_disga_sage_bwd")
    d.flags = base
    return gX


class SageFused(torch.autograd.Function):
    """Scoring -> softmax -> dropout -> aggregation of the RAW layer input x, shared by all channels.

    plain=False: gnn_type=SAGE neighbour mean, divided by the detached (row sum + 1); replaces
    layers.py:349-394 + 400-403 + SageConv.forward's aggregation (layers.py:96-103, incl. its N x N
    `to_dense()`).  plain=True: sum_j alpha_drop_ij x_j, i.e. gnn_type AT / GCN executed as
    aggregate-then-project ((sum_j a_ij x_j) W == sum_j a_ij (x_j W)): the per-edge gather of the
    aggregated operand shrinks from C*D to F floats; ChannelLinear applies W afterwards.

    forward(graph, att, C, D, proj, off_p, off_q, sdst, ssrc, a, X, training, p, seed, plain)
        -> (agg[N, C*F], edge_e[E, C]);   score operands as in DisGAFused.
    """

    @staticmethod
    def forward(ctx, graph, att, C, D, proj, off_p, off_q, sdst, ssrc, a, X, training, p, seed, plain):
        X, ldx = _rows(X, "X")
        if att == 1:
            sdst, ssrc = sdst.contiguous(), ssrc.contiguous()
            P, Q, ldp, ldq = _ptr(sdst), _ptr(ssrc), C, C
        else:
            proj, ld = _rows(proj, "proj")
            P, Q, ldp, ldq = _off(proj, off_p), _off(proj, off_q), ld, ld
        a = a.contiguous() if a is not None else None
        d = _desc(att, C, D, training, p, seed)
        d.Dv = X.shape[1]
        d.flags = (_lib.FLAG_PLAIN_MEAN if plain else 0) | (0 if ctx.needs_input_grad[10] else _lib.FLAG_NO_GX)
        agg, edge_e, stats, esign = sage_forward_raw(graph, d, P, ldp, Q, ldq, X, a, any(ctx.needs_input_grad))
        ctx.graph, ctx.d, ctx.offs, ctx.plain = graph, d, (off_p, off_q), bool(plain)
        ctx.has_a = a is not None
        ctx.save_for_backward(proj, sdst, ssrc, a, X, agg, edge_e, stats, esign)
        ctx.set_materialize_grads(False)
        return agg, edge_e

    @staticmethod
    def backward(ctx, g_agg, g_edge_e):
        proj, sdst, ssrc, a, X, agg, edge_e, stats, esign = ctx.saved_tensors
        graph, d = ctx.graph, ctx.d
        C, D, att = d.C, d.D, d.att
        CD = C * D
        n, nc = graph.n, graph.n_cols
        rect = nc > n
        off_p, off_q = ctx.offs
        dev = X.device
        if g_agg is None:
            g_agg = torch.zeros_like(agg)
        g_agg = g_agg.contiguous()
        if g_edge_e is not None:
            g_edge_e = g_edge_e.contiguous()
        g_proj = g_sd = g_ss = gq_sep = None
        if att == 1:
            g_sd = (torch.zeros if rect else torch.empty)(nc, C, dtype=torch.float32, device=dev)
            g_ss = torch.empty(nc, C, dtype=torch.float32, device=dev)
            P, Q, ldp, ldq = _ptr(sdst), _ptr(ssrc), C, C
            gP, gQ, ldgp, ldgq = _ptr(g_sd), _ptr(g_ss), C, C
        else:
            ld, W = proj.stride(0), proj.shape[1]
            covered = CD * (2 if att == 3 else 1)
            g_proj = (torch.empty if W == covered and not rect else torch.zeros)(nc, W, dtype=torch.float32,
                                                                                 device=dev)
            P, Q, ldp, ldq = _off(proj, off_p), _off(proj, off_q), ld, ld
            gP, ldgp = _off(g_proj, off_p), W
            if off_q == off_p:
                gq_sep = torch.empty(nc, CD, dtype=torch.float32, device=dev)
                gQ, ldgq = _ptr(gq_sep), CD
            else:
                gQ, ldgq = _off(g_proj, off_q), W
        need_gx = not (d.flags & _lib.FLAG_NO_GX)
        ga = torch.zeros(C, D, dtype=torch.float32, device=dev) if att == 3 else None
        gX = sage_backward_raw(graph, d, P, ldp, Q, ldq, X, a, agg, edge_e, stats, esign, g_agg, g_edge_e, gP, ldgp,
                               gQ, ldgq, ga, need_gx)
        if gq_sep is not None:
            g_proj[:, off_p:off_p + CD] += gq_sep
        return (None, None, None, None, g_proj, None, None, g_sd, g_ss, ga if ctx.has_a else None, gX,
                None, None, None, None)


# Node count from which the layer projection runs as 3xTF32 on the tensor cores instead of the fp32 SIMT
# GEMM.  3xTF32 carries ~2^-21 relative error (dropped xl*Wl term + the TF32 rounding of the low parts)
# against ~2^-24 sqrt(F) for fp32: forward values stay inside 1e-5, but WEIGHT GRADIENTS measured against a
# float64 evaluation move from < 2e-5 to 7e-5 on cora_full (tests/test_gpu_bundled.py) -- a logit's
# gradient is discontinuous at P_i + Q_j = 0 (leaky-relu kink), so a few more sign flips near zero show up
# there.  Below this size the GEMM is a negligible part of the step, so the exact one is used; above it
# (EDIS_PROJ3X=1 forces it on everywhere, =0 off) the projection would otherwise be 15 % of the step.
PROJ3X_MIN_ROWS = 65536


def use_proj3x(n_rows):
    import os
    mode = os.environ.get("EDIS_PROJ3X", "auto")
    return mode == "1" or (mode != "0" and n_rows >= PROJ3X_MIN_ROWS)


def _tf32_hi(t):
    """Round-to-nearest onto the TF32 grid (10 explicit mantissa bits), result still fp32."""
    return ((t.view(torch.int32) + 0x1000) & -0x2000).view(torch.float32)


def _xt_g(x, g, chunks=256):
    """x^T g for a very long reduction dimension (K = number of nodes): the node dimension is cut
    into `chunks` slabs reduced by one batched fp32 GEMM and the slab results are summed.  Faster
    than the single split-K GEMM cuBLAS picks for [F, N] x [N, W] (B200, N = 2.4M: 14.7 vs 18.4 ms at
    F = 100, W = 1536) and the two-level sum is also closer to the float64 result."""
    n = x.shape[0]
    if n < chunks * 1024:
        return x.t() @ g
    m = (n // chunks) * chunks
    out = torch.bmm(x[:m].view(chunks, m // chunks, -1).transpose(1, 2), g[:m].view(chunks, m // chunks, -1)).sum(0)
    if m < n:
        out += x[m:].t() @ g[m:]
    return out


class Proj3xTF32(torch.autograd.Function):
    """x @ W at fp32 accuracy on the tensor cores: x = xh + xl, W = Wh + Wl on the TF32 grid and
    x W ~= xh Wh + xh Wl + xl Wh = [xh | xh | xl] @ [Wh ; Wl ; Wh]  -- ONE library TF32 GEMM with
    3x the K (the dropped xl Wl term is ~2^-22 relative).  Used for the node projection of a layer
    (small K = F, wide output), where the fp32 SIMT GEMM is compute-bound and this one is bound by
    writing the output.  Backward stays plain fp32 (its big operand is the [N, W] gradient)."""

    @staticmethod
    def forward(ctx, x, w):
        xh, wh = _tf32_hi(x), _tf32_hi(w)
        xc = torch.cat([xh, xh, x - xh], 1)
        wc = torch.cat([wh, w - wh, wh], 0)
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        try:
            out = xc @ wc
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev
        ctx.save_for_backward(x, w)
        return out

    @staticmethod
    def backward(ctx, g):
        x, w = ctx.saved_tensors
        gx = g @ w.t() if ctx.needs_input_grad[0] else None
        gw = _xt_g(x, g) if ctx.needs_input_grad[1] else None
        return gx, gw


def _mm_3xtf32(x, w):
    """x @ w at fp32 accuracy on the tensor cores (see Proj3xTF32): for SMALL inner dimensions only --
    the operands are concatenated along K, and TF32 accumulation over very long K loses ~1e-3."""
    xh, wh = _tf32_hi(x), _tf32_hi(w)
    xc = torch.cat([xh, xh, x - xh], 1)
    wc = torch.cat([wh, w - wh, wh], 0)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        return xc @ wc
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


class NodeLinear(torch.autograd.Function):
    """F.linear(x, weight, bias) for a node tensor x[N, in] with N in the millions (FuseLayer,
    layers.py:896-921).  Forward = the library fp32 GEMM.  Backward: the input gradient
    g[N, out] @ weight[out, in] has a tiny inner dimension (out = nhid) and is bound by writing
    [N, in] -> 3xTF32 on the tensor cores; the weight gradient reduces over N -> slab-wise fp32."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return torch.nn.functional.linear(x, weight, bias)

    @staticmethod
    def backward(ctx, g):
        x, weight = ctx.saved_tensors
        g = g.contiguous()
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = _mm_3xtf32(g, weight) if weight.shape[0] <= 128 else g @ weight
        if ctx.needs_input_grad[1]:
            gw = _xt_g(g, x)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = g.sum(0)
        return gx, gw, gb


def node_linear(lin, x):
    """nn.Linear `lin` applied to a node tensor; the custom backward only where it pays."""
    if x.is_cuda and x.dim() == 2 and x.shape[0] >= 262144 and x.dtype == torch.float32:
        return NodeLinear.apply(x, lin.weight, lin.bias)
    return lin(x)


class ChannelLinear(torch.autograd.Function):
    """out[:, c*D:(c+1)*D] = agg[:, c*F:(c+1)*F] @ W[c]  for every channel c (plain cuBLAS GEMMs
    writing straight into column blocks: no [C, N, .] transposes).  agg [N, C*F], W [C, F, D]."""

    @staticmethod
    def forward(ctx, agg, W):
        C, Fin, D = W.shape
        out = torch.empty(agg.shape[0], C * D, dtype=agg.dtype, device=agg.device)
        for c in range(C):
            torch.mm(agg[:, c * Fin:(c + 1) * Fin], W[c], out=out[:, c * D:(c + 1) * D])
        ctx.save_for_backward(agg, W)
        return out

    @staticmethod
    def backward(ctx, g):
        agg, W = ctx.saved_tensors
        C, Fin, D = W.shape
        g = g.contiguous()
        g_agg = torch.empty_like(agg) if ctx.needs_input_grad[0] else None
        g_w = torch.empty_like(W) if ctx.needs_input_grad[1] else None
        for c in range(C):
            gc = g[:, c * D:(c + 1) * D]
            if g_agg is not None:
                torch.mm(gc, W[c].t(), out=g_agg[:, c * Fin:(c + 1) * Fin])
            if g_w is not None:
                torch.mm(agg[:, c * Fin:(c + 1) * Fin].t(), gc, out=g_w[c])
        return g_agg, g_w


class PairList:
    """One (i, j) pair set [2, M] (int64, CUDA) plus what the kernels derive from it once per
    set rather than once per layer: the column-sorted permutation the att-3 backward walks."""

    def __init__(self, pairs):
        self.pi, self.pj = pairs[0].contiguous(), pairs[1].contiguous()
        self._perm = None

    @staticmethod
    def wrap(p):
        return p if isinstance(p, PairList) else PairList(p)

    def col_perm(self):
        """Pair ids sorted by column j, int32 (one radix sort per sampled pair set)."""
        if self._perm is None:
            self._perm = torch.sort(self.pj.to(torch.int32))[1].to(torch.int32)
        return self._perm


class PairScore(torch.autograd.Function):
    """Raw attention logits of channels [c_lo, c_hi) on an arbitrary (i, j) pair list.
    Replaces layers.py:355-360 / 368-372 / 381-389.  Returns [M, c_hi - c_lo]."""

    @staticmethod
    def forward(ctx, att, C, D, pi, pj, c_lo, c_hi, P, Q, a, plist=None):
        P, ldp = _rows(P, "P")
        Q, ldq = _rows(Q, "Q")
        a = a.contiguous() if a is not None else None
        pi = pi.contiguous()
        pj = pj.contiguous()
        if pi.dtype != torch.int64 or pj.dtype != torch.int64 or not pi.is_cuda:
            raise _lib.EdisError("pair indices must be int64 CUDA tensors")
        m, n = pi.numel(), P.shape[0]
        out = torch.empty(m, c_hi - c_lo, dtype=torch.float32, device=P.device)
        d = _desc(att, C, D)
        psign = None
        if att == 3 and any(ctx.needs_input_grad) and 0 < m < 2 ** 31 and ldp % 4 == 0 and ldq % 4 == 0 \
                and P.data_ptr() % 16 == 0 and Q.data_ptr() % 16 == 0:
            nb = check(lib.edis_pair_sign_bytes(ctypes.byref(d), m, c_lo, c_hi), "edis_pair_sign_bytes")
            psign = torch.empty(int(nb), dtype=torch.uint8, device=P.device)
        with _timed("pair_fwd", None, 1):
            check(lib.edis_pair_score_fwd(ctypes.byref(d), n, m, _ptr(pi), _ptr(pj), c_lo, c_hi, _ptr(P), ldp,
                                          _ptr(Q), ldq, _ptr(a), _ptr(out), _ptr(psign), _stream()),
                  "edis_pair_score_fwd")
        ctx.d, ctx.rng, ctx.lds = d, (c_lo, c_hi), (ldp, ldq)
        ctx.has_a = a is not None
        ctx.plist = plist if plist is not None else (PairList(torch.stack([pi, pj])) if psign is not None else None)
        ctx.save_for_backward(pi, pj, P, Q, a, psign)
        return out

    @staticmethod
    def backward(ctx, g_out):
        pi, pj, P, Q, a, psign = ctx.saved_tensors
        d = ctx.d
        c_lo, c_hi = ctx.rng
        ldp, ldq = ctx.lds
        n, m = P.shape[0], pi.numel()
        wdt = d.C if d.att == 1 else d.C * d.D
        gP = torch.zeros(n, wdt, dtype=torch.float32, device=P.device)
        gQ = torch.zeros(Q.shape[0], wdt, dtype=torch.float32, device=P.device)   # P and Q may differ in rows
        ga = torch.zeros(d.C, d.D, dtype=torch.float32, device=P.device) if d.att == 3 else None
        g_out = g_out.contiguous()
        perm = ctx.plist.col_perm() if psign is not None else None
        with _timed("pair_bwd", None, 2 if psign is not None else 1):
            check(lib.edis_pair_score_bwd(ctypes.byref(d), n, m, _ptr(pi), _ptr(pj), c_lo, c_hi, _ptr(P), ldp,
                                          _ptr(Q), ldq, _ptr(a), _ptr(g_out), _ptr(psign), _ptr(perm), _ptr(gP),
                                          _ptr(gQ), _ptr(ga), _stream()), "edis_pair_score_bwd")
        return (None, None, None, None, None, None, None, gP, gQ, ga if ctx.has_a else None, None)


class SslWmse(torch.autograd.Function):
    """mean_k w_k (sigmoid(sum_c scores[k, c]) - target_k)^2 with the reference's class
    weights.  Replaces pretrainer.py:730-737 / 613-627 + utils.adj_mse_loss (utils.py:287-298)."""

    @staticmethod
    def forward(ctx, scores, target, n_pos, m_total=None):
        """m_total / n_pos: size and positive count of the whole pair set when `scores` is one
        rank's slice of it (parallel.ssl_pair_loss_partitioned); default m_total = len(scores)."""
        scores = scores.contiguous()
        target = target.contiguous()
        m, cs = scores.shape
        m_total = m if m_total is None else int(m_total)
        ctx.n_pos, ctx.m_total = int(n_pos), m_total
        if m == 0:
            # a rank whose slice of a partitioned pair set is empty contributes 0 (and must not raise while
            # its peers sit in the next collective)
            ctx.save_for_backward(scores, target)
            return scores.new_zeros(())
        loss = torch.empty(1, dtype=torch.float32, device=scores.device)
        ws = torch.empty(8, dtype=torch.uint8, device=scores.device)
        check(lib.edis_ssl_wmse_fwd(m, cs, _ptr(scores), _ptr(target), int(n_pos), m_total, _ptr(loss), _ptr(ws), 8,
                                    _stream()), "edis_ssl_wmse_fwd")
        ctx.n_pos, ctx.m_total = int(n_pos), m_total
        ctx.save_for_backward(scores, target)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g_loss):
        scores, target = ctx.saved_tensors
        m, cs = scores.shape
        if m == 0:
            return torch.zeros_like(scores), None, None, None
        g_scores = torch.empty_like(scores)
        g_loss = g_loss.reshape(1).contiguous().float()
        check(lib.edis_ssl_wmse_bwd(m, cs, _ptr(scores), _ptr(target), ctx.n_pos, ctx.m_total, _ptr(g_loss),
                                    _ptr(g_scores), _stream()), "edis_ssl_wmse_bwd")
        return g_scores, None, None, None


class NllConstLabel(torch.autograd.Function):
    """mean_i -log_softmax(logits[i])[label], one label for all rows (DifHead tail,
    pretrainer.py:825-832 + models.py:540-541)."""

    @staticmethod
    def forward(ctx, logits, label):
        logits = logits.contiguous()
        n, k = logits.shape
        loss = torch.empty(1, dtype=torch.float32, device=logits.device)
        ws = torch.empty(8, dtype=torch.uint8, device=logits.device)
        check(lib.edis_nll_const_label_fwd(n, k, _ptr(logits), int(label), _ptr(loss), _ptr(ws), 8, _stream()),
              "edis_nll_const_label_fwd")
        ctx.label = int(label)
        ctx.save_for_backward(logits)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g_loss):
        (logits,) = ctx.saved_tensors
        n, k = logits.shape
        g_logits = torch.empty_like(logits)
        g_loss = g_loss.reshape(1).contiguous().float()
        check(lib.edis_nll_const_label_bwd(n, k, _ptr(logits), ctx.label, _ptr(g_loss), _ptr(g_logits),
                                           _stream()), "edis_nll_const_label_bwd")
        return g_logits, None


class SpSoftmax(torch.autograd.Function):
    """utils.sp_softmax (utils.py:192-200) on a COO row index list."""

    @staticmethod
    def forward(ctx, row, values, n):
        shape = values.shape
        v = values.reshape(-1).contiguous()
        row = row.contiguous()
        out = torch.empty_like(v)
        denom = torch.empty(n, dtype=torch.float32, device=v.device)
        vmax = torch.empty(1, dtype=torch.float32, device=v.device)
        check(lib.edis_sp_softmax_fwd(n, v.numel(), _ptr(row), _ptr(v), _ptr(out), _ptr(denom), _ptr(vmax),
                                      _stream()), "edis_sp_softmax_fwd")
        ctx.n, ctx.shape = n, shape
        ctx.save_for_backward(row, out)
        return out.reshape(shape)

    @staticmethod
    def backward(ctx, g):
        row, out = ctx.saved_tensors
        g = g.reshape(-1).contiguous()
        gv = torch.empty_like(out)
        rowdot = torch.empty(ctx.n, dtype=torch.float32, device=out.device)
        check(lib.edis_sp_softmax_bwd(ctx.n, out.numel(), _ptr(row), _ptr(out), _ptr(g), _ptr(gv), _ptr(rowdot),
                                      _stream()), "edis_sp_softmax_bwd")
        return None, gv.reshape(ctx.shape), None


class SpMatmul(torch.autograd.Function):
    """utils.sp_matmul (utils.py:203-207) on COO (row, col) index lists."""

    @staticmethod
    def forward(ctx, row, col, values, mat):
        v = values.reshape(-1).contiguous()
        mat = mat.contiguous()
        row, col = row.contiguous(), col.contiguous()
        n, f = mat.shape
        out = torch.empty_like(mat)
        check(lib.edis_sp_matmul_fwd(n, v.numel(), f, _ptr(row), _ptr(col), _ptr(v), _ptr(mat), _ptr(out),
                                     _stream()), "edis_sp_matmul_fwd")
        ctx.vshape = values.shape
        ctx.save_for_backward(row, col, v, mat)
        return out

    @staticmethod
    def backward(ctx, g):
        row, col, v, mat = ctx.saved_tensors
        n, f = mat.shape
        g = g.contiguous()
        gv = torch.empty_like(v)
        gm = torch.empty_like(mat)
        check(lib.edis_sp_matmul_bwd(n, v.numel(), f, _ptr(row), _ptr(col), _ptr(v), _ptr(mat), _ptr(g),
                                     _ptr(gv), _ptr(gm), _stream()), "edis_sp_matmul_bwd")
        return None, None, gv.reshape(ctx.vshape), gm
