#!/usr/bin/env python
"""bench.py -- DISGAT fwd+bwd edges/s on B200 (the BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl edis|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = DISGAT.get_em forward + backward of a scalar loss, 2 layers x C channels, train
mode (dropout on), on the synthetic power-law graph of BASELINE config[3] (2.4M nodes, ~63M
edges, F=100, C=8, D=64, att=3, gnn_type=AT).  Prints ONE JSON line (rank 0).
  value      edges/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e        same through the public API with the features coming from pinned HOST memory
             every step (H2D inside the timed region) and the loss read back (D2H)
  roofline   the dominant kernel's algorithmic bytes / CUDA-event time vs the measured HBM peak
  breakdown  ms per step: sparse kernels / projection GEMMs / exposed exchange / the rest
  cpu_baseline  the UNMODIFIED reference (oracle/_ref) on a bounded sample of the workload, host cores
N > 1 (one rank per GPU, NCCL): by default STRONG scaling -- the SAME 63M-edge graph, destination rows
range-partitioned over the ranks (BASELINE config[3] "at 1/2/4/8 B200 with dst-partitioned CSR");
`--scaling weak` is the round-1 community workload (one 2.4M-node community per rank, a stated
`locality` fraction of edges inside it).  `--config B` = BASELINE config[4] (10M nodes / 500M edges).
`--impl reference` times the reference's own CPU path (rank 0 only, no GPU work, no libedis).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
DUMP_BYTES = 64_000_000
NPY_HEADER = 4096                                  # allowance per .npy file for its header


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="edis", choices=["edis", "reference"])
    ap.add_argument("--config", default="A", choices=["A", "B"], help="A = BASELINE config[3], B = config[4]")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--locality", type=float, default=0.9, help="weak scaling: fraction of edge draws inside a rank")
    ap.add_argument("--nodes", type=int, default=None)
    ap.add_argument("--raw-edges", type=int, default=None, help="directed draws before symmetrise/dedup")
    ap.add_argument("--feat", type=int, default=None)
    ap.add_argument("--nhead", type=int, default=8)
    ap.add_argument("--nhid", type=int, default=64)
    ap.add_argument("--att", type=int, default=3)
    ap.add_argument("--gnn_type", default="AT")
    ap.add_argument("--dropout", type=float, default=0.1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-budget-s", type=float, default=12.0, help="cpu_baseline leg: seconds per reference step")
    ap.add_argument("--ref-total-s", type=float, default=200.0, help="--impl reference: budget of the whole run")
    ap.add_argument("--cpu-probe-edges", type=int, default=250_000, help="CPU arm: edges of the calibration sample")
    ap.add_argument("--max-chunk", type=int, default=0)
    ap.add_argument("--no-epoch-metric", action="store_true", help="skip the cora_full epoch-ms secondary metric")
    ap.add_argument("--no-ssl-metric", action="store_true", help="skip the SupEdge step secondary metric")
    # no cache unless asked for: a run writes nothing into the (possibly read-only) source tree and leaves no
    # GB-sized graph files behind, and every run builds its graph with the code under test
    ap.add_argument("--cache-dir", default=os.environ.get("EDIS_CACHE_DIR", ""),
                    help="graph cache directory kept between runs (default: none; the graph is generated in every "
                         "run, by every rank at N > 1)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last of the --steps timed steps behind `value` computed to DIR/<name>.npy "
                         "(float32): "
                         "get_em's two embeddings at a fixed seeded sample of rows, the loss and every parameter "
                         "gradient, at most %d bytes in all" % DUMP_BYTES)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    base = {"A": (2_400_000, 30_600_000, 100), "B": (10_000_000, 246_000_000, 64)}[a.config]
    a.nodes = a.nodes or base[0]
    a.raw_edges = a.raw_edges or base[1]
    a.feat = a.feat or base[2]
    return a


def model_args(a):
    from edgedisentangle_ssl_b200.utils import get_parser
    args = get_parser().parse_args(["--model=DISGAT", "--sparse", "--att=%d" % a.att, "--gnn_type=" + a.gnn_type,
                                    "--nhead=%d" % a.nhead, "--nhid=%d" % a.nhid, "--dropout=%g" % a.dropout])
    args.size = a.feat
    return args


def workload_config(a, world, e_full=None, extra=None):
    name = {"A": "ogbn-products shape (BASELINE config[3])", "B": "10M nodes / 500M edges (BASELINE config[4])"}[a.config]
    if world > 1 and a.scaling == "weak":
        shape = ("WEAK scaling: %d communities of N=%d nodes / %d raw draws each (one per rank), locality=%.2f of the "
                 "draws inside the rank's community" % (world, a.nodes, a.raw_edges, a.locality))
    else:
        shape = "ONE graph N=%d, raw draws=%d%s" % (
            a.nodes, a.raw_edges, "" if world == 1 else ", destination rows range-partitioned over %d ranks (strong "
            "scaling, no planted locality%s)" % (world, "; generated block-wise per rank with uniform mixing between "
                                                 "the rank ranges" if a.config == "B" else ""))
    cfg = {"workload": "synthetic power-law graph, %s: %s, F=%d, C=%d, D=%d, att=%d, gnn_type=%s, full-batch "
                       "DISGAT.get_em fwd+bwd, train mode dropout=%g" % (name, shape, a.feat, a.nhead, a.nhid, a.att,
                                                                         a.gnn_type, a.dropout),
           "scaling": "n/a (1 GPU)" if world == 1 else a.scaling,
           "locality": (a.locality if (world > 1 and a.scaling == "weak") else None),
           "l2_policy": "inputs larger than L2 (node tensors are GBs; no flush needed)"}
    if e_full is not None:
        cfg["edges"] = int(e_full)
    if extra:
        cfg.update(extra)
    return cfg


# ---------------------------------------------------------------------------------- CPU arm
def cpu_reference_leg(a, step_budget_s, steps, warmup, threads):
    """The reference's own CPU path (oracle/_ref, unmodified; the oracle port only if that is absent) on a
    bounded power-law sample sized for ~`step_budget_s` seconds per step (oracle.ref_arm.sized_workload:
    E = 2M doubling, BASELINE.md section 4, or smaller when 2M does not fit the budget)."""
    from oracle import ref_arm
    wl, _ = ref_arm.sized_workload(a.feat, a.nhead, a.nhid, a.att, a.gnn_type, a.dropout, threads, step_budget_s,
                                   probe_edges=a.cpu_probe_edges)
    for _ in range(max(warmup, 1)):
        wl.step()
    times = [wl.step() for _ in range(max(steps, 1))]
    sec = float(np.mean(times))
    return {"value": wl.e / sec, "unit": "edges/s", "cores": threads, "kind": wl.kind,
            "sample": "%s, same F/C/D/att/gnn/dropout, %d timed steps of %.1f s (config A/B themselves do not fit the "
                      "reference: [E, 2F] temporaries and N x N samplers)" % (wl.describe(), len(times), sec)}, sec, wl


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    budget = max(1.0, a.ref_total_s / max(a.steps + max(a.warmup, 1) + 3, 1))
    cpu, sec, wl = cpu_reference_leg(a, budget, a.steps, a.warmup, threads)
    world = int(os.environ.get("WORLD_SIZE", str(a.gpus)))
    line = {
        "impl": "reference", "metric": "DISGAT fwd+bwd edges/s", "value": cpu["value"], "unit": "edges/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak" if world == 1 else a.scaling, "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(a, world),
        "same_config": False,
        "same_config_note": "same model / F / C / D / att / gnn / dropout and the same graph law; the graph is a bounded "
                            "sample (E in the line) because the reference cannot hold the full one -- its rate is per "
                            "edge, so the ratio compares edges/s, not wall time of equal work",
        "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------- cora_full epoch
def cora_full_epoch_ms():
    """BASELINE's second metric: one main.py epoch on bundled cora_full with the flags of
    example_bashs/Example_cora_full.sh:38 (5 CLS steps + SupEdge + DisEdge + DifHead, sampling and
    Adam included).  Median of epochs 2..4; three settings."""
    import contextlib
    import io
    from edgedisentangle_ssl_b200.main import run
    argv = ["--seed=4", "--model=DISGAT", "--used_edge=1", "--finetune", "--downstream=CLS", "--down_weight=1.0",
            "--steps=5", "--nhead=4", "--dataset=cora_full", "--pretrain", "SupEdge", "DisEdge", "DifHead",
            "--pre_weight", "1", "1", "1", "--pre_edge", "1", "1", "1", "--sparse", "--att=3",
            "--constrain_layer=0", "--epochs=4", "--gnn_type=AT"]
    out = {}
    for name, env in (("reference_rng_sampler_sklearn", {"EDIS_SAMPLER": "exact", "EDIS_HOST_METRICS": "1"}),
                      ("reference_rng_sampler_device_metrics", {"EDIS_SAMPLER": "exact", "EDIS_HOST_METRICS": "device"}),
                      ("device_sampler_sklearn", {"EDIS_SAMPLER": "device", "EDIS_HOST_METRICS": "1"}),
                      ("device_sampler_device_metrics", {"EDIS_SAMPLER": "device", "EDIS_HOST_METRICS": "device"}),
                      ("device_sampler_no_metrics", {"EDIS_SAMPLER": "device", "EDIS_HOST_METRICS": "0"})):
        env = dict(env, EDIS_SYNTH_FEATURES="1")      # cora_full's feature blob is missing from the snapshot
        old = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            with contextlib.redirect_stdout(io.StringIO()):
                hist = run(argv, data_root=os.path.join(ROOT, "data"))
            out[name] = float(np.median([h["epoch_ms"] for h in hist[1:]]))
        finally:
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
    out["note"] = ("rows: SSL pair sampler (exact = the reference's CPU RNG stream replayed bit for bit, O(N^2) "
                   "MT19937 outputs per draw, edis_rand_hits_host; device = same law in O(M) on the GPU) x validation "
                   "AUC / macro-F1 per CLS step (sklearn on host copies like the reference / computed on the device / "
                   "dropped).  reference_rng_sampler_device_metrics is the package default at this size.  "
                   "cora_full N=19793 E=146635, synthetic 64-d features (the feature blob is missing from the "
                   "reference snapshot); epoch 1 (graph build, warm-up) excluded; the reference's CPU path "
                   "took ~49 s per epoch in the survey probe (BASELINE.md)")
    return out


def supedge_step(margs, enc, graph, x_dev, steps=2):
    """BASELINE config[3] names "full-batch DISGAT + SSL losses": one SupEdgeTrainer.train_step on the
    same synthetic graph (device sampler: ~3.33 E pairs; pair scoring on both layers; fused weighted
    MSE; backward; Adam), CUDA events around the whole step incl. sampling."""
    import contextlib
    import io
    from edgedisentangle_ssl_b200 import trainer as T
    margs.cuda = True
    old = os.environ.get("EDIS_SAMPLER")
    os.environ["EDIS_SAMPLER"] = "device"
    try:
        tr = T.SupEdgeTrainer(margs, enc, 1.0)
        lab = tr.get_label_all(x_dev, graph)
        with contextlib.redirect_stdout(io.StringIO()):
            tr.train_step([x_dev, graph], lab)                      # warm-up
            m = int(tr.sample_train(lab)[1][0].shape[1])
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(steps):
                log = tr.train_step([x_dev, graph], lab)
            ev1.record()
            torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / steps
        return {"ms_per_step": ms, "pairs": m, "pairs_per_s": m / (ms * 1e-3), "edges_per_s": graph.e / (ms * 1e-3),
                "loss": float(log["loss_heads_sup"]), "steps": steps,
                "note": "SupEdgeTrainer.train_step on the bench graph: O(M) device sampler + pair scoring "
                        "(2 layers x %d channels) + edis_ssl_wmse + backward + Adam" % margs.nhead}
    except Exception as exc:                                       # secondary metric: never lose the headline
        return {"error": "%s: %s" % (type(exc).__name__, exc)}
    finally:
        if old is None:
            os.environ.pop("EDIS_SAMPLER", None)
        else:
            os.environ["EDIS_SAMPLER"] = old


def supedge_step_partitioned(a, enc, fus, part, x_dev, params, steps=2):
    """The same SupEdge step over the destination-range partition (pretrainer.py:683-763 per rank: pairs
    sampled in the rank's rows, columns scored against the all-gathered layer input, losses normalised by
    the GLOBAL counts, gradients all-reduced, Adam)."""
    import torch.distributed as dist
    from edgedisentangle_ssl_b200 import parallel as par
    try:
        dev = x_dev.device
        ex = part.graph.export()
        rows = np.repeat(np.arange(part.n_local, dtype=np.int64), np.diff(ex["rowptr"])) + part.lo
        src_ids = np.concatenate([np.arange(part.lo, part.hi, dtype=np.int64), part.halo_ids])
        pos_key = torch.from_numpy(rows * part.n_total + src_ids[ex["col"].astype(np.int64)]).to(dev)
        pos_key = torch.sort(pos_key)[0]
        opt = torch.optim.Adam(params, lr=1e-3)
        gen = torch.Generator(device=dev).manual_seed(7 + part.rank)

        def one():
            pairs, lab, n_pos, m_tot = par.sample_pairs_partitioned(part, pos_key, gen)
            loss = par.ssl_pair_loss_partitioned(enc, fus, x_dev, part, [pairs], [lab], [(0, a.nhead)], [n_pos], [m_tot])
            opt.zero_grad(set_to_none=True)
            loss.backward()
            par.allreduce_grads(params)
            opt.step()
            return loss.detach(), m_tot
        one()
        dist.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            loss, m_tot = one()
        ev1.record()
        dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([ev0.elapsed_time(ev1) / steps, float(loss)], device=dev, dtype=torch.float64)
        tm = t.clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(t)
        return {"ms_per_step": float(tm[0]), "pairs": int(m_tot), "pairs_per_s": m_tot / (float(tm[0]) * 1e-3),
                "loss": float(t[1]), "steps": steps,
                "note": "SupEdge step over the partition: per-rank O(M) sampler, pair scoring vs the all-gathered "
                        "layer input, edis_ssl_wmse with global counts, backward, grad all-reduce, Adam; max over ranks"}
    except Exception as exc:
        return {"error": "%s: %s" % (type(exc).__name__, exc)}


# ---------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------- workload
def _gen_key(a):
    """64-bit key of the generator's parameters: names a cached graph without generating it."""
    s = "power_law_graph v1 n=%d m=%d seed=0 max_chunk=%d" % (a.nodes, a.raw_edges, a.max_chunk)
    return int.from_bytes(hashlib.blake2b(s.encode(), digest_size=8).digest(), "little")


def global_graph_indices(a, rank, world, dev="cuda"):
    """[2, E] processed adjacency of the ONE bench graph.  With a cache directory it is generated once per box
    (rank 0) and shared with the other ranks / later runs as a memory-mapped .npy; without one (or when it cannot
    be written) every rank generates it from the same seed.
    Every decision that changes which collectives run is taken by rank 0 and broadcast, so ranks that
    arrive at different times cannot take different branches."""
    from edgedisentangle_ssl_b200.synthetic import power_law_graph
    path = os.path.join(a.cache_dir, "coo_%016x.npy" % _gen_key(a)) if a.cache_dir else None

    def agree(value):
        if world == 1:
            return value
        import torch.distributed as dist
        flag = torch.tensor([1 if value else 0], device=dev)
        dist.broadcast(flag, 0)
        return bool(int(flag.item()))

    if agree(bool(path) and os.path.exists(path)):
        return np.load(path, mmap_mode="r"), True
    idx = None
    saved = False
    if rank == 0:
        idx = power_law_graph(a.nodes, a.raw_edges, seed=0)
        if path:
            try:                                   # the cache is an optimisation: a read-only tree must not fail the run
                os.makedirs(a.cache_dir, exist_ok=True)
                tmp = path + ".tmp%d.npy" % os.getpid()
                np.save(tmp, idx)
                os.replace(tmp, path)
                saved = True
            except OSError:
                saved = False
    saved = agree(saved)                           # also the point where the other ranks wait for rank 0
    if idx is None:
        idx = np.load(path, mmap_mode="r") if saved else power_law_graph(a.nodes, a.raw_edges, seed=0)
    return idx, False


def dump_row_bytes(grad_numels, n_feats):
    """Bytes --dump-outputs has left for embedding rows next to the loss, the gradients and every file's header."""
    return DUMP_BYTES - 4 - 4 * sum(grad_numels) - (1 + len(grad_numels) + n_feats) * NPY_HEADER


def dump_outputs(out_dir, last, n_total, lo):
    """--dump-outputs: what the last timed step returned to its caller, as float32 .npy files.  The rows of
    get_em's two [N, D] embeddings are a sample drawn with a fixed seed over the global row ids, as many as fit
    DUMP_BYTES next to the loss and the gradients, so runs with the same arguments write the same rows; with
    several ranks, rank 0 writes the sampled rows of its own range."""
    arrays = {"loss": last["loss"].reshape(1)}
    arrays.update(("grad." + name, g) for name, g in last["grads"])
    feats = last["feats"]
    room = dump_row_bytes([g.numel() for _, g in last["grads"]], len(feats))
    k = min(n_total, room // (4 * sum(f.shape[1] for f in feats)))      # >= 1: checked in main() before timing
    rows =np.sort(np.random.RandomState(0).choice(n_total, k, replace=False))
    rows = rows[(rows >= lo) & (rows < lo + feats[0].shape[0])] - lo
    idx = torch.from_numpy(rows).to(feats[0].device)
    for i, f in enumerate(feats):
        arrays["get_em_%d" % i] = f[idx]
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), v.detach().float().cpu().numpy())


def main():
    a = parse()
    if a.impl == "reference":
        return run_reference_arm(a)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.gpus > 1 and world == 1:
        # launched without torchrun: start one rank per GPU ourselves
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(a.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29511"] + sys.argv
        raise SystemExit(subprocess.call(cmd))

    import torch.distributed as dist
    import edgedisentangle_ssl_b200 as edis
    from edgedisentangle_ssl_b200 import functional as Fn

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the edis arm has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    par = part = None
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=600))
        from edgedisentangle_ssl_b200 import parallel as par

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- workload ---------------------------------------------------------------------------
    t0 = time.time()
    cache_hit = False
    strong = world == 1 or a.scaling == "strong"
    if world == 1:
        gpath = os.path.join(a.cache_dir, "graph_%016x.edisg" % _gen_key(a)) if a.cache_dir else None
        graph = edis.Graph.load(gpath, _gen_key(a), dev, a.max_chunk) if gpath else None
        cache_hit = graph is not None
        if graph is None:
            idx, _ = global_graph_indices(a, 0, 1, dev)
            graph = edis.Graph(a.nodes, idx[0], idx[1], device=dev, max_chunk=a.max_chunk)
            if gpath:
                try:
                    graph.save(gpath, _gen_key(a))
                except Exception:                  # read-only tree: run without the cache
                    pass
            del idx
        n_local, n_total, e_local, lo = a.nodes, a.nodes, graph.e, 0
    elif strong and a.config == "B":
        # config[4] (10M nodes / 500M edges) does not fit one host process per rank as ONE generated edge
        # list; every rank generates only the blocks of the global graph its rows touch (same seeds on both
        # ends of a block), with UNIFORM mixing between the rank ranges: locality = 1 / world, i.e. no planted
        # locality -- a node's neighbours are spread over all ranks
        # (the block generator counts an in-range draw as two directed edges and a cross-range draw as one per
        # rank: uniform mixing with 2 * raw + N directed edges in total <=> these two arguments)
        n_total = a.nodes
        part = par.build_partitioned_power_law(n_total, a.raw_edges * (2 * world - 1) // world, seed=0, rank=rank,
                                                world=world, device=dev, locality=1.0 / (2 * world - 1),
                                                max_chunk=a.max_chunk)
        graph, n_local, e_local, lo = part.graph, part.n_local, part.graph.e, part.lo
    elif strong:
        n_total = a.nodes
        idx, cache_hit = global_graph_indices(a, rank, world, dev)
        part = par.partition_of_global_graph(idx, n_total, rank, world, device=dev, max_chunk=a.max_chunk)
        del idx
        graph, n_local, e_local, lo = part.graph, part.n_local, part.graph.e, part.lo
    else:
        n_total = a.nodes * world
        part = par.build_partitioned_power_law(n_total, a.raw_edges * world, seed=0, rank=rank, world=world,
                                                device=dev, locality=a.locality, max_chunk=a.max_chunk)
        graph, n_local, e_local, lo = part.graph, part.n_local, part.graph.e, part.lo
    setup_s = time.time() - t0

    margs = model_args(a)
    torch.manual_seed(4)
    enc = edis.DISGAT(margs, nfeat=a.feat, nhid=a.nhid, nclass=a.nhid, nheads=a.nhead, dropout=a.dropout).to(dev)
    fus = [edis.FuseLayer(margs, a.nhead, nfeat=a.nhid).to(dev), edis.FuseLayer(margs, a.nhead, nfeat=a.nhid).to(dev)]
    enc.train()
    named = [("encoder." + n, p) for n, p in enc.named_parameters()] + \
        [("fuser%d.%s" % (i, n), p) for i, f in enumerate(fus) for n, p in f.named_parameters()]
    params = [p for _, p in named]
    # every rank decides this the same way before any timing, so no rank is left waiting at a collective
    if a.dump_outputs and dump_row_bytes([p.numel() for p in params], 2) < 4 * 2 * a.nhid:
        raise SystemExit("--dump-outputs: the gradients alone exceed %d bytes" % DUMP_BYTES)
    # features / loss weights: rows [lo, lo + n_local) of one global seeded stream per 64K-row block, so the
    # strong-scaling runs at every N work on the SAME node features
    def rows_of(width, seed):
        blk = 65536
        out = torch.empty(n_local, width)
        b0 = lo // blk
        pos = 0
        while pos < n_local:
            g = torch.Generator().manual_seed(seed * 1_000_003 + b0)
            chunk = torch.randn(blk, width, generator=g)
            s = (lo + pos) - b0 * blk
            take = min(blk - s, n_local - pos)
            out[pos:pos + take] = chunk[s:s + take]
            pos += take
            b0 += 1
        return out
    x_host = rows_of(a.feat, 1234).pin_memory()
    x_dev = x_host.to(dev)
    R = rows_of(a.nhid, 99).to(dev)
    # e2e: double-buffered input -- the H2D copy of step k+1 runs on a side stream under step k
    x_bufs = [x_dev, torch.empty_like(x_dev)]
    copy_stream = torch.cuda.Stream(device=dev)
    copied = [torch.cuda.Event(), torch.cuda.Event()]      # buffer b holds the next step's features
    consumed = [torch.cuda.Event(), torch.cuda.Event()]    # the step that read buffer b has finished
    state = {"k": 0}

    def enqueue_copy(b):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[b])
            x_bufs[b].copy_(x_host, non_blocking=True)
            copied[b].record(copy_stream)
    loss_host = torch.zeros(1).pin_memory()

    def step(from_host, keep=None):
        xin = x_dev
        if from_host:
            b = state["k"] % 2
            torch.cuda.current_stream().wait_event(copied[b])     # this step's features have landed
            enqueue_copy(1 - b)                                   # next step's copy overlaps this step
            xin = x_bufs[b]
        if world == 1:
            feats = enc.get_em(xin, graph, fus)
        else:
            feats = par.get_em_partitioned(enc, fus, xin, part)
        loss = (feats[-1] * R).sum()
        loss.backward()
        if world > 1:
            with Fn.phase("grad_allreduce"):
                par.allreduce_grads(params)
        if keep is not None:                       # references only: no copy, no sync inside the timed window
            keep.update(feats=[f.detach() for f in feats], loss=loss.detach(),
                        grads=[(n, p.grad) for n, p in named if p.grad is not None])
        if from_host:
            loss_host.copy_(loss.detach().reshape(1), non_blocking=True)
            consumed[state["k"] % 2].record(torch.cuda.current_stream())
            state["k"] += 1
        for p in params:
            p.grad = None
        return loss

    def timed(from_host, k, keep=None):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for i in range(k):
            step(from_host, keep if i == k - 1 else None)
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            tms = torch.tensor([ms], device=dev)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms = float(tms.item())
        return ms

    for _ in range(max(a.warmup, 3)):
        step(False)
    clocks = ClockSampler(local)
    clocks.start()
    Fn.TIMER.reset()
    Fn.TIMER.enabled = True
    last = {} if (a.dump_outputs and rank == 0) else None
    ms_res = timed(False, a.steps, last)
    Fn.TIMER.enabled = False
    kernel_list = Fn.TIMER.durations_ms()
    kernel_bytes = Fn.TIMER.bytes()
    plan = os.environ.get("EDIS_AT_PLAN") or "proj"
    launches = Fn.TIMER.launches
    for b in (0, 1):
        consumed[b].record(torch.cuda.current_stream())
    enqueue_copy(0)
    step(True)
    ms_e2e = timed(True, a.steps)
    clk = clocks.stop()
    if last:                                       # after the clock samples: they cover GPU work only
        dump_outputs(a.dump_outputs, last, n_total, lo)
        del last

    e_total = e_local
    if world > 1:
        te = torch.tensor([e_local], device=dev, dtype=torch.int64)
        dist.all_reduce(te)
        e_total = int(te.item())
    value = e_total * a.steps / (ms_res * 1e-3)
    e2e_value = e_total * a.steps / (ms_e2e * 1e-3)

    # ---- roofline of the dominant kernel (rank 0's launches) ---------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    # per kernel: SURVEY 8(d) algorithmic bytes and this implementation's own byte model, both
    # recorded per call by functional.kernel_bytes (layer 1 and layer 2 may run different plans)
    per, phases = {}, {}
    for k, v in kernel_list.items():
        if not v:
            continue
        if k.startswith("phase:"):
            phases[k[6:]] = float(np.sum(v) / a.steps)
            continue
        if kernel_bytes[k][0] is None:
            phases[k] = float(np.sum(v) / a.steps)
            continue
        ms = np.array(v)
        alg_b = sum(m["alg"] for m in kernel_bytes[k])
        mov_b = sum(m["moved"] for m in kernel_bytes[k])
        per[k] = {"ms_per_launch": float(ms.mean()), "launches_per_step": len(ms) / a.steps,
                  "gbs": alg_b / (ms.sum() * 1e-3) / 1e9, "moved_gbs": mov_b / (ms.sum() * 1e-3) / 1e9,
                  "bytes_per_launch": alg_b / len(ms), "moved_bytes_per_launch": mov_b / len(ms),
                  "ms_per_step": float(ms.sum() / a.steps)}
    dom = max(per, key=lambda k: per[k]["ms_per_step"]) if per else None
    roof = None
    tot_ms = sum(v["ms_per_step"] for v in per.values())
    if dom:
        tot_alg = sum(v["bytes_per_launch"] * v["launches_per_step"] for v in per.values())
        roof = {"bound": "hbm", "kernel": dom, "achieved": per[dom]["gbs"], "peak": peak, "unit": "GB/s",
                "frac": per[dom]["gbs"] / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": per[dom]["bytes_per_launch"],
                "moved_frac": per[dom]["moved_gbs"] / peak,
                "note": "achieved = SURVEY 8(d) gather-model bytes of the reference layer / CUDA-event time; "
                        "moved_* = bytes this implementation must move with no L2 reuse (sign record instead "
                        "of re-gathered rows, F floats for a shared operand); traffic = ncu DRAM bytes "
                        "(profiles/traffic.json, config A on one GPU)",
                "all_sparse_kernels": {"ms_per_step": tot_ms, "gbs": tot_alg / (tot_ms * 1e-3) / 1e9,
                                       "frac": tot_alg / (tot_ms * 1e-3) / 1e9 / peak},
                "plan": plan, "kernels": per}
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath) and world == 1 and a.config == "A":
            tj = json.load(open(tpath))
            roof["traffic"] = tj.get(dom) or tj.get(dom + "_ring")       # the ring kernels are the ones config A runs
    step_ms = ms_res / a.steps
    breakdown = {"ms_per_step": step_ms, "sparse_kernels_ms": tot_ms,
                 "projection_gemm_ms": phases.get("gemm_fwd", 0.0) + phases.get("gemm_bwd", 0.0) or None,
                 "exchange_exposed_ms": phases.get("exchange_exposed"),
                 "grad_allreduce_ms": phases.get("grad_allreduce"),
                 "note": "rank 0, CUDA events on the compute stream; projection_gemm = node projections and their "
                         "backward inside the partitioned layer (N > 1 only: at N = 1 they are ordinary autograd "
                         "GEMMs and sit in the remainder); exchange_exposed = time the compute stream waits for the "
                         "source all-gather / reduce-scatter; remainder = fuser GEMMs, dropout, ELU, loss"}
    known = sum(v for v in (breakdown["sparse_kernels_ms"], breakdown["projection_gemm_ms"],
                            breakdown["exchange_exposed_ms"], breakdown["grad_allreduce_ms"]) if v)
    breakdown["remainder_ms"] = step_ms - known

    secondary = None
    if not a.no_ssl_metric:
        if world == 1:
            secondary = {"supedge_step": supedge_step(margs, enc, graph, x_dev)}
        else:
            secondary = {"supedge_step": supedge_step_partitioned(a, enc, fus, part, x_dev, params)}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    cpu = None
    if world == 1 and not a.no_cpu_baseline:
        cpu, _, _ = cpu_reference_leg(a, a.cpu_budget_s, 1, 1, os.cpu_count() or 1)
    graph_info = graph.info
    part_info = None
    if part is not None:
        part_info = {"rows_rank0": part.n_local, "sources_rank0": part.n_src, "halo_rank0": len(part.halo_ids),
                     "exchange": part.mode}
    if world == 1 and not a.no_epoch_metric and a.config == "A":
        del enc, fus, x_dev, R, graph, x_bufs
        torch.cuda.empty_cache()
        secondary = secondary or {}
        try:
            secondary["cora_full_epoch_ms"] = cora_full_epoch_ms()
        except Exception as exc:
            secondary["cora_full_epoch_ms"] = {"error": "%s: %s" % (type(exc).__name__, exc)}
    line = {
        "metric": "DISGAT fwd+bwd edges/s", "value": value, "unit": "edges/s", "n_gpus": world,
        "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": step_ms, "higher_is_better": True,
        "scaling": "weak" if world == 1 else a.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(a, world, e_total, {
            "nodes_total": n_total, "setup_s": round(setup_s, 1), "graph_cache_hit": bool(cache_hit),
            "parallelism": "single GPU" if world == 1 else "dst-range x%d" % world,
            "graph": graph_info, "partition": part_info}),
        "e2e": {"value": e2e_value, "unit": "edges/s", "ms_per_step": ms_e2e / a.steps,
                "h2d_bytes_per_step": int(n_total * a.feat * 4), "d2h_bytes_per_step": 4 * world,
                "note": "every step's features come from pinned host memory (one H2D copy per step and rank, "
                        "double-buffered: the copy for step k+1 runs on a side stream under step k) and the loss is "
                        "read back; graph handle resident (built once, like the reference's adj.cuda())"},
        "gpu_launches": launches, "clocks": clk, "roofline": roof, "breakdown": breakdown, "cpu_baseline": cpu,
        "secondary": secondary,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
