"""CPU tests: the C-ABI library loads, exports every symbol include/edis.h declares, and the
host-side (integer) entry points are bit-exact against the reference goldens.  No GPU calls."""
import ctypes
import hashlib
import os
import re

import numpy as np
import pytest
import torch

import edgedisentangle_ssl_b200 as edis
from edgedisentangle_ssl_b200 import _lib
from edgedisentangle_ssl_b200.sampler import sample_pairs, homo_hetero_split
from helpers import load

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "edis.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(edis_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    syms = declared_symbols()
    assert len(syms) >= 20
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for s in syms:
        assert hasattr(lib, s), "libedis.so does not export %s" % s
    assert set(syms) == set(_lib.SIGNATURES), set(syms) ^ set(_lib.SIGNATURES)
    assert "sm_100a" in _lib.version()


def test_library_is_sm100a_only():
    import subprocess
    out = subprocess.run(["cuobjdump", "-lelf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_ops_fail_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_lib.EdisError):
        edis.Graph(3, [0, 1, 2], [0, 1, 2], device="cuda:0")
    with pytest.raises(_lib.EdisError):
        edis.Graph(3, [0, 1, 2], [0, 1, 2], device="cpu")
    lay = edis.DisGALayer(4, 8, 0.0, 0.1, att_type=2)
    adj = torch.sparse_coo_tensor(torch.tensor([[0, 1], [1, 0]]), torch.ones(2), (2, 2))
    with pytest.raises(_lib.EdisError):
        lay(torch.randn(2, 4), adj)


def test_bad_arguments_report_errors():
    r = _lib.lib.edis_build_adjacency_host(0, 0, None, None, None, None, None, None)
    assert r < 0 and "bad arguments" in _lib.last_error()
    with pytest.raises(_lib.EdisError):
        edis.build_adjacency(3, [0, 5], [1, 1])  # out of range


# ------------------------------------------------------------------ graph builder (bit-exact)
def test_build_adjacency_edge_list():
    g = load("graph_small")
    e = g["el_edges"]
    idx, val = edis.build_adjacency(int(e.max()) + 1, e[:, 0], e[:, 1])
    assert np.array_equal(idx, g["el_indices"]) and np.array_equal(val, g["el_values"])


def test_build_adjacency_weighted_csr():
    g = load("graph_small")
    idx, val = edis.build_adjacency(int(g["csr_n"]), g["csr_row"], g["csr_col"], g["csr_val"])
    assert np.array_equal(idx, g["csr_indices"]) and np.array_equal(val, g["csr_values"])


def test_build_adjacency_empty_and_isolated():
    idx, val = edis.build_adjacency(4, [], [])
    assert np.array_equal(idx, np.stack([np.arange(4), np.arange(4)])) and np.all(val == 1.0)


@pytest.mark.parametrize("ds", ["cora", "chameleon", "cora_full"])
def test_build_adjacency_bundled(ds):
    from edgedisentangle_ssl_b200.data_load import load_graph_arrays
    g = load("graph_bundled")
    n, r, c, v = load_graph_arrays(os.path.join(ROOT, "data", ds) + "/")
    idx, val = edis.build_adjacency(n, r, c, v)
    assert n == int(g[ds + "_n"]) and idx.shape[1] == int(g[ds + "_e"])
    assert sha(idx) == str(g[ds + "_idx_sha"]) and sha(val) == str(g[ds + "_val_sha"])


# ------------------------------------------------------------------ sampler (bit-exact)
def seed_all(s):
    import random
    random.seed(s)
    np.random.seed(s)
    torch.manual_seed(s)


@pytest.mark.parametrize("tag", ["model_a3_AT", "model_a2_GCN"])
def test_sampler_small(tag):
    g = load(tag)
    n, idx = int(g["n"]), g["indices"]
    seed_all(8)
    pairs, lab = sample_pairs(n, idx, chunk_rows=7)
    assert np.array_equal(pairs, g["sup.sample_idx"]) and np.array_equal(lab, g["sup.sample_lab"])
    homo, het = homo_hetero_split(idx, g["labels"])
    seed_all(9)
    p0, l0 = sample_pairs(n, homo)
    p1, l1 = sample_pairs(n, het, chunk_rows=5)
    assert np.array_equal(p0, g["dis.sample_idx0"]) and np.array_equal(l0, g["dis.sample_lab0"])
    assert np.array_equal(p1, g["dis.sample_idx1"]) and np.array_equal(l1, g["dis.sample_lab1"])


def test_sampler_cora():
    from edgedisentangle_ssl_b200.data_load import load_graph_arrays
    g = load("graph_bundled")
    n, r, c, v = load_graph_arrays(os.path.join(ROOT, "data", "cora") + "/")
    idx, _ = edis.build_adjacency(n, r, c, v)
    seed_all(4)
    pairs, lab = sample_pairs(n, idx)
    assert pairs.shape[1] == int(g["cora_sample_m"])
    assert sha(pairs) == str(g["cora_sample_idx_sha"]) and sha(lab) == str(g["cora_sample_lab_sha"])


@pytest.mark.parametrize("seed,n,thr", [(0, 1000, 0.013), (4, 3001, 0.00217), (11, 50, 0.5), (3, 700, 1e-9),
                                        (5, 333, 1.0), (9, 1, 0.3)])
def test_rand_hits_replays_torch_cpu_generator_bit_exactly(seed, n, thr):
    """edis_rand_hits_host == (torch.rand(N, N) < thr).nonzero() on the CPU default generator,
    hit for hit, and leaves the generator in the same state (the reference samples its SSL pairs
    from exactly this stream, pretrainer.py:692)."""
    import numpy as np
    import torch
    from edgedisentangle_ssl_b200.sampler import bernoulli_hits
    torch.manual_seed(seed)
    torch.rand(seed * 7 + 3)                      # start in the middle of a 624-word block
    st0 = torch.get_rng_state().clone()
    ref = (torch.rand(size=(n, n)) < thr).nonzero()
    ref_key = (ref[:, 0] * n + ref[:, 1]).numpy()
    after_ref = torch.rand(7)
    torch.set_rng_state(st0)
    got = bernoulli_hits(n * n, thr)
    assert got is not None and np.array_equal(got, ref_key)
    assert torch.equal(torch.rand(7), after_ref)


def test_load_data_refuses_missing_features_unless_opted_in(monkeypatch, tmp_path):
    """data_load.py:36 fails on a missing feature file; so does the drop-in.  Label-derived synthetic
    features are an explicit opt-in (EDIS_SYNTH_FEATURES=1) for benchmarks / tests only."""
    from edgedisentangle_ssl_b200 import data_load
    from edgedisentangle_ssl_b200.utils import get_parser
    args = get_parser().parse_args(["--model=DISGAT", "--sparse", "--dataset=cora"])
    path = os.path.join(ROOT, "data", "cora") + "/"
    monkeypatch.delenv("EDIS_SYNTH_FEATURES", raising=False)
    with pytest.raises(FileNotFoundError):
        data_load.load_data(args, path=path, dataset="cora", edge_type=1)
    monkeypatch.setenv("EDIS_SYNTH_FEATURES", "1")
    adj, feats, labels = data_load.load_data(args, path=path, dataset="cora", edge_type=1)
    assert feats.shape == (2708, 64) and adj.shape == (2708, 2708)


def test_load_data_cache_round_trip_and_stale_input(monkeypatch, tmp_path):
    """EDIS_CACHE_DIR: the processed adjacency is cached keyed by the raw input file's bytes; a second
    load returns identical tensors from the cache, and a changed input file gets a new key (no stale hit)."""
    import shutil
    from edgedisentangle_ssl_b200 import data_load
    from edgedisentangle_ssl_b200.utils import get_parser
    ds = tmp_path / "cham"
    shutil.copytree(os.path.join(ROOT, "data", "chameleon"), ds)
    cache = tmp_path / "cache"
    monkeypatch.setenv("EDIS_CACHE_DIR", str(cache))
    args = get_parser().parse_args(["--model=DISGAT", "--sparse", "--dataset=chameleon"])
    a1, _, _ = data_load.load_data(args, path=str(ds) + "/", dataset="chameleon", edge_type=1)
    files = sorted(os.listdir(cache))
    assert len(files) == 1 and files[0].startswith("adj_1_")
    a2, _, _ = data_load.load_data(args, path=str(ds) + "/", dataset="chameleon", edge_type=1)
    assert torch.equal(a1.coalesce().indices(), a2.coalesce().indices())
    assert torch.equal(a1.coalesce().values(), a2.coalesce().values())
    edge = np.load(ds / "adj_1.npy")
    np.save(ds / "adj_1.npy", edge[:-7])                       # the input changes -> new key, rebuilt
    a3, _, _ = data_load.load_data(args, path=str(ds) + "/", dataset="chameleon", edge_type=1)
    assert len(os.listdir(cache)) == 2 and a3._nnz() != a1._nnz()


def test_header_compiles_as_c_and_struct_layout(tmp_path):
    """include/edis.h is a C header (no CUDA / C++ needed to bind it): compile a C translation unit
    against it, independent of _lib.py, and pin the edis_layer_desc layout binders rely on."""
    import subprocess
    src = tmp_path / "abi_check.c"
    src.write_text('''
#include <stddef.h>
#include "edis.h"
_Static_assert(sizeof(edis_layer_desc) == 40, "edis_layer_desc must be 40 bytes");
_Static_assert(offsetof(edis_layer_desc, att) == 0 && offsetof(edis_layer_desc, C) == 4, "att, C");
_Static_assert(offsetof(edis_layer_desc, D) == 8 && offsetof(edis_layer_desc, Dv) == 12, "D, Dv");
_Static_assert(offsetof(edis_layer_desc, training) == 16 && offsetof(edis_layer_desc, p) == 20, "training, p");
_Static_assert(offsetof(edis_layer_desc, seed) == 24, "seed");
_Static_assert(offsetof(edis_layer_desc, flags) == 32 && offsetof(edis_layer_desc, reserved) == 36, "flags");
/* every entry point must be declared with a prototype a C caller can take the address of */
static const void* table[] = {
  (const void*)edis_last_error, (const void*)edis_version, (const void*)edis_build_adjacency_host,
  (const void*)edis_graph_create, (const void*)edis_graph_create_rect, (const void*)edis_graph_destroy,
  (const void*)edis_graph_info, (const void*)edis_graph_export, (const void*)edis_graph_workspace_bytes,
  (const void*)edis_edge_list_key, (const void*)edis_graph_save, (const void*)edis_graph_load,
  (const void*)edis_disga_fwd, (const void*)edis_disga_bwd, (const void*)edis_disga_bwd_dst,
  (const void*)edis_disga_bwd_src, (const void*)edis_pair_score_fwd, (const void*)edis_pair_score_bwd,
  (const void*)edis_ssl_wmse_fwd, (const void*)edis_ssl_wmse_bwd };
int main(void) { return table[0] == 0; }
''')
    lib_dir = os.path.join(ROOT, "edgedisentangle_ssl_b200")
    exe = tmp_path / "abi_check"
    cmd = ["gcc", "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
           "-L", lib_dir, "-l:libedis.so", "-Wl,-rpath," + lib_dir]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr


def test_reference_arm_runs_without_the_package():
    """`bench.py --impl reference` (the reference arm): times the UNMODIFIED reference from oracle/_ref on the host
    cores, prints one JSON line with impl / cpu_baseline / e2e, and never maps libedis.so (it must not import
    edgedisentangle_ssl_b200).  Tiny sample here.  The reference sources are not part of this repository: only
    where build() found them and made oracle/_ref does this cover the unmodified reference.  Everywhere else it
    covers the oracle-port arm (the line must say kind "port"), which shares the no-package, no-libedis property."""
    import json
    import subprocess
    import sys
    kind = "reference" if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "MANIFEST.json")) else "port"
    code = ("import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '1', "
            "'--ref-total-s', '1', '--cpu-probe-edges', '20000']; runpy.run_path(%r, run_name='__main__'); "
            "mods = [m for m in sys.modules if m.startswith('edgedisentangle_ssl_b200')]; "
            "maps = open('/proc/self/maps').read(); print('LOADED', mods, 'libedis' in maps)") % os.path.join(ROOT, "bench.py")
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "edges/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == kind and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["gpu_launches"] == 0
    assert "LOADED [] False" in p.stdout, p.stdout[-400:]
