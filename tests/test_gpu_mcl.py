"""GPU Markov clustering (K7m, pangenome_b200/csrc/mcl.cu) against the CPU oracle (oracle/mcl.c): bit-identical
matrices for inflations that are multiples of 1/2, equal partitions otherwise, and the stage inside seq2graph, the
CLI, the standalone `python -m pangenome_b200.mcl` and the multi-GPU CLI."""
import io
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from conftest import ROOT, load_small_cases
from oracle import mcl as omcl
from pangenome_b200.synth import pangenome, survey_4x1m

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def dense_edges(c0, v0, c1, v1, w):
    """.xyz edges -> (n, src, dst, w, names): dense ids in (code, v5) order."""
    names = np.stack([np.concatenate([c0, c1]).astype(np.int64), np.concatenate([v0, v1]).astype(np.int64)], axis=1)
    uniq, inv = np.unique(names, axis=0, return_inverse=True)
    inv = inv.reshape(-1)
    m = len(c0)
    return uniq.shape[0], inv[:m], inv[m:], np.asarray(w, dtype=np.int64), uniq


def planted_graph(seed=7, groups=40, size=25):
    rng = np.random.default_rng(seed)
    n = groups * size
    a = rng.integers(0, n, 12 * n)
    same = rng.integers(0, size, 12 * n) + (a // size) * size
    b = np.where(rng.random(12 * n) < 0.9, same, rng.integers(0, n, 12 * n))
    w = np.where(a // size == b // size, rng.integers(2, 20, a.size), 1)
    return n, a, b, w


def star_graph(leaves=1100):
    return leaves + 1, np.zeros(leaves, np.int64), np.arange(1, leaves + 1), np.ones(leaves, np.int64)


def hub_graph(seed=5, n=6000, hub_deg=5000):
    """A hub linked to most nodes over a sparse random graph: its column and its neighbours' columns take the CTA path
    with the accumulator in global memory (more than PG_MCL_SMEM_SLOTS / 2 products)."""
    rng = np.random.default_rng(seed)
    a = np.r_[np.zeros(hub_deg, np.int64), rng.integers(1, n, 3 * n)]
    b = np.r_[rng.choice(np.arange(1, n), hub_deg, replace=False), rng.integers(1, n, 3 * n)]
    w = rng.integers(1, 6, a.size)
    return n, a, b, w


@pytest.fixture(scope="module")
def survey_edges(torch):
    from pangenome_b200 import engine, graph
    data = survey_4x1m()
    packed = engine.PackedSeqs(engine.to_device_bytes(data))
    t, _ = engine.build_dbg(packed, 27)
    res = graph.seq2graph_device(packed, t.select_rdbg(), 27)
    assert len(res.edges[0]) == 142203
    return dense_edges(*res.edges)[:4]


def gpu_run(torch, n, src, dst, w, r, iters=None, min_weight=1):
    from pangenome_b200 import mcl
    t = lambda x: torch.as_tensor(np.asarray(x, dtype=np.int64), device="cuda")
    return mcl.markov_cluster(n, t(src), t(dst), t(w), r, min_weight=min_weight, iters=iters)


def assert_same_matrix(g, o):
    cp = g.colptr.cpu().numpy()
    assert np.array_equal(cp, o["colptr"])
    nnz = int(cp[-1])
    assert np.array_equal(g.rows[:nnz].cpu().numpy(), o["rows"])
    assert np.array_equal(g.vals[:nnz].cpu().numpy().view(np.uint32), o["vals"].view(np.uint32))


@pytest.mark.parametrize("r", [1.5, 2.0, 3.0])
@pytest.mark.parametrize("which", ["planted", "star", "hub", "survey_4x1m"])
def test_bit_exact_matrices(torch, request, which, r):
    n, src, dst, w = {"planted": planted_graph, "star": star_graph, "hub": hub_graph}[which]() if which != "survey_4x1m" \
        else request.getfixturevalue("survey_edges")
    for iters in (1, 2, 3):
        g = gpu_run(torch, n, src, dst, w, r, iters)
        o = omcl.run(n, src, dst, w, r, iters=iters)
        assert_same_matrix(g, o)
        assert [s["nnz"] for s in g.stats] == [s["nnz"] for s in o["stats"]]
        assert [s["products"] for s in g.stats] == [s["products"] for s in o["stats"]]
        if which == "hub" and iters == 1:
            assert g.stats[0]["large_columns"] > 0
    g = gpu_run(torch, n, src, dst, w, r)
    o = omcl.run(n, src, dst, w, r)
    assert g.iterations == o["iterations"] < omcl.MAX_ITER
    assert_same_matrix(g, o)
    assert np.array_equal(g.root.cpu().numpy(), o["root"])


@pytest.mark.parametrize("which", ["planted", "hub"])
def test_non_half_integer_inflation_same_partition(torch, which):
    n, src, dst, w = {"planted": planted_graph, "hub": hub_graph}[which]()
    g = gpu_run(torch, n, src, dst, w, 1.7)
    o = omcl.run(n, src, dst, w, 1.7)
    assert omcl.partition(g.root.cpu().numpy()) == omcl.partition(o["root"])


def test_deterministic_on_config2(torch):
    from pangenome_b200 import engine, graph
    data = pangenome(10, 5_000_000)
    packed = engine.PackedSeqs(engine.to_device_bytes(data))
    t, _ = engine.build_dbg(packed, 27)
    rd = t.select_rdbg()
    a = graph.seq2graph_device(packed, rd, 27, cluster="mcl")
    b = graph.seq2graph_device(packed, rd, 27, cluster="mcl")
    for x, y in zip(a.nodes[1:], b.nodes[1:]):           # (code, v5, label); node slots vary with K6's CAS races
        assert np.array_equal(x, y)
    assert a.rows(packed, data) == b.rows(packed, data)


def oracle_lines(edges, min_weight=1, r=1.5):
    """The oracle's MCL on .xyz edges, as cluster-file lines: clusters ranked by (size desc, smallest (code, v5))."""
    n, src, dst, w, names = dense_edges(*edges)
    o = omcl.run(n, src, dst, w, r, min_weight=min_weight)
    groups = {}
    for i, root in enumerate(o["root"].tolist()):
        groups.setdefault(root, []).append(i)              # dense ids ascend = (code, v5) ascend
    ranked = sorted(groups.values(), key=lambda g: (-len(g), g[0]))
    return ["\t".join("%d_%d" % (names[i, 0], names[i, 1]) for i in g) for g in ranked], o


def many_components_input():
    from pangenome_b200.synth import fasta_bytes, _ACGT
    rng = np.random.default_rng(11)
    recs = []
    for fam in range(5):
        anc = rng.integers(0, 4, 3000 + 500 * fam, dtype=np.uint8)
        for g in range(2 + fam % 3):
            s = anc.copy()
            m = rng.random(anc.size) < 0.02
            s[m] = (s[m] + rng.integers(1, 4, int(m.sum()), dtype=np.uint8)) % 4
            recs.append((b"fam%d_g%d" % (fam, g), _ACGT[s]))
    return fasta_bytes(recs, width=70)


@pytest.mark.parametrize("which,k,c", [("many_components", 9, 3), ("many_components", 21, 2), ("pangenome4x30k", 15, 2)])
def test_pipeline(torch, which, k, c):
    from pangenome_b200 import engine, graph
    data = many_components_input() if which == "many_components" else pangenome(4, 30000, snp=0.02, seed=9)
    packed = engine.PackedSeqs(engine.to_device_bytes(data))
    t, _ = engine.build_dbg(packed, k, rc=bool(c & 2))
    rd = t.select_rdbg()
    base = graph.seq2graph_device(packed, rd, k, rc=bool(c & 1))
    res = graph.seq2graph_device(packed, rd, k, rc=bool(c & 1), cluster="mcl")
    assert res.xyz_lines() == base.xyz_lines() == oracle.run(data, k, c=c)["xyz"]
    lines, o = oracle_lines(res.edges)
    assert res.mcl_lines() == lines
    pinned = graph.seq2graph_device(packed, rd, k, rc=bool(c & 1), mcl_lines=lines)
    assert res.rows(packed, data) == pinned.rows(packed, data)
    if which == "pangenome4x30k":
        n_mcl, n_cc = len(set(res.nodes[3].tolist())), len(set(base.nodes[3].tolist()))
        assert n_mcl > n_cc, (n_mcl, n_cc)
    # --min-edge-weight 3 with MCL: the oracle on the filtered edge list
    r3 = graph.seq2graph_device(packed, rd, k, rc=bool(c & 1), min_weight=3, cluster="mcl")
    assert r3.mcl_lines() == oracle_lines(res.edges, min_weight=3)[0]


def run_cli(argv):
    from pangenome_b200 import cli
    out = io.StringIO()
    cli.entry_point(argv, out=out)
    text = out.getvalue()
    return text, [l for l in text.split("\n") if l and not l.startswith("#")]


def test_cli_cluster_mcl_and_standalone(torch, tmp_path):
    from pangenome_b200 import graph, mcl
    fa = tmp_path / "pg.fa"
    data = pangenome(4, 30000, snp=0.02, seed=9)
    fa.write_bytes(data)
    _, rows = run_cli(["prog", "-i", str(fa), "-k", "15", "--cluster", "mcl", "--inflation", "1.5", "--no-dump-db"])
    xyz = str(fa) + "_rdbg_weight.xyz"
    edges = mcl.read_xyz(xyz)
    lines, _ = oracle_lines(edges)
    got = open(xyz + ".mcl").read().split("\n")[:-1]
    assert got == lines
    # the rows are those of the pinned label path for the same cluster file
    from pangenome_b200 import engine
    packed = engine.PackedSeqs(engine.to_device_bytes(data))
    t, _ = engine.build_dbg(packed, 15)
    pinned = graph.seq2graph_device(packed, t.select_rdbg(), 15, mcl_lines=lines)
    assert rows == ["%s\t%d\t%d\t%s\t%d" % r for r in pinned.rows(packed, data)]
    # second run: the cluster file wins
    text2, rows2 = run_cli(["prog", "-i", str(fa), "-k", "15", "--cluster", "mcl", "--no-dump-db"])
    assert "# the mcl has been ran" in text2 and rows2 == rows
    # the standalone clusterer writes the same bytes
    out = tmp_path / "x.mcl"
    p = subprocess.run([sys.executable, "-m", "pangenome_b200.mcl", xyz, "--abc", "-I", "1.5", "-te", "8", "-o", str(out),
                        "-q", "x", "-V", "all"], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    assert out.read_bytes() == open(xyz + ".mcl", "rb").read()
    # test.fsa at k = 27: empty edge set -> no rows, exit 0, an empty cluster file
    case = {c["name"]: c for c in load_small_cases()}["test_fsa_k5"]
    tf = tmp_path / "test.fsa"
    tf.write_bytes(case["input_latin1"].encode("latin-1"))
    _, rows27 = run_cli(["prog", "-i", str(tf), "-k", "27", "--cluster", "mcl", "--no-dump-db"])
    assert rows27 == []


def test_multigpu_cli_cluster_mcl(torch, tmp_path):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    fa = tmp_path / "pg.fa"
    fa.write_bytes(pangenome(4, 30000, snp=0.02, seed=9))
    _, rows = run_cli(["prog", "-i", str(fa), "-k", "15", "--cluster", "mcl", "--no-dump-db"])
    mcl_one = open(str(fa) + "_rdbg_weight.xyz.mcl").read()
    os.remove(str(fa) + "_rdbg_weight.xyz.mcl")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29591", os.path.join(ROOT, "kmer_b200.py"), "-i", str(fa), "-k", "15", "--cluster", "mcl", "--no-dump-db"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
    assert [l for l in p.stdout.split("\n") if l and not l.startswith("#")] == rows
    assert open(str(fa) + "_rdbg_weight.xyz.mcl").read() == mcl_one
