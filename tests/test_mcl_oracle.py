"""CPU tests of the Markov clustering stage: the C oracle (oracle/mcl.c) against an independent float64 MCL written
here with scipy, its per-iteration invariants, and the CLI options that select the stage."""
import io

import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.csgraph import connected_components

from oracle import mcl as omcl

THETA, S, TAU, T = omcl.THETA, omcl.S, omcl.TAU, omcl.MAX_ITER


def scipy_mcl(n, src, dst, w, r=1.5, min_weight=1):
    """The definition of DESIGN.md §3 in float64 with scipy, sharing no code with the oracle."""
    src, dst, w = (np.asarray(x, dtype=np.int64) for x in (src, dst, w))
    keep = w >= max(min_weight, 1)
    src, dst, w = src[keep], dst[keep], w[keep].astype(np.float64)
    best = {}                                                     # symmetrise, duplicates merged by max
    for a, b, x in zip(np.r_[src, dst].tolist(), np.r_[dst, src].tolist(), np.r_[w, w].tolist()):
        best[(a, b)] = max(best.get((a, b), 0.0), x)
    keys = np.array(list(best), dtype=np.int64).reshape(-1, 2)
    A = sp.csc_matrix((np.array(list(best.values()), dtype=np.float64), (keys[:, 0], keys[:, 1])), shape=(n, n))
    loop = np.asarray(A.max(axis=0).todense()).ravel()
    loop[loop == 0] = 1.0
    A = A.tolil()
    A.setdiag(loop)
    M = A.tocsc()
    M = M.multiply(1.0 / np.asarray(M.sum(axis=0)).ravel()).tocsc()
    for _ in range(T):
        E = (M @ M).tocsc()
        cols = []
        for j in range(n):
            lo, hi = E.indptr[j], E.indptr[j + 1]
            r_, v_ = E.indices[lo:hi], E.data[lo:hi]
            n_theta = int((v_ >= THETA).sum())
            want = 1 if n_theta == 0 else min(n_theta, S)
            o = np.lexsort((r_, -v_))[:want]
            r_, v_ = r_[o], v_[o] ** r
            cols.append((r_, v_ / v_.sum(), np.full(r_.size, j)))
        rr, vv, cc = (np.concatenate(x) for x in zip(*cols))
        M = sp.csc_matrix((vv, (rr, cc)), shape=(n, n))
        mx = np.asarray(M.max(axis=0).todense()).ravel()
        sq = np.asarray(M.multiply(M).sum(axis=0)).ravel()
        if np.max(mx / sq - 1) < TAU:
            break
    _, lab = connected_components(M, directed=False)
    return lab


def partition_of_labels(lab):
    groups = {}
    for i, l in enumerate(np.asarray(lab).tolist()):
        groups.setdefault(l, []).append(i)
    return sorted(tuple(g) for g in groups.values())


def two_cliques():
    src, dst, w = [], [], []
    for base in (0, 5):
        for a in range(5):
            for b in range(a + 1, 5):
                src.append(base + a); dst.append(base + b); w.append(10)
    src.append(4); dst.append(5); w.append(1)
    return 10, src, dst, w


def ring_of_cliques(n_cliques=6, size=5):
    src, dst, w = [], [], []
    for c in range(n_cliques):
        base = c * size
        for a in range(size):
            for b in range(a + 1, size):
                src.append(base + a); dst.append(base + b); w.append(4)
        src.append(base + size - 1); dst.append(((c + 1) % n_cliques) * size); w.append(1)
    return n_cliques * size, src, dst, w


def path(n=30):
    return n, list(range(n - 1)), list(range(1, n)), [1] * (n - 1)


def star(leaves=2000):
    return leaves + 1, [0] * leaves, list(range(1, leaves + 1)), [1] * leaves


def planted(groups=10, size=20, p_in=0.5, p_out=0.01, seed=3):
    rng = np.random.default_rng(seed)
    n = groups * size
    src, dst, w = [], [], []
    for a in range(n):
        for b in range(a + 1, n):
            same = a // size == b // size
            if rng.random() < (p_in if same else p_out):
                src.append(a); dst.append(b); w.append(int(rng.integers(3, 9)) if same else 1)
    return n, src, dst, w


GRAPHS = {"two_cliques": two_cliques, "ring_of_cliques": ring_of_cliques, "path30": path, "star2000": star, "planted10x20": planted}


@pytest.mark.parametrize("name", sorted(GRAPHS))
def test_oracle_partition_matches_float64_scipy(name):
    n, src, dst, w = GRAPHS[name]()
    got = omcl.run(n, src, dst, w, 1.5)
    assert got["iterations"] < T
    assert omcl.partition(got["root"]) == partition_of_labels(scipy_mcl(n, src, dst, w, 1.5))
    if name == "two_cliques":
        assert omcl.partition(got["root"]) == [tuple(range(5)), tuple(range(5, 10))]
    if name == "planted10x20":
        assert omcl.partition(got["root"]) == [tuple(range(g * 20, g * 20 + 20)) for g in range(10)]


@pytest.mark.parametrize("name", sorted(GRAPHS))
def test_oracle_invariants_after_every_iteration(name):
    """Columns sum to 1, hold at most S entries with rows ascending, and no entry below theta survives the first
    pruning (checked against a float64 expansion of the oracle's start matrix)."""
    n, src, dst, w = GRAPHS[name]()
    seen = []

    def check(it, cp, rows, vals):
        seen.append(it)
        nnz = np.diff(cp)
        assert nnz.min() >= 1 and nnz.max() <= S
        sums = np.add.reduceat(vals.astype(np.float64), cp[:-1])
        # 1e-6, widened for long columns: each float32 quotient x / sum carries its own rounding of up to 2^-24
        assert np.all(np.abs(sums - 1.0) <= np.maximum(1e-6, nnz * 2.0 ** -23))
        for j in range(n):
            r = rows[cp[j]:cp[j + 1]]
            assert np.all(np.diff(r) > 0)                       # rows strictly ascending inside a column
    out = omcl.run(n, src, dst, w, 2.0, trace=check)
    assert seen == list(range(1, out["iterations"] + 1))
    # theta: recompute one expansion in float64 from the oracle's start and compare the kept set of iteration 1
    one = omcl.run(n, src, dst, w, 2.0, iters=1)
    zero = omcl.run(n, src, dst, w, 2.0, iters=0)
    M = sp.csc_matrix((zero["vals"].astype(np.float64), zero["rows"], zero["colptr"]), shape=(n, n))
    E = (M @ M).tocsc()
    for j in range(n):
        e = E[:, j].toarray().ravel()
        kept = one["rows"][one["colptr"][j]:one["colptr"][j + 1]]
        if (e >= THETA * 1.001).sum() >= 1:
            assert np.all(e[kept] >= THETA * 0.999)


def test_oracle_iteration_count_and_stats():
    n, src, dst, w = two_cliques()
    out = omcl.run(n, src, dst, w, 1.5)
    st = out["stats"]
    assert len(st) == out["iterations"] and st[-1]["chaos"] < TAU and all(s["chaos"] >= TAU for s in st[:-1])
    assert st[-1]["nnz"] == out["rows"].size == 10     # converged: every column holds its attractor only


def test_min_weight_drops_weak_edges():
    n, src, dst, w = two_cliques()
    out = omcl.run(n, src, dst, w, 1.5, min_weight=2)
    assert omcl.partition(out["root"]) == [tuple(range(5)), tuple(range(5, 10))]


def test_cli_cluster_options():
    from pangenome_b200 import cli
    a, extra, _ = cli.parse_args(["prog", "-i", "x.fa", "--cluster", "mcl", "--inflation", "2.5"])
    assert cli.cluster_options(extra) == ("mcl", 2.5)
    _, extra, _ = cli.parse_args(["prog", "-i", "x.fa"])
    assert cli.cluster_options(extra) == ("components", 1.5)
    for bad in (["--cluster", "louvain"], ["--inflation", "1"], ["--inflation", "0.5"], ["--inflation", "x"],
                ["--inflation", "nan"], ["--cluster", "mcl", "--inflation", "-3"]):
        with pytest.raises(SystemExit) as e:
            cli.entry_point(["prog", "-i", "x.fa", "-k", "27"] + bad, out=io.StringIO())
        assert ("--cluster" in str(e.value)) or ("--inflation" in str(e.value))


def test_standalone_mcl_arguments(tmp_path):
    """python -m pangenome_b200.mcl accepts the reference's argument list (kmer_numba.py:1911) and rejects bad ones
    before touching a GPU."""
    from pangenome_b200 import mcl
    for bad in (["x.xyz", "-I", "1.0"], ["x.xyz", "-I"], ["x.xyz", "--bogus"], [], ["a.xyz", "b.xyz"]):
        with pytest.raises(SystemExit):
            mcl.main(bad)
    f = tmp_path / "g.xyz"
    f.write_text("12_3\t45_6\t7\n45_6\t7625597484986_544\t1\n")
    c0, v0, c1, v1, w = mcl.read_xyz(str(f))
    assert c1.tolist() == [45, 7625597484986] and v1.tolist() == [6, 544] and w.tolist() == [7, 1]
