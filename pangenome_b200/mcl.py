"""Markov clustering of a weighted edge list on the GPU (K7m: pangenome_b200/csrc/mcl.cu, definition in DESIGN.md §3).

    python -m pangenome_b200.mcl <file.xyz> --abc -I 1.5 -te 8 -o <out> -q x -V all

clusters an existing ``<F>_rdbg_weight.xyz`` the way the reference's ``mcl`` call does (kmer_numba.py:1911) and
writes the cluster file: one line of ``code_v5`` names per cluster, clusters ranked by (size descending, smallest
(code, v5)).  ``--abc``, ``-te``, ``-q`` and ``-V`` are accepted and ignored; ``-o`` defaults to ``<file.xyz>.mcl``.
"""
import ctypes
import sys
import time

import numpy as np
import torch

from . import _lib
from ._lib import PgError, check
from .engine import _ptr, _stream

WS_BYTES = 1 << 30          # global accumulator slabs of the large-column CTAs (at least one slab is always granted)


class MclResult:
    """root: int32 device tensor, one root (smallest dense id of its cluster) per dense node; stats: one dict per
    iteration (nnz, products, chaos, large_columns, ms = host clock between the device synchronisations that end
    consecutive iterations); colptr / rows / vals: the final matrix (CSC, device)."""

    def __init__(self, root, stats, iterations, colptr, rows, vals):
        self.root, self.stats, self.iterations = root, stats, iterations
        self.colptr, self.rows, self.vals = colptr, rows, vals


def build_matrix(n, src, dst, w, min_weight=1):
    """The column-normalised start matrix in CSC form (device tensors): edges of weight >= max(min_weight, 1),
    symmetrised, duplicates merged by max, A[j,j] = max_i A[i,j] (1 for a node left without an edge)."""
    dev = src.device
    keep = w >= max(int(min_weight), 1)
    src, dst, wf = src[keep].long(), dst[keep].long(), w[keep].float()       # integer weights: exact below 2^24
    col, row, val = torch.cat([dst, src]), torch.cat([src, dst]), torch.cat([wf, wf])
    loop = torch.zeros(n, dtype=torch.float32, device=dev).scatter_reduce_(0, col, val, "amax")
    loop[loop == 0] = 1.0
    ar = torch.arange(n, dtype=torch.int64, device=dev)
    col, row, val = torch.cat([col, ar]), torch.cat([row, ar]), torch.cat([val, loop])
    key, inv = torch.unique(col * n + row, return_inverse=True)               # sorted: column, then row ascending
    vals = torch.zeros(key.numel(), dtype=torch.float32, device=dev).scatter_reduce_(0, inv, val, "amax", include_self=False)
    colptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    colptr[1:] = torch.cumsum(torch.bincount(key // n, minlength=n), 0)
    return colptr, (key % n).to(torch.int32), vals


def _chaos(word):
    return float(np.array([word], dtype=np.uint32).view(np.float32)[0])


def markov_cluster(n, src, dst, w, inflation=1.5, min_weight=1, iters=None):
    """MCL over nodes 0..n-1 and edges (src, dst, w) (device tensors).  ``iters`` = None: iterate until the max
    chaos falls below tau or T iterations ran; an integer stops after exactly that many iterations (tests compare
    the matrix bit for bit with the CPU oracle there)."""
    inflation = float(inflation)
    if not 1.0 < inflation < 64.0:
        raise PgError("inflation must be in (1, 64), got %r" % inflation)
    L = _lib.load()
    S = _stream
    n = int(n)
    dev = src.device
    if n >= 1 << 31:
        raise PgError("more than 2^31 - 1 nodes")
    cp, rows, vals = build_matrix(n, src, dst, w, min_weight)
    i64 = torch.int64
    stats = torch.zeros(_lib.PG_MCL_STAT_WORDS, dtype=i64, device=dev)
    check(L.pg_mcl_normalise(_ptr(cp), _ptr(rows), _ptr(vals), n, _ptr(stats), S()), "pg_mcl_normalise")
    scan_bytes = int(L.pg_mcl_scan_workspace_bytes(n))
    scan_ws = torch.empty(scan_bytes, dtype=torch.uint8, device=dev)
    prod = torch.empty(max(n, 1), dtype=i64, device=dev)
    stage_off = torch.empty(n + 1, dtype=i64, device=dev)
    large = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    kept = torch.empty(max(n, 1), dtype=i64, device=dev)
    max_ctas = 4 * int(L.pg_device_sms())
    log = []
    it, limit = 0, _lib.PG_MCL_MAX_ITER if iters is None else int(iters)
    t0 = time.perf_counter()
    while it < limit and n > 0:
        stats.zero_()
        check(L.pg_mcl_plan(_ptr(cp), _ptr(rows), n, _ptr(prod), _ptr(stage_off), _ptr(large), _ptr(stats), _ptr(scan_ws),
                            scan_bytes, S()), "pg_mcl_plan")
        h = torch.cat([stats, stage_off[n:]]).cpu().numpy()
        n_large, max_prod, n_stage = int(h[_lib.PG_MCL_STAT_LARGE]), int(h[_lib.PG_MCL_STAT_MAXPROD]), int(h[-1])
        srows = torch.empty(max(n_stage, 1), dtype=torch.int32, device=dev)
        svals = torch.empty(max(n_stage, 1), dtype=torch.float32, device=dev)
        slab = int(L.pg_mcl_slab_slots(max_prod, n))
        n_ctas = max(1, min(n_large, max_ctas))
        ws, ws_bytes = None, 0
        if n_large and slab > _lib.PG_MCL_SMEM_SLOTS:     # larger accumulators live in global memory
            n_ctas = max(1, min(n_ctas, WS_BYTES // (8 * slab)))
            ws_bytes = n_ctas * slab * 8
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        check(L.pg_mcl_expand(_ptr(cp), _ptr(rows), _ptr(vals), n, _ptr(prod), _ptr(stage_off), _ptr(large), n_large, max_prod,
                              ctypes.c_float(inflation), _ptr(srows), _ptr(svals), _ptr(kept), _ptr(stats),
                              _ptr(ws) if ws is not None else None, ws_bytes, n_ctas, S()), "pg_mcl_expand")
        h2 = stats.cpu().numpy()
        nnz, chaos = int(h2[_lib.PG_MCL_STAT_NNZ]), _chaos(h2[_lib.PG_MCL_STAT_CHAOS])
        cp = torch.empty(n + 1, dtype=i64, device=dev)
        rows = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
        vals = torch.empty(max(nnz, 1), dtype=torch.float32, device=dev)
        check(L.pg_mcl_compact(_ptr(stage_off), _ptr(srows), _ptr(svals), _ptr(kept), n, _ptr(cp), _ptr(rows), _ptr(vals),
                               _ptr(scan_ws), scan_bytes, S()), "pg_mcl_compact")
        rows, vals = rows[:nnz], vals[:nnz]
        it += 1
        t1 = time.perf_counter()
        log.append({"nnz": nnz, "products": int(h[_lib.PG_MCL_STAT_PRODUCTS]), "chaos": chaos, "large_columns": n_large,
                    "ms": 1e3 * (t1 - t0)})
        t0 = t1
        if iters is None and np.float32(chaos) < np.float32(_lib.PG_MCL_CHAOS_TAU):
            break
    root = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    check(L.pg_mcl_components(_ptr(cp), _ptr(rows), n, _ptr(root), S()), "pg_mcl_components")
    return MclResult(root[:n], log, it, cp, rows, vals)


def read_xyz(path):
    """(c0, v0, c1, v1, w) int64 arrays of a ``.xyz`` file ("code_v5\\tcode_v5\\tweight" lines), parsed by numpy's C
    reader (codes are < 5^27 < 2^63)."""
    import io
    with open(path, "rb") as f:
        raw = f.read().replace(b"_", b"\t")
    if not raw.strip():
        z = np.zeros(0, np.int64)
        return z, z, z, z, z
    a = np.loadtxt(io.BytesIO(raw), dtype=np.int64, delimiter="\t", ndmin=2)
    if a.shape[1] != 5:
        raise PgError("%s: expected lines 'code_v5<TAB>code_v5<TAB>weight'" % path)
    return tuple(np.ascontiguousarray(a[:, i]) for i in range(5))


def cluster_xyz(path, out, inflation=1.5, device="cuda"):
    """Cluster the edges of a ``.xyz`` file and write the cluster file ``out``."""
    from . import graph
    c0, v0, c1, v1, w = read_xyz(path)
    names = np.stack([np.concatenate([c0, c1]), np.concatenate([v0, v1])], axis=1)
    uniq, inv = np.unique(names, axis=0, return_inverse=True) if names.size else (np.zeros((0, 2), np.int64), np.zeros(0, np.int64))
    n, m = uniq.shape[0], c0.size
    code = torch.from_numpy(np.ascontiguousarray(uniq[:, 0])).to(device)
    v5 = torch.from_numpy(np.ascontiguousarray(uniq[:, 1])).to(device)
    root = torch.zeros(0, dtype=torch.int64, device=device)
    if n:
        inv = torch.from_numpy(inv.reshape(-1).astype(np.int64)).to(device)
        res = markov_cluster(n, inv[:m], inv[m:], torch.from_numpy(w).to(device), inflation)
        root = res.root.long()
    order, label_sorted, _ = graph.rank_clusters(code, v5, root)
    o3 = torch.argsort(label_sorted, stable=True)
    fin = order[o3]
    code_h = np.ascontiguousarray(code[fin].cpu().numpy().view(np.uint64))
    v5_h = np.ascontiguousarray(v5[fin].cpu().numpy().astype(np.uint32))
    lab_h = np.ascontiguousarray(label_sorted[o3].cpu().numpy().astype(np.int64))
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    check(_lib.load().pg_host_write_mcl(out.encode(), P(code_h), P(v5_h), P(lab_h), int(code_h.size)), "pg_host_write_mcl")


def main(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    inp, out, inflation = None, None, 1.5
    with_value = {"-I", "-o", "-te", "-q", "-V"}
    i = 0
    while i < len(argv):
        a = argv[i]
        if a in with_value:
            if i + 1 >= len(argv):
                raise SystemExit("pangenome_b200.mcl: %s needs a value" % a)
            if a == "-I":
                try:
                    inflation = float(argv[i + 1])
                except ValueError:
                    raise SystemExit("pangenome_b200.mcl: -I needs a number, got %r" % argv[i + 1])
            elif a == "-o":
                out = argv[i + 1]
            i += 2
            continue
        if a == "--abc":
            i += 1
            continue
        if a.startswith("-") and a != "-":
            raise SystemExit("pangenome_b200.mcl: unknown option %s" % a)
        if inp is not None:
            raise SystemExit("pangenome_b200.mcl: more than one input file")
        inp = a
        i += 1
    if inp is None:
        raise SystemExit("usage: python -m pangenome_b200.mcl <file.xyz> --abc -I 1.5 [-o out]")
    if not 1.0 < inflation < 64.0:
        raise SystemExit("pangenome_b200.mcl: -I must be in (1, 64), got %r" % inflation)
    cluster_xyz(inp, out or inp + ".mcl", inflation)
    return 0


if __name__ == "__main__":
    sys.exit(main())
