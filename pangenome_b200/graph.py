"""Host side of K5-K8: path hits, rdBG edges/weights, components, region rows.

Mirrors what the reference's ``seq2graph`` (kmer_numba.py:1853-1951) does after
the rdBG exists, with the external ``mcl`` process replaced by an on-GPU
union-find (connected components of the edge list, optionally restricted to
edges of weight >= ``min_weight``) or, opt-in, by Markov clustering on the GPU
(``cluster="mcl"``, pangenome_b200/mcl.py).  The host only sizes buffers, orders
the (small) cluster list and formats text.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import PgError, PgGraph, check
from .engine import _ptr, _stream, next_pow2


class Hits:
    def __init__(self, g, node, rec, v6, n, strand):
        self.g, self.node, self.rec, self.v6, self.n, self.strand = g, node, rec, v6, n, strand
        self.nslot = torch.empty(max(n, 1), dtype=torch.int32, device=g.device)


def path_hits(packed, rd, n_rec, strand=0, cap=None):
    """K5 over records [0, n_rec) of ``packed`` against the rdBG table ``rd``."""
    L = _lib.load()
    dev = packed.pk2.device
    if n_rec == 0:
        z = torch.empty(1, dtype=torch.int64, device=dev)
        return Hits(z, z, torch.empty(1, dtype=torch.int32, device=dev), torch.empty(1, dtype=torch.int16, device=dev), 0, strand)
    g_begin, g_end = int(packed.seq_off[0]), int(packed.seq_off[n_rec])
    ws_bytes = int(L.pg_path_workspace_bytes(g_end))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    cap = cap or max(1024, (g_end - g_begin) // 8)
    d_n = torch.zeros(1, dtype=torch.int64, device=dev)
    while True:
        hg = torch.empty(cap, dtype=torch.int64, device=dev)
        hn = torch.empty(cap, dtype=torch.int64, device=dev)
        hr = torch.empty(cap, dtype=torch.int32, device=dev)
        hv = torch.empty(cap, dtype=torch.int16, device=dev)
        check(L.pg_path_hits(ctypes.byref(rd.c), _ptr(packed.pk2), _ptr(packed.amb), _ptr(packed.d_seq_off), n_rec,
                             g_begin, g_end, strand, _ptr(hg), _ptr(hn), _ptr(hr), _ptr(hv), cap, _ptr(d_n), _ptr(ws),
                             ws_bytes, _stream()), "pg_path_hits")
        n = int(d_n.item())
        if n <= cap:
            return Hits(hg, hn, hr, hv, n, strand)
        cap = n + 1024


def _no_nodes():
    z = np.zeros(0, np.uint32)
    return z, np.zeros(0, np.uint64), z, np.zeros(0, np.int64)


def dense_order(code, v5):
    """Node order ascending by (code, v5) (device sort): codes are < 5^27 < 2^63, so int64 order is the unsigned order."""
    o1 = torch.argsort(v5, stable=True)
    return o1[torch.argsort(code[o1], stable=True)]


def rank_clusters(code, v5, root):
    """(order, label per node in that order, cluster count): ``order`` = dense_order(code, v5); clusters are ranked
    by (size descending, smallest (code, v5)).  Device sorts only."""
    nn = int(code.numel())
    dev = code.device
    order = dense_order(code, v5)
    if nn == 0:
        return order, torch.zeros(0, dtype=torch.int64, device=dev), 0
    roots_sorted = root[order]
    uniq, inverse, counts = torch.unique(roots_sorted, return_inverse=True, return_counts=True)
    rank = torch.arange(nn, device=dev)
    first_idx = torch.full((uniq.numel(),), nn, dtype=torch.int64, device=dev).scatter_reduce_(0, inverse, rank, "amin")
    c1 = torch.argsort(first_idx, stable=True)
    comp_order = c1[torch.argsort(-counts[c1], stable=True)]          # (size desc, smallest node asc)
    label_of_comp = torch.empty_like(comp_order)
    label_of_comp[comp_order] = torch.arange(uniq.numel(), device=dev)
    return order, label_of_comp[inverse], int(uniq.numel())          # labels per node, in (code, v5) order


class RdbgGraph:
    """Device node/edge/visit tables (pg_graph) + the host read-outs."""

    def __init__(self, n_hits_total, device):
        self.L = _lib.load()
        cap = next_pow2(max(1024, 2 * n_hits_total + 2))
        if cap > 1 << 32:
            raise PgError("more than 2^31 hits: shard the input across GPUs")
        self.cap = cap
        i64, i32 = torch.int64, torch.int32
        self.node_keys = torch.empty(cap, dtype=i64, device=device)
        self.node_parent = torch.empty(cap, dtype=i32, device=device)
        self.node_label = torch.empty(cap, dtype=i32, device=device)
        self.edge_keys = torch.empty(cap, dtype=i64, device=device)
        self.edge_w = torch.empty(cap, dtype=i32, device=device)
        self.edge_first = torch.empty(cap, dtype=i64, device=device)
        self.visit_keys = torch.empty(cap, dtype=i64, device=device)
        self.stats = torch.zeros(8, dtype=i64, device=device)
        self.c = PgGraph(self.node_keys.data_ptr(), self.node_parent.data_ptr(), self.node_label.data_ptr(),
                         self.edge_keys.data_ptr(), self.edge_w.data_ptr(), self.edge_first.data_ptr(),
                         self.visit_keys.data_ptr(), self.stats.data_ptr(), cap, cap, cap)
        check(self.L.pg_graph_clear(ctypes.byref(self.c), _stream()), "pg_graph_clear")

    def add_hits(self, hits, n_strands):
        check(self.L.pg_graph_add_hits(ctypes.byref(self.c), _ptr(hits.node), _ptr(hits.rec), hits.n, _ptr(hits.nslot),
                                       hits.strand, n_strands, _stream()), "pg_graph_add_hits")

    def counts(self):
        s = self.stats.cpu().numpy()
        if s[0]:
            raise PgError("graph table overflow")
        return int(s[1]), int(s[2])

    def edges(self, rd):
        """(c0, v0, c1, v1, w) sorted into the reference's .xyz file order
        (first-insertion order of the edge dict).  The sort runs on the device."""
        _, ne = self.counts()
        dev = self.stats.device
        c0 = torch.empty(max(ne, 1), dtype=torch.int64, device=dev)
        c1 = torch.empty_like(c0)
        first = torch.empty_like(c0)
        v0 = torch.empty(max(ne, 1), dtype=torch.int32, device=dev)
        v1 = torch.empty_like(v0)
        w = torch.empty_like(v0)
        d_n = torch.zeros(1, dtype=torch.int64, device=dev)
        check(self.L.pg_graph_export_edges(ctypes.byref(self.c), ctypes.byref(rd.c), _ptr(c0), _ptr(v0), _ptr(c1), _ptr(v1),
                                           _ptr(w), _ptr(first), ne, _ptr(d_n), _stream()), "pg_graph_export_edges")
        assert int(d_n.item()) == ne
        order = torch.argsort(first[:ne], stable=True)        # ordinals are < 2^63: signed order == unsigned order
        f = lambda t, dt: t[:ne][order].cpu().numpy().view(dt)
        return f(c0, np.uint64), f(v0, np.uint32), f(c1, np.uint64), f(v1, np.uint32), f(w, np.uint32)

    def components(self, rd, min_weight=1, to_host=True):
        """K7 + cluster ordering.  Returns (nslot, code, v5, label) per graph node; label = rank
        of the node's component under (size descending, smallest (code, v5)).  The union-find is
        a kernel; the ordering uses device sorts; labels are written to the node table directly."""
        check(self.L.pg_graph_components(ctypes.byref(self.c), int(min_weight), _stream()), "pg_graph_components")
        nodes = self._export_nodes(rd)
        if nodes is None:
            return _no_nodes()
        nslot, code, v5, root = nodes
        return self._label(nslot, code, v5, root, to_host)

    def mcl(self, rd, min_weight=1, inflation=1.5, to_host=True):
        """K7m: Markov clustering (pangenome_b200/mcl.py) of the live edges (node slot a, node slot b, weight), nodes
        numbered densely in (code, v5) order.  Returns what components() returns; the run's per-iteration
        statistics stay in ``self.mcl_result``."""
        from . import mcl
        nodes = self._export_nodes(rd)
        if nodes is None:
            return _no_nodes()
        nslot, code, v5, _ = nodes
        nn = int(nslot.numel())
        order = dense_order(code, v5)
        dense = torch.full((self.cap,), -1, dtype=torch.int64, device=nslot.device)
        dense[nslot[order]] = torch.arange(nn, device=nslot.device)
        ek = self.edge_keys
        live = ek != -1                                                   # PG_EMPTY
        ek = ek[live]
        a, b = dense[(ek >> 32) & 0xFFFFFFFF], dense[ek & 0xFFFFFFFF]
        w = self.edge_w[live].long()                                      # uint32 weights in an int32 tensor: < 2^31
        self.mcl_result = mcl.markov_cluster(nn, a, b, w, inflation, min_weight)
        root = torch.empty(nn, dtype=torch.int64, device=nslot.device)
        root[order] = self.mcl_result.root.long()
        return self._label(nslot, code, v5, root, to_host)

    def _export_nodes(self, rd):
        """(nslot, code, v5, union-find parent) of the nodes that appear in an edge, or None when there is none;
        every node label is reset to -1."""
        nn, _ = self.counts()
        dev = self.stats.device
        nslot = torch.empty(max(nn, 1), dtype=torch.int32, device=dev)
        code = torch.empty(max(nn, 1), dtype=torch.int64, device=dev)
        v5 = torch.empty(max(nn, 1), dtype=torch.int32, device=dev)
        root = torch.empty(max(nn, 1), dtype=torch.int32, device=dev)
        d_n = torch.zeros(1, dtype=torch.int64, device=dev)
        check(self.L.pg_graph_export_nodes(ctypes.byref(self.c), ctypes.byref(rd.c), _ptr(nslot), _ptr(code), _ptr(v5),
                                           _ptr(root), nn, _ptr(d_n), _stream()), "pg_graph_export_nodes")
        nn = int(d_n.item())          # nodes that appear in at least one edge (<= inserted node slots)
        self.node_label.fill_(-1)
        if nn == 0:
            return None
        return nslot[:nn].long(), code[:nn], v5[:nn].long(), root[:nn].long()

    def _label(self, nslot, code, v5, root, to_host):
        """Label every node with the rank of its cluster (``root`` = any id shared by exactly the nodes of one
        cluster) and write the labels into the node table."""
        order, label_sorted, self.n_components = rank_clusters(code, v5, root)
        self.node_label.index_put_((nslot[order],), label_sorted.to(torch.int32))
        if not to_host:
            return None
        # host copies, sorted by (label, code, v5) - the order the cluster file is written in
        o3 = torch.argsort(label_sorted, stable=True)
        fin = order[o3]
        return (nslot[fin].cpu().numpy().astype(np.uint32), code[fin].cpu().numpy().view(np.uint64),
                v5[fin].cpu().numpy().astype(np.uint32), label_sorted[o3].cpu().numpy())

    def set_labels(self, nslot, label):
        """Upload one label per graph node; every other node slot gets -1 (never matches in K8)."""
        self.node_label.fill_(-1)
        if nslot.size:
            idx = torch.from_numpy(nslot.astype(np.int64)).to(self.node_label.device)
            val = torch.from_numpy(label.astype(np.int32)).to(self.node_label.device)
            self.node_label.index_put_((idx,), val)

    def regions(self, hits, packed, k):
        """K8 for one strand: rows (rec, start, end, label) in walk order."""
        L = self.L
        dev = self.stats.device
        if hits.n == 0:
            return np.zeros(0, np.int32), np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0, np.int32)
        ws_bytes = int(L.pg_label_workspace_bytes(hits.n))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        cap = hits.n
        rr = torch.empty(cap, dtype=torch.int32, device=dev)
        re_ = torch.empty(cap, dtype=torch.int64, device=dev)
        rl = torch.empty(cap, dtype=torch.int32, device=dev)
        d_n = torch.zeros(2, dtype=torch.int64, device=dev)
        check(L.pg_label_regions(ctypes.byref(self.c), _ptr(hits.g), _ptr(hits.node), _ptr(hits.rec), _ptr(hits.v6), hits.n,
                                 _ptr(packed.d_seq_off), k, hits.strand, _ptr(rr), _ptr(re_), _ptr(rl), cap, _ptr(d_n),
                                 _ptr(ws), ws_bytes, _stream()), "pg_label_regions")
        n = int(d_n[0].item())
        rec = rr[:n].cpu().numpy()
        end = re_[:n].cpu().numpy()
        lab = rl[:n].cpu().numpy()
        start = np.zeros(n, np.int64)
        if n > 1:
            same = rec[1:] == rec[:-1]
            start[1:][same] = end[:-1][same]
        return rec, start, end, lab


class GraphResult:
    def __init__(self):
        self.edges = None
        self.nodes = None
        self.rows_raw = []          # list of (rec, start, end, strand_sign, label) arrays per strand

    def xyz_lines(self):
        c0, v0, c1, v1, w = self.edges
        return ["%d_%d\t%d_%d\t%d" % t for t in zip(c0.tolist(), v0.tolist(), c1.tolist(), v1.tolist(), w.tolist())]

    def write_xyz(self, path):
        """<qry>_rdbg_weight.xyz (kmer_numba.py:1893-1904) through the C++ writer of libpgdbg."""
        c0, v0, c1, v1, w = [np.ascontiguousarray(x) for x in self.edges]
        L = _lib.load()
        P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        check(L.pg_host_write_xyz(path.encode(), P(c0), P(v0), P(c1), P(v1), P(w), int(c0.size)), "pg_host_write_xyz")

    def write_mcl(self, path):
        """The cluster file (what `mcl -o` leaves, :1911): one line of node names per component."""
        nslot, code, v5, label = self.nodes
        label = label.astype(np.int64)
        if label.size > 1 and not (np.all(label[1:] >= label[:-1])):      # components() already delivers (label, code, v5) order
            order = np.lexsort((v5, code, label))
            code, v5, label = code[order], v5[order], label[order]
        code, v5, label = [np.ascontiguousarray(x) for x in (code, v5, label)]
        L = _lib.load()
        P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        check(L.pg_host_write_mcl(path.encode(), P(code), P(v5), P(label), int(code.size)), "pg_host_write_mcl")

    def mcl_lines(self):
        """One line per component, like the cluster file the reference reads (:1918-1929)."""
        nslot, code, v5, label = self.nodes
        order = np.lexsort((v5, code, label))
        lines, cur, lab_prev = [], [], None
        for c, v, l in zip(code[order].tolist(), v5[order].tolist(), label[order].tolist()):
            if l != lab_prev and cur:
                lines.append("\t".join(cur))
                cur = []
            cur.append("%d_%d" % (c, v))
            lab_prev = l
        if cur:
            lines.append("\t".join(cur))
        return lines

    def rows(self, packed, data):
        """[(seqid, start, end, strand, label)] in the reference's print order:
        per record, forward rows then rc rows mirrored to (n-end, n-start, '-')."""
        ids = packed.ids if data is None else record_ids(packed, data)     # a multi-GPU global index brings its ids
        lens = packed.seq_lengths
        parts = []
        for rec, start, end, sign, lab in self.rows_raw:
            rec = np.asarray(rec, dtype=np.int64)
            if rec.size == 0:
                continue
            start, end, lab = np.asarray(start, np.int64), np.asarray(end, np.int64), np.asarray(lab, np.int64)
            if sign > 0:
                parts.append((rec, np.zeros(rec.size, np.int64), start, end, lab))
            else:
                n = lens[rec].astype(np.int64)
                parts.append((rec, np.ones(rec.size, np.int64), n - end, n - start, lab))
        if not parts:
            return []
        rec, strand, start, end, lab = [np.concatenate(c) for c in zip(*parts)]
        order = np.lexsort((np.arange(rec.size), strand, rec))             # stable: walk order inside a record-strand
        sym = ("+", "-")
        return [(ids[r], s, e, sym[d], l) for r, d, s, e, l in
                zip(rec[order].tolist(), strand[order].tolist(), start[order].tolist(), end[order].tolist(), lab[order].tolist())]


def record_ids(packed, data):
    """seqid = header line minus '>' and minus its last byte (kmer_numba.py:156, 1947).  ``data``: bytes or a uint8
    array (np.memmap of the input file); header ends are found with windowed vector searches, never by scanning the file."""
    a = np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray, memoryview)) else np.asarray(data)
    offs = np.asarray(packed.hdr_off, dtype=np.int64)
    n = int(a.size)
    ends = np.empty(offs.size, dtype=np.int64)
    W, B = 128, 1 << 15
    win = np.arange(W, dtype=np.int64)[None, :]
    for lo in range(0, offs.size, B):
        o = offs[lo:lo + B]
        nl = a[np.minimum(o[:, None] + win, n - 1)] == 10
        has = nl.any(axis=1)
        e = np.where(has, o + nl.argmax(axis=1), -1)
        for j in np.nonzero(~has)[0].tolist():      # a header longer than the window: chunked search
            p, found = int(o[j]) + W, -1
            while p < n and found < 0:
                hit = np.nonzero(a[p:p + (1 << 16)] == 10)[0]
                found = p + int(hit[0]) if hit.size else -1
                p += 1 << 16
            e[j] = found
        ends[lo:lo + B] = e
    ends[ends < 0] = n - 1                           # Q8: the final line loses its last byte even without a newline
    return [bytes(a[o + 1:e]).decode("utf-8", errors="replace") for o, e in zip(offs.tolist(), ends.tolist())]


def labels_from_mcl(lines, xyz_edges):
    """label_dct as the reference builds it from a cluster file (:1916-1944): cluster line index,
    then fresh labels for nodes of the .xyz missing from it, scanning column 1 then column 2."""
    lab = {}
    flag = 0
    for line in lines:
        for name in line.rstrip("\n").split("\t"):
            if not name:
                continue
            a, b = name.split("_")[:2]
            lab[(int(a), int(b))] = flag
        flag += 1
    c0, v0, c1, v1, _ = xyz_edges
    for a, b, c, d in zip(c0.tolist(), v0.tolist(), c1.tolist(), v1.tolist()):
        if (a, b) not in lab:
            lab[(a, b)] = flag
            flag += 1
        if (c, d) not in lab:
            lab[(c, d)] = flag
            flag += 1
    return lab


def cluster_nodes(g, rd, min_weight=1, cluster="components", inflation=1.5):
    """(nslot, code, v5, label) per graph node under the chosen clustering: "components" (K7, the default) or "mcl"
    (K7m, Markov clustering with inflation ``inflation``)."""
    if cluster == "components":
        return g.components(rd, min_weight)
    if cluster == "mcl":
        return g.mcl(rd, min_weight, inflation)
    raise ValueError("cluster must be 'components' or 'mcl', got %r" % (cluster,))


def seq2graph_device(packed, rd, k, Ns=2 ** 63, rc=False, min_weight=1, mcl_lines=None, cluster="components", inflation=1.5):
    """Stages 3-5 on the GPU.  ``rd`` = rdBG table from DbgTable.select_rdbg().  ``cluster``: "components" or "mcl"
    (see cluster_nodes); an externally produced cluster file (``mcl_lines``) overrides either."""
    k = int(min(max(1, k), 27))
    n_rec = packed.record_prefix(Ns, 1)
    n_strands = 2 if rc else 1
    hits = [path_hits(packed, rd, n_rec, s) for s in range(n_strands)]
    total = sum(h.n for h in hits)
    g = RdbgGraph(total, packed.pk2.device)
    for h in hits:
        g.add_hits(h, n_strands)
    res = GraphResult()
    res.edges = g.edges(rd)
    nslot, code, v5, label = cluster_nodes(g, rd, min_weight, cluster if mcl_lines is None else "components", inflation)
    if mcl_lines is not None:      # an externally produced cluster file wins (the "# the mcl has been ran" path)
        lab = labels_from_mcl(mcl_lines, res.edges)
        label = np.array([lab[(c, v)] for c, v in zip(code.tolist(), v5.tolist())], dtype=np.int64)
    res.nodes = (nslot, code, v5, label)
    if mcl_lines is not None:
        g.set_labels(nslot, label)
    for h in hits:
        rec, start, end, lab_ = g.regions(h, packed, k)
        res.rows_raw.append((rec, start, end, 1 if h.strand == 0 else -1, lab_))
    res.n_hits = total
    res.graph = g
    return res
