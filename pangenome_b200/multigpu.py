"""Multi-GPU plumbing around the streaming builder (pangenome_b200/builder.py; one process per GPU,
``torch.distributed``; NCCL over NVLink on the GPU box, gloo in the CPU tests).

The reference has no distributed path; this is the split SURVEY.md 8(e) prescribes.  The dBG build itself
(records bucketed by owner rank and stored into the owners' receive buffers over NVLink, receiver-side split
into table regions, region sweep) lives in builder.RoundBuilder.  Here: the merged read-out of the
hash-partitioned table, and stages 2-5 on it -

  * every key lives on exactly one rank, so tables never need merging; the merged export is the
    concatenation of the ranks' exports (the short-record sentinel is summed).  Count saturation happens at
    export, after all occurrences of a key - from every rank - were added on its owner (SURVEY 8e "result
    invariance");
  * rdBG selection is local to the keys a rank owns; the small per-rank rdBG tables are all-gathered so every
    rank holds the full membership table; path hits (K5) run on each rank's own records; the hits (a few % of
    the positions) are gathered in rank-independent form and rank 0 runs K6-K8 on them.
"""
import ctypes
import os

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from .builder import log2_exact  # noqa: F401  (re-exported: the host tests and older callers import it from here)


def gather_export(table, world, rank):
    """Merged (keys, vals, cnts) of the distributed dBG on rank 0 (test / small outputs only)."""
    k, v, c = table.export(sort=False)
    short = int(table.stats_host()[_lib.PG_STAT_SHORT])
    sent = np.uint64(0xFFFFFFFFFFFFFFFF)
    keep = k != sent                               # the sentinel is merged separately
    k, v, c = k[keep], v[keep], c[keep]
    if world == 1:
        parts, shorts = [(k, v, c)], [short]
    else:
        parts, shorts = [None] * world, [None] * world
        dist.all_gather_object(parts, (k, v, c))
        dist.all_gather_object(shorts, short)
    if rank != 0:
        return None
    K = np.concatenate([p[0] for p in parts])
    V = np.concatenate([p[1] for p in parts])
    C = np.concatenate([p[2] for p in parts])
    tot_short = sum(shorts)
    if tot_short > 0:
        K = np.append(K, sent)
        V = np.append(V, np.uint16(32))
        C = np.append(C, np.uint8(min(tot_short, 255)))
    o = np.argsort(K, kind="stable")
    return K[o], V[o], C[o]


_PAIR_GROUPS = {}
GATHER_PIECE = 64 << 20       # bytes one rank sends to rank 0 per broadcast


def _pair_groups(world):
    """The process groups {0, r}, r = 1 .. world - 1: a broadcast from r inside one reaches rank 0 alone, for NCCL and
    for gloo on CUDA tensors alike (gloo has no point-to-point or gather for CUDA tensors).  Collective: every rank
    creates every pair, in order, once per default group."""
    key = (id(dist.group.WORLD), world)
    if key not in _PAIR_GROUPS:
        _PAIR_GROUPS[key] = [None] + [dist.new_group([0, q]) for q in range(1, world)]
    return _PAIR_GROUPS[key]


def gather_entries_rank0(table, world, rank, fits=None):
    """The distributed dBG's entries on rank 0 only, moved as device tensors (sizes first, then each rank's bytes in
    pieces of GATHER_PIECE): each rank drops its short-record sentinel and rank 0 adds one whose count is the sum over
    ranks, clamped to 255 (the rule of gather_export).  ``fits(n)``: rank 0's choice, given the number of entries,
    between device arrays (True) and host arrays received through a device bounce buffer (False).
    Returns on rank 0 (on_device, keys, vals, cnts) - int64 / int16 / uint8 tensors, or u64 / u16 / u8 numpy arrays -
    and None elsewhere."""
    k, v, c = table.export_device()
    dev = k.device
    keep = k != -1
    k, v, c = k[keep], v[keep], c[keep]
    short = int(table.stats_host()[_lib.PG_STAT_SHORT])
    mine = torch.tensor([k.numel(), short], dtype=torch.int64, device=dev)
    sizes = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(sizes, mine)
    ns = [int(s[0]) for s in sizes]
    tot_short = sum(int(s[1]) for s in sizes)
    total = sum(ns) + (1 if tot_short > 0 else 0)
    parts = [(k, 8), (v, 2), (c, 1)]
    groups = _pair_groups(world)
    if rank == 0:
        on_dev = True if fits is None else bool(fits(total))
        if on_dev:
            out = [torch.empty(total, dtype=t.dtype, device=dev) for t, _ in parts]
        else:
            out = [torch.from_numpy(np.empty(total, dtype=d)) for d in (np.int64, np.int16, np.uint8)]
        for o, (t, _) in zip(out, parts):
            o[:ns[0]].copy_(t)
        bounce = None if on_dev else torch.empty(GATHER_PIECE, dtype=torch.uint8, device=dev)
    for r in range(1, world):
        if rank not in (0, r):
            continue
        g = groups[r]
        base = sum(ns[:r])
        for i, (t, width) in enumerate(parts):
            step = GATHER_PIECE // width
            for a in range(0, ns[r], step):
                m = min(step, ns[r] - a)
                if rank == r:
                    dist.broadcast(t[a:a + m].view(torch.uint8), src=r, group=g)
                elif on_dev:
                    dist.broadcast(out[i][base + a:base + a + m].view(torch.uint8), src=r, group=g)
                else:
                    buf = bounce[:m * width]
                    dist.broadcast(buf, src=r, group=g)
                    out[i][base + a:base + a + m].view(torch.uint8).copy_(buf.cpu())
    if rank != 0:
        return None
    if tot_short > 0:
        out[0][-1], out[1][-1], out[2][-1] = -1, 32, min(tot_short, 255)
    if on_dev:
        return True, out[0], out[1], out[2]
    return False, out[0].numpy().view(np.uint64), out[1].numpy().view(np.uint16), out[2].numpy()


def dump_rank0(table, world, rank, fn, budget=None):
    """``<fn>.npz`` of the distributed dBG, written by rank 0 (other ranks return None after a barrier).  The entries
    are gathered to rank 0 (gather_entries_rank0); rank 0 writes the image on the GPU when its free device memory (or
    ``budget`` bytes) holds the gathered entries, the image and the encoder's slab pair, else on the host from the same
    gather, and says so on stderr.  The file is the one the same entries give on one GPU."""
    import sys
    from . import npz
    dev = table.slots.device

    def fits(n):
        room = budget if budget is not None else torch.cuda.mem_get_info(dev)[0]
        return 11 * n + npz.device_bytes_needed(n) <= room

    got = gather_entries_rank0(table, world, rank, fits)
    out = None
    if rank == 0:
        on_dev, k, v, c = got
        if on_dev:
            out = npz.dump_device(k, v, c, fn)
        else:
            print("pangenome_b200: %d dBG entries do not fit rank 0's free device memory next to their image: "
                  "writing %s.npz on the host" % (k.size, fn), file=sys.stderr)
            out = npz.dump_entries(k, v, c, fn)
    dist.barrier()
    return out


def gather_varlen(t, world):
    """Concatenation over ranks of 1-D tensors of different lengths (padded all_gather).
    Returns (concatenated tensor, per-rank lengths)."""
    if world == 1:
        return t, [int(t.numel())]
    n = torch.tensor([t.numel()], dtype=torch.int64, device=t.device)
    sizes = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(sizes, n)
    sizes = [int(x.item()) for x in sizes]
    m = max(max(sizes), 1)
    pad = torch.zeros(m, dtype=t.dtype, device=t.device)
    pad[:t.numel()] = t
    parts = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad)
    return torch.cat([p[:sz] for p, sz in zip(parts, sizes)]), sizes


class _GlobalIndex:
    """What graph.RdbgGraph.regions / GraphResult.rows need from a PackedSeqs, for the records of all ranks."""

    def __init__(self, seq_off, hdr_ids, device):
        self.seq_off = seq_off
        self.d_seq_off = torch.from_numpy(seq_off).to(device)
        self.ids = hdr_ids

    @property
    def seq_lengths(self):
        return np.diff(self.seq_off)


def seq2graph_distributed(packed, table, k, world, rank, data, rc=False, min_weight=1, n_rec=None, mcl_lines=None,
                          cluster="components", inflation=1.5):
    """Stages 2-5 after a distributed dBG build (SURVEY 8e): every rank selects the rdBG members
    among ITS keys, the small rdBG tables are all-gathered into one full table per rank, each rank
    walks its own records (K5), the hits (a few % of the positions) are gathered in rank-independent
    form (record, position, literal code, v5, v6) and rank 0 runs K6-K8 on them (with the clustering
    ``cluster`` / ``inflation`` of graph.cluster_nodes).
    Returns (GraphResult, rows) on rank 0 and (None, None) elsewhere."""
    from . import engine, graph
    L = _lib.load()
    dev = table.slots.device
    chk, P, S = engine.check, engine._ptr, engine._stream
    n_rec = packed.n_rec if n_rec is None else n_rec          # this rank's records the path stages walk (-n)
    # ---- rdBG: local select, all-gather of the raw slots, full table on every rank
    rd_local = table.select_rdbg()
    n_loc = rd_local.n_slots_used
    keys = torch.empty(max(n_loc, 1), dtype=torch.int64, device=dev)
    vals = torch.empty(max(n_loc, 1), dtype=torch.int64, device=dev)
    d_n = torch.zeros(1, dtype=torch.int64, device=dev)
    chk(L.pg_table_export_raw(ctypes.byref(rd_local.c), P(keys), P(vals), n_loc, P(d_n), S()), "pg_table_export_raw")
    assert int(d_n.item()) == n_loc
    K_all, _ = gather_varlen(keys[:n_loc], world)
    V_all, _ = gather_varlen(vals[:n_loc], world)
    rd = engine.DbgTable(max(1024, 2 * int(K_all.numel()) + 2), table.k, table.mode, device=dev)
    chk(L.pg_table_insert_raw(ctypes.byref(rd.c), P(K_all), P(V_all), int(K_all.numel()), S()), "pg_table_insert_raw")
    short = table.stats[_lib.PG_STAT_SHORT:_lib.PG_STAT_SHORT + 1].clone()
    if world > 1:
        dist.all_reduce(short, op=dist.ReduceOp.SUM)
    rd.stats[_lib.PG_STAT_SHORT] = short[0]
    members = torch.tensor([rd_local.n_members - (1 if int(table.stats_host()[_lib.PG_STAT_SHORT]) > 0 else 0)],
                           dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(members, op=dist.ReduceOp.SUM)
    rd.n_members = int(members.item()) + (1 if int(short.item()) > 0 else 0)
    if rd.overflowed():
        raise _lib.PgError("rdBG table overflow")
    # ---- record index of all ranks (host objects: small)
    lens_all, ids_all = [None] * world, [None] * world
    my_ids = graph.record_ids(packed, data)
    if world > 1:
        dist.all_gather_object(lens_all, packed.seq_lengths[:n_rec].tolist())
        dist.all_gather_object(ids_all, my_ids[:n_rec])
    else:
        lens_all, ids_all = [packed.seq_lengths[:n_rec].tolist()], [my_ids[:n_rec]]
    rec_base = sum(len(x) for x in lens_all[:rank])
    g_seq_off = np.concatenate([[0], np.cumsum(np.concatenate([np.asarray(x, dtype=np.int64) for x in lens_all]))]).astype(np.int64)
    gidx = _GlobalIndex(g_seq_off, [i for ids in ids_all for i in ids], dev)
    # ---- K5 on the local records, hits to rank-independent form, gather
    n_strands = 2 if rc else 1
    all_hits = []
    for strand in range(n_strands):
        h = graph.path_hits(packed, rd, n_rec, strand)
        n = h.n
        code = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
        chk(L.pg_hits_decode(ctypes.byref(rd.c), P(h.node), n, P(code), S()), "pg_hits_decode")
        rec = h.rec[:n].long()
        pos = h.g[:n] - packed.d_seq_off[:packed.n_rec + 1][rec] if n else h.g[:0]
        v5 = (h.node[:n] & 2047).to(torch.int32)
        g_code, _ = gather_varlen(code[:n], world)
        g_pos, _ = gather_varlen(pos, world)
        g_rec, _ = gather_varlen(rec + rec_base, world)
        g_v5, _ = gather_varlen(v5, world)
        g_v6, _ = gather_varlen(h.v6[:n].to(torch.int32), world)      # NCCL has no int16
        all_hits.append((g_code, g_pos, g_rec, g_v5, g_v6))
    if rank != 0:
        return None, None
    # ---- rank 0: re-key against its own rdBG table and run K6-K8 exactly like the single-GPU path
    hits = []
    for strand, (g_code, g_pos, g_rec, g_v5, g_v6) in enumerate(all_hits):
        n = int(g_code.numel())
        node = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
        chk(L.pg_hits_rekey(ctypes.byref(rd.c), P(g_code), P(g_v5.contiguous()), n, P(node), S()), "pg_hits_rekey")
        gg = gidx.d_seq_off[g_rec] + g_pos if n else g_pos
        hits.append(graph.Hits(gg.contiguous(), node, g_rec.to(torch.int32).contiguous(), g_v6.to(torch.int16).contiguous(), n, strand))
    total = sum(h.n for h in hits)
    g = graph.RdbgGraph(total, dev)
    for h in hits:
        g.add_hits(h, n_strands)
    res = graph.GraphResult()
    res.edges = g.edges(rd)
    res.nodes = graph.cluster_nodes(g, rd, min_weight, cluster if mcl_lines is None else "components", inflation)
    if mcl_lines is not None:      # an externally produced cluster file wins (the "# the mcl has been ran" path, :1908)
        nslot, code, v5, _ = res.nodes
        lab = graph.labels_from_mcl(mcl_lines, res.edges)
        label = np.array([lab[(c, v)] for c, v in zip(code.tolist(), v5.tolist())], dtype=np.int64)
        res.nodes = (nslot, code, v5, label)
        g.set_labels(nslot, label)
    for h in hits:
        rec, start, end, lab = g.regions(h, gidx, table.k)
        res.rows_raw.append((rec, start, end, 1 if h.strand == 0 else -1, lab))
    res.graph = g
    res.rdbg = rd
    rows = res.rows(gidx, None)
    return res, rows
