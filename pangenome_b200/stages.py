"""The reference's stage API on the B200 path: ``seq2rdbg``, ``dbg2rdbg``,
``seq2graph`` (kmer_numba.py:1234-1268, 1313-1321, 1853-1951) with the same
argument meaning.  ``seq2graph`` prints the table rows on stdout and writes
``<qry>_rdbg_weight.xyz`` (+ ``.mcl``) beside the input, like the reference.
"""
import os
import sys

import numpy as np

from . import _lib, engine, graph


class DbgHandle:
    """What seq2rdbg returns: the device table plus the packed sequences it was
    built from (later stages reuse them instead of re-reading the file).  ``world`` / ``rank``: the
    hash-partitioned table of a multi-GPU run (this rank's keys, this rank's records)."""

    def __init__(self, table, packed, data, n_rec, world=1, rank=0, builder=None):
        self.table, self.packed, self.data, self.n_rec = table, packed, data, n_rec
        self.world, self.rank, self.builder = world, rank, builder


def _read(qry):
    """(host bytes, device bytes) of the whole input, decompressed when it is gzip / BGZF (seqfile.load).  Plain FASTA
    stays a read-only np.memmap on the host: nothing is copied there, the H2D copy streams straight out of the mapping."""
    from . import seqfile
    return seqfile.load(qry)


def _dist_env():
    """(world, rank) when launched under torchrun with more than one rank, else (1, 0)."""
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            return dist.get_world_size(), dist.get_rank()
    except ImportError:
        pass
    return 1, 0


def seq_chk(qry):
    """kmer_numba.py:873-886: peek 40 bytes, '>' anywhere at a line start -> fasta; but '@' as the first byte -> fastq
    (seqfile.detect).  The bytes are those of the decompressed stream when the file is gzip / BGZF compressed."""
    from . import seqfile
    return seqfile.input_format(qry)


def _pack(qry, d_bytes, fmt, begin=0, world=1):
    """PackedSeqs of the device bytes.  A malformed FASTQ exits naming the byte offset (in the decompressed input) of its
    first bad record; ``begin`` = where this rank's range starts.  Under torchrun every rank learns whether any range was
    malformed, so all of them stop before the first collective of the build."""
    err = None
    try:
        packed = engine.PackedSeqs(d_bytes, fmt=fmt)
    except engine.FastqError as e:
        packed, err = None, (begin + e.offset, e.reason)
    if world > 1 and fmt == "fastq":
        import torch.distributed as dist
        errs = [None] * world
        dist.all_gather_object(errs, err)
        err = min((e for e in errs if e is not None), default=None)
    if err is not None:
        raise SystemExit("pangenome_b200: %s: malformed FASTQ: the record at byte %d: %s" % (qry, err[0], err[1]))
    return packed


def seq2rdbg(qry, kmer=13, bits=5, Ns=1e6, chunk=2 ** 32, brkpt="./breakpoint", saved="dBG_disk", hashfunc=None,
             jit=True, rc=True, data=None):
    """Stage 1: build the dBG (both strands when ``rc``).

    Chunk checkpoints as upstream (:1252-1266): whenever a call has consumed more than ``chunk`` bases
    (both strands counted) the table is written to ``<qry>_db_brkpt.npz`` together with the byte offset
    of the next header line; an existing ``brkpt`` file (``-r``) is loaded and the build resumes at its
    offset.  Inputs below ``chunk`` with no ``brkpt`` file take the one-shot two-phase build.

    A FASTQ input gives what the FASTA of its header and sequence lines gives, and always takes the one-shot build:
    the checkpoint loop and its offsets are those of the reference's FASTA reader, so resuming from ``brkpt`` exits."""
    if bits != 5:
        raise ValueError("only the reference's base-5 code (bits=5) is supported")
    kmer = min(max(1, int(kmer)), 27)
    world, rank = _dist_env()
    d_bytes, fmt, begin = None, "fasta", 0
    resume = bool(brkpt) and os.path.isfile(brkpt)
    if data is None:
        fmt = seq_chk(qry)
        if fmt not in ("fasta", "fastq"):
            raise SystemExit("pangenome_b200: %s is neither FASTA nor FASTQ" % qry)
        if fmt == "fastq" and resume:
            raise SystemExit("pangenome_b200: -r (dBG checkpoint resume) reads FASTA only; %s is FASTQ" % qry)
        if world > 1:      # this rank's record-aligned byte range of the one file (SURVEY 8e)
            from . import shard
            data, (begin, _), _ = shard.read_rank_range(qry, world, rank)
            data = np.frombuffer(data, dtype=np.uint8)
        else:
            data, d_bytes = _read(qry)
    packed = _pack(qry, d_bytes if d_bytes is not None else engine.to_device_bytes(data), fmt, begin, world)
    strands = 2 if rc else 1
    from . import builder
    if world > 1:
        if resume:
            raise SystemExit("pangenome_b200: -r (dBG checkpoint resume) runs on one GPU; launch without torchrun")
        table, n_rec, b = builder.build_table(packed, kmer, rc=bool(rc), Ns=Ns, world=world, rank=rank)
        return DbgHandle(table, packed, data, n_rec, world, rank, b)
    if fmt == "fastq" or (not resume and strands * int(packed.n_bases) <= chunk):
        # the streaming two-phase build (K2a partition + K3 region sweep): what bench.py times
        table, n_rec, b = builder.build_table(packed, kmer, rc=bool(rc), Ns=Ns)
        return DbgHandle(table, packed, data, n_rec, builder=b)
    raw = data.tobytes() if isinstance(data, np.ndarray) else bytes(data)
    table = _build_chunked(qry, raw, packed, kmer, Ns, chunk, brkpt if resume else None, bool(rc))
    return DbgHandle(table, packed, data, packed.n_rec)


def plan_chunks(lens, chunk, Ns):
    """The record ranges the ``while 1`` loop of seq2rdbg (:1252-1266) hands to seq2dbg_jit_ (:1202-1230):
    yields (first record, end record, checkpoint written afterwards?, tail?).  ``lens`` = bases per record
    with both strands counted when rc.  ``tail`` marks the extra call upstream makes after a checkpoint that
    fell on the last record: it parses again from the file's last line and finds no sequence.  Inside a call N and chk restart at 0 and the chunk test comes before
    the -n test (:1224-1228); after a checkpoint the call's N joins a running total that ends the loop
    once it exceeds Ns (:1263-1265)."""
    n_rec, r, total = len(lens), 0, 0
    while True:
        N = chk = 0
        r0, done = r, 1
        while r < n_rec:
            N += int(lens[r])
            chk += int(lens[r])
            r += 1
            if chk > chunk:
                done = -1
                break
            if N > Ns:
                break
        yield r0, r, done == -1, False
        if done != -1:
            return
        total += N
        if total > Ns:
            return
        if r >= n_rec:
            yield r, r, False, True
            return


def _last_line_start(raw):
    """Byte offset of the last line readline_jit_ (:122-132) yields."""
    end = len(raw) - 1 if raw.endswith(b"\n") else len(raw)
    return raw.rfind(b"\n", 0, max(end, 0)) + 1


def _build_chunked(qry, raw, packed, kmer, Ns, chunk, brkpt, rc):
    """The ``while 1`` loop of seq2rdbg (:1252-1266) around seq2dbg_jit_ (:1202-1230)."""
    from . import npz
    strands = 2 if rc else 1
    mode = _lib.PG_MODE_LITERAL_RC if rc else _lib.PG_MODE_LITERAL      # checkpoint images hold literal keys
    p, shift = packed, 0               # records still to insert, and what to add to their header offsets
    if brkpt is None:
        table = engine.DbgTable(int(strands * packed.n_positions(kmer) / 0.5) + 1024, kmer, mode, device=packed.pk2.device)
    else:
        offset = int(np.load(brkpt)["parameters"][5])
        # readline_jit_ with an offset: the first "line" runs from byte 0 to the first newline at or after
        # ``offset``; starting with '>' it is taken for a header, so the record resumes right after it
        nl = raw.find(b"\n", offset)
        rest = raw[nl + 1:] if nl >= 0 else None
        if rest is None:
            p = None
        else:
            pre = b">\n" if raw[:1] == b">" else b""       # a file not starting with '>': those lines belong to no record
            p = engine.PackedSeqs(engine.to_device_bytes(pre + rest))
            shift = nl + 1 - len(pre)
        n_more = strands * p.n_positions(kmer) if p is not None else 0
        _, table = npz.load(brkpt, kmer, device=packed.pk2.device, mode=mode, with_offset=True,
                            min_capacity=int((n_more + 2 * int(np.load(brkpt)["parameters"][2])) / 0.5) + 1024)
    if p is None or p.n_rec == 0:
        return table
    hdr_off, n_rec = p.hdr_off, p.n_rec
    for r0, r, checkpoint, tail in plan_chunks(p.seq_lengths.astype(np.int64) * strands, chunk, Ns):
        if tail:
            # upstream re-parses from the last line: with a newline at or after it the whole file becomes a header
            # and an EMPTY record follows (one short-record sentinel hit per strand); without one nothing does
            ptr = _last_line_start(raw)
            if raw.find(b"\n", ptr) >= 0 and raw[:1] == b">":
                table.stats[_lib.PG_STAT_SHORT] += strands
            break
        if r > r0:
            table.insert(p, n_rec=r, rec_begin=r0)
            if table.overflowed():
                raise _lib.PgError("dBG table overflow in the chunked build")
        if not checkpoint:
            break
        ptr = int(hdr_off[r]) + shift if r < n_rec else _last_line_start(raw)
        npz.dump(table, qry + "_db_brkpt", offset=ptr)
    return table


def dump(kmer_dict, fn):
    """kmer_numba.py dump (:243-261): ``<fn>.npz`` in the reference's oakht layout.  A hash-partitioned table is merged on
    rank 0 first (every key lives on exactly one rank)."""
    from . import npz
    if kmer_dict.world > 1:
        from . import multigpu
        merged = multigpu.gather_export(kmer_dict.table, kmer_dict.world, kmer_dict.rank)
        if kmer_dict.rank != 0:
            return None
        return npz.dump_entries(*merged, fn)
    return npz.dump(kmer_dict.table, fn)


def load_dbg(qry, fn, kmer):
    """``-d`` / ``-D``: a table saved by the reference (or by ``dump``) + the packed input."""
    from . import npz
    kmer = min(max(1, int(kmer)), 27)
    fmt = seq_chk(qry)
    data, d_bytes = _read(qry)
    packed = _pack(qry, d_bytes, "fastq" if fmt == "fastq" else "fasta")
    table = npz.load(fn, kmer, device=packed.pk2.device)
    return DbgHandle(table, packed, data, packed.n_rec)


def dbg2rdbg(kmer_dict):
    """Stage 2: keep nodes with indegree != 1 or outdegree != 1.  On a hash-partitioned table (multi-GPU) the selection
    is part of seq2graph (every rank selects among its keys, the small rdBG tables are all-gathered there)."""
    if kmer_dict.world > 1:
        return kmer_dict
    rd = kmer_dict.table.select_rdbg()
    return DbgHandle(rd, kmer_dict.packed, kmer_dict.data, kmer_dict.n_rec)


def seq2graph(qry, kmer=13, bits=5, Ns=1e6, brkpt="./breakpoint_rdbg.npz", rdbg_dict=None, saved=None, hashfunc=None,
              jit=True, chunk=2 ** 33, rc=False, cluster=True, min_weight=1, out=None, write_mcl=True,
              cluster_method="components", inflation=1.5):
    """Stages 3-5: edge weights -> ``<qry>_rdbg_weight.xyz``; clusters (connected components, or Markov clustering
    with ``cluster_method="mcl"`` and ``inflation``; an existing ``.xyz.mcl`` cluster file wins) -> labels; region
    table on ``out`` (stdout)."""
    out = out or sys.stdout
    kmer = min(max(1, int(kmer)), 27)
    packed, data = rdbg_dict.packed, rdbg_dict.data
    world, rank = rdbg_dict.world, rdbg_dict.rank
    oname = qry + "_rdbg_weight.xyz"
    mcl_lines = None
    if cluster and os.path.isfile(oname + ".mcl"):
        if rank == 0:
            print("# the mcl has been ran", file=out)
        with open(oname + ".mcl") as f:
            mcl_lines = f.read().split("\n")
            if mcl_lines and mcl_lines[-1] == "":
                mcl_lines.pop()
    if world > 1:
        from . import builder, multigpu
        import torch.distributed as dist
        n_rec = builder.global_record_prefix(packed, Ns, 1, world)
        res, rows = multigpu.seq2graph_distributed(packed, rdbg_dict.table, kmer, world, rank, data, rc=bool(rc), min_weight=min_weight,
                                                   n_rec=n_rec, mcl_lines=mcl_lines, cluster=cluster_method, inflation=inflation)
        if rank == 0:
            res.write_xyz(oname)
            if mcl_lines is None and write_mcl:
                res.write_mcl(oname + ".mcl")
            out.write("".join("%s\t%d\t%d\t%s\t%d\n" % r for r in rows))
        dist.barrier()
        return LabelDict(res.nodes[1], res.nodes[2], res.nodes[3]) if rank == 0 else None
    res = graph.seq2graph_device(packed, rdbg_dict.table, kmer, Ns=Ns, rc=bool(rc), min_weight=min_weight, mcl_lines=mcl_lines,
                                 cluster=cluster_method, inflation=inflation)
    res.write_xyz(oname)
    if mcl_lines is None and write_mcl:
        res.write_mcl(oname + ".mcl")
    out.write("".join("%s\t%d\t%d\t%s\t%d\n" % r for r in res.rows(packed, data)))
    return LabelDict(res.nodes[1], res.nodes[2], res.nodes[3])


class LabelDict(dict):
    """The reference returns label_dct {(code, v5): label}; building millions of Python tuples is the
    slowest thing left in the CLI, so the dict is only materialised when somebody looks at it."""

    def __init__(self, code, v5, label):
        super().__init__()
        self._arrays, self._built = (code, v5, label), False

    def _build(self):
        if not self._built:
            self._built = True
            code, v5, label = self._arrays
            super().update({(int(c), int(v)): int(l) for c, v, l in zip(code.tolist(), v5.tolist(), label.tolist())})

    def __getitem__(self, k):
        self._build()
        return super().__getitem__(k)

    def __contains__(self, k):
        self._build()
        return super().__contains__(k)

    def __len__(self):
        return int(self._arrays[0].size)

    def __iter__(self):
        self._build()
        return super().__iter__()

    def items(self):
        self._build()
        return super().items()
