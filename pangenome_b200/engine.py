"""Host side of the B200 dBG path: device buffers (torch), launches through the
C-ABI (ctypes), and the small amount of host logic the reference keeps in its
un-jitted stage functions (record prefix for ``-n``, table sizing).

torch is plumbing only (allocation, streams, H2D/D2H); every computation on the
sequence data is a kernel of libpgdbg.so.  No CPU fallback: constructing any of
these objects without CUDA raises.
"""
import ctypes
import os

import numpy as np
import torch

from . import _lib
from ._lib import PgError, PgTable, check

_DEFAULT_LOAD = float(os.environ.get("PG_TABLE_LOAD", "0.5"))     # positions (upper bound of keys) per slot when sizing a table


def _require_cuda():
    if not torch.cuda.is_available():
        raise PgError("pangenome_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def next_pow2(n):
    n = max(2, int(n))
    return 1 << (n - 1).bit_length()


def to_device_bytes(data, device="cuda"):
    """bytes / bytearray / numpy uint8 / torch uint8 -> 16-byte aligned uint8 CUDA tensor."""
    _require_cuda()
    if isinstance(data, torch.Tensor):
        t = data if data.is_cuda else data.to(device, non_blocking=True)
        return t.contiguous().view(torch.uint8)
    if isinstance(data, (bytes, bytearray, memoryview)):
        arr = np.frombuffer(data, dtype=np.uint8)
    else:
        arr = np.ascontiguousarray(data, dtype=np.uint8)
    if arr.size == 0:
        return torch.empty(0, dtype=torch.uint8, device=device)
    return torch.from_numpy(arr.copy() if not arr.flags.writeable else arr).to(device)


class PackedSeqs:
    """Result of K1 (pg_fasta_scan_pack): the 2-bit packed base stream plus the
    record index.  Replaces what seqio_jit_ (kmer_numba.py:135-168) yields.
    ``fmt="fastq"``: the same outputs from a FASTQ stream (pg_fastq_scan_pack), as the FASTA of its header and sequence
    lines would give them; a malformed file raises FastqError when the record index is read."""

    def __init__(self, d_fasta, cap_records=1 << 12, lazy=False, fmt="fasta"):
        """``lazy``: enqueue K1 and return without reading the record index back; ``n_rec``,
        ``seq_off`` ... are fetched (one D2H, synchronising) the first time the host asks for them.
        The device-argument kernels (pg_kmer_partition_dev, ...) never need them on the host."""
        _require_cuda()
        if fmt not in ("fasta", "fastq"):
            raise PgError("PackedSeqs: fmt must be 'fasta' or 'fastq', got %r" % (fmt,))
        self.L = L = _lib.load()
        self.fmt = fmt
        self.d_fasta = d_fasta
        nbytes = int(d_fasta.numel())
        dev = d_fasta.device
        self.nbytes = nbytes
        words = int(L.pg_pack_words(nbytes))
        self.pk2 = torch.empty(words, dtype=torch.int32, device=dev)
        self.amb = torch.empty(words, dtype=torch.int32, device=dev)
        if fmt == "fasta":
            self._ws_bytes = int(L.pg_fasta_workspace_bytes(nbytes))
            self._ws = torch.empty(self._ws_bytes, dtype=torch.uint8, device=dev)
        self.launches = 3 if fmt == "fasta" else 5
        self._host = None
        self._launch(cap_records)
        if not lazy:
            self._fetch()

    def _launch(self, cap_records):
        # counts, seq_off and hdr_off (and the FASTQ status) share ONE device buffer so the record index comes back in one D2H
        L, nbytes = self.L, self.nbytes
        self.cap_records = cap_records
        fq = self.fmt == "fastq"
        idx = torch.empty(4 + (cap_records + 2) + (cap_records + 1) + (2 if fq else 0), dtype=torch.int64, device=self.pk2.device)
        self._idx = idx
        self.d_counts = idx[:4]
        self.d_seq_off = idx[4:4 + cap_records + 2]
        self.d_hdr_off = idx[4 + cap_records + 2:4 + cap_records + 2 + cap_records + 1]
        src = _ptr(self.d_fasta) if nbytes else None
        if not fq:
            check(L.pg_fasta_scan_pack(src, nbytes, _ptr(self.pk2), _ptr(self.amb), nbytes, _ptr(self.d_hdr_off),
                                       _ptr(self.d_seq_off), cap_records, _ptr(self.d_counts), _ptr(self._ws), self._ws_bytes,
                                       _stream()), "pg_fasta_scan_pack")
            return
        self.d_status = idx[-2:]
        self._ws_bytes = int(L.pg_fastq_workspace_bytes(nbytes, cap_records))
        self._ws = torch.empty(self._ws_bytes, dtype=torch.uint8, device=self.pk2.device)
        check(L.pg_fastq_scan_pack(src, nbytes, _ptr(self.pk2), _ptr(self.amb), nbytes, _ptr(self.d_hdr_off),
                                   _ptr(self.d_seq_off), cap_records, _ptr(self.d_counts), _ptr(self.d_status), _ptr(self._ws),
                                   self._ws_bytes, _stream()), "pg_fastq_scan_pack")

    def _fetch(self):
        if self._host is not None:
            return self._host
        while True:
            cap = self.cap_records
            if cap <= 1 << 16:
                h = self._idx.cpu().numpy()              # synchronises: the host needs the record index
                counts = h[:4]
            else:
                h = None
                counts = self.d_counts.cpu().numpy()
            n_rec = int(counts[0])
            if n_rec <= cap:
                break
            self._launch(next_pow2(n_rec + 1))           # the index was truncated: pack again with room for it
        if self.fmt == "fastq":
            off, kind = (h[-2:] if h is not None else self.d_status.cpu().numpy()).tolist()
            if off >= 0:
                raise FastqError(off, kind)
        if h is not None:
            seq_off = h[4:4 + n_rec + 1].copy()
            hdr_off = h[4 + cap + 2:4 + cap + 2 + n_rec].copy()
        else:
            seq_off = self.d_seq_off[:n_rec + 1].cpu().numpy()
            hdr_off = self.d_hdr_off[:n_rec].cpu().numpy()
        self._host = dict(n_rec=n_rec, n_bases=int(counts[1]), n_newlines=int(counts[2]), seq_off=seq_off, hdr_off=hdr_off)
        return self._host

    n_rec = property(lambda self: self._fetch()["n_rec"])
    n_bases = property(lambda self: self._fetch()["n_bases"])
    n_newlines = property(lambda self: self._fetch()["n_newlines"])
    seq_off = property(lambda self: self._fetch()["seq_off"])
    hdr_off = property(lambda self: self._fetch()["hdr_off"])

    @property
    def seq_lengths(self):
        return np.diff(self.seq_off)

    def record_prefix(self, Ns, strands):
        """How many records a stage processes under ``-n``: records are consumed
        until the running base count exceeds Ns; the record that crosses is
        still processed (kmer_numba.py:1227, 1820, 1847)."""
        lens = self.seq_lengths.astype(np.int64) * strands
        if lens.size == 0:
            return 0
        cum = np.cumsum(lens)
        over = np.nonzero(cum > Ns)[0]
        return int(over[0]) + 1 if over.size else int(lens.size)

    def n_positions(self, k, n_rec=None):
        lens = self.seq_lengths[:n_rec]
        return int(np.maximum(lens - k + 1, 0).sum())

    def n_insertions(self, k, n_rec=None, rc=True):
        """The metric's unit: sum over record-strands of max(n-k+1, 1)."""
        lens = self.seq_lengths[:n_rec]
        return int(np.maximum(lens - k + 1, 1).sum()) * (2 if rc else 1)


class FastqError(PgError):
    """A malformed FASTQ stream: ``offset`` = byte offset (in the packed stream) of the first bad record's header line,
    ``kind`` = include/pgdbg.h PG_FQ_* code."""

    def __init__(self, offset, kind):
        self.offset, self.kind = int(offset), int(kind)
        super().__init__("malformed FASTQ: the record at byte %d: %s" % (self.offset, self.reason))

    @property
    def reason(self):
        return _lib.PG_FQ_ERRORS.get(self.kind, "error %d" % self.kind)


class _StatsFuture:
    def __init__(self, pinned, event):
        self.pinned, self.event = pinned, event

    def wait(self):
        self.event.synchronize()
        return self.pinned.numpy().copy()


class DbgTable:
    """Device hash table behind the C-ABI ``pg_table`` struct (replaces oakht,
    kmer_numba.py:340-679).  ``mode``: 0 literal one strand, 1 literal both
    strands, 2 canonical pairs."""

    def __init__(self, capacity, k, mode, device="cuda"):
        _require_cuda()
        self.L = _lib.load()
        self.capacity = next_pow2(capacity)
        self.k = int(min(max(1, k), 27))
        self.mode = int(mode)
        self.slots = torch.empty(2 * self.capacity, dtype=torch.int64, device=device)
        self.stats = torch.zeros(_lib.PG_STAT_WORDS, dtype=torch.int64, device=device)
        # alloc_capacity: what an epoch wrap must rewrite even while set_capacity() selects a prefix of the buffer
        self.c = PgTable(self.slots.data_ptr(), self.capacity, self.stats.data_ptr(), self.mode, self.k, 1, 0, self.capacity)
        # a fresh allocation holds arbitrary tags: write every slot once; from then on clear() is an epoch bump
        check(self.L.pg_table_clear(ctypes.byref(self.c), _stream()), "pg_table_clear")

    def clear(self):
        """Empty the table: the epoch advances and every slot written so far reads as free - no HBM traffic
        (pg_table_reset rewrites the slots only when the 10-bit generation tag wraps)."""
        check(self.L.pg_table_reset(ctypes.byref(self.c), _stream()), "pg_table_reset")

    def reallocate(self, capacity):
        """Replace the slot buffer by one of ``capacity`` slots IN PLACE (every holder of this object sees the new table;
        the old buffer is released before the new one is requested).  The contents are gone: epoch 1, all slots cleared."""
        dev = self.slots.device
        self.capacity = next_pow2(capacity)
        self.slots = None
        self.c.d_slots = None
        torch.cuda.empty_cache()          # hand the old segment back whole: a smaller table must not pin it by living inside it
        self.slots = torch.empty(2 * self.capacity, dtype=torch.int64, device=dev)
        self.c.d_slots, self.c.capacity, self.c.alloc_capacity, self.c.epoch = self.slots.data_ptr(), self.capacity, self.capacity, 1
        check(self.L.pg_table_clear(ctypes.byref(self.c), _stream()), "pg_table_clear")

    def set_capacity(self, capacity):
        """Use only the first ``capacity`` (power of two) slots of the allocated buffer."""
        capacity = next_pow2(capacity)
        if 2 * capacity > self.slots.numel():
            raise PgError("set_capacity(%d) exceeds the allocated %d slots" % (capacity, self.slots.numel() // 2))
        self.capacity = capacity
        self.c.capacity = capacity

    def insert(self, packed, n_rec=None, g_begin=None, g_end=None, rec_begin=0):
        """Insert records [rec_begin, n_rec) (fused K2+K3).  With ``rec_begin`` the kernel is handed the record
        index from that record on, so zero-length records at the boundary belong to exactly one call."""
        n_rec = packed.n_rec if n_rec is None else n_rec
        if n_rec - rec_begin <= 0:
            return
        g_begin = int(packed.seq_off[rec_begin]) if g_begin is None else g_begin
        g_end = int(packed.seq_off[n_rec]) if g_end is None else g_end
        check(self.L.pg_kmer_insert(ctypes.byref(self.c), _ptr(packed.pk2), _ptr(packed.amb), ctypes.c_void_p(packed.d_seq_off.data_ptr() + 8 * rec_begin),
                                    n_rec - rec_begin, g_begin, g_end, _stream()), "pg_kmer_insert")

    def stats_host(self):
        return self.stats.cpu().numpy()

    def stats_async(self, slot=0):
        """Enqueue the D2H copy of the statistics words into pinned host memory (two slots, so a loop can
        read step i-1's result while step i runs) and return a handle whose ``wait()`` yields them."""
        if getattr(self, "_pinned", None) is None:
            self._pinned = torch.empty((2, _lib.PG_STAT_WORDS), dtype=torch.int64).pin_memory()
        dst = self._pinned[slot & 1]
        dst.copy_(self.stats, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        return _StatsFuture(dst, ev)

    def n_keys(self):
        """Occupied slots as counted by the inserts themselves (one atomicAdd per warp on claim):
        distinct canonical pairs in PG_MODE_CANONICAL, distinct literal keys otherwise."""
        return int(self.stats_host()[_lib.PG_STAT_USED])

    def count(self):
        check(self.L.pg_table_count(ctypes.byref(self.c), _stream()), "pg_table_count")
        s = self.stats_host()
        return int(s[_lib.PG_STAT_USED]), int(s[_lib.PG_STAT_ENTRIES])

    def overflowed(self):
        return bool(self.stats_host()[_lib.PG_STAT_OVERFLOW])

    def checksum(self):
        out = torch.zeros(3, dtype=torch.int64, device=self.slots.device)
        check(self.L.pg_table_checksum(ctypes.byref(self.c), _ptr(out), _stream()), "pg_table_checksum")
        v = out.cpu().numpy().view(np.uint64)
        return int(v[0]), int(v[1]), int(v[2])

    def export(self, sort=True):
        """(keys u64, vals u16, cnts u8) in the reference's convention."""
        _, n = self.count()
        dev = self.slots.device
        keys = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
        vals = torch.empty(max(n, 1), dtype=torch.int16, device=dev)
        cnts = torch.empty(max(n, 1), dtype=torch.uint8, device=dev)
        d_n = torch.zeros(1, dtype=torch.int64, device=dev)
        check(self.L.pg_table_export(ctypes.byref(self.c), _ptr(keys), _ptr(vals), _ptr(cnts), n, _ptr(d_n), _stream()),
              "pg_table_export")
        got = int(d_n.item())
        if got != n:
            raise PgError("pg_table_export produced %d entries, pg_table_count said %d" % (got, n))
        k = keys[:n].cpu().numpy().view(np.uint64)
        v = vals[:n].cpu().numpy().view(np.uint16)
        c = cnts[:n].cpu().numpy()
        if sort:
            o = np.argsort(k, kind="stable")
            k, v, c = k[o], v[o], c[o]
        return k, v, c

    # ---- K4 ----
    def rdbg_count(self):
        out = torch.zeros(2, dtype=torch.int64, device=self.slots.device)
        check(self.L.pg_rdbg_count(ctypes.byref(self.c), _ptr(out), _stream()), "pg_rdbg_count")
        o = out.cpu().numpy()
        return int(o[0]), int(o[1])

    def select_rdbg(self):
        n_slots, n_members = self.rdbg_count()
        rd = DbgTable(max(1024, int(n_slots / _DEFAULT_LOAD) + 1), self.k, self.mode, device=self.slots.device)
        check(self.L.pg_rdbg_select(ctypes.byref(self.c), ctypes.byref(rd.c), _stream()), "pg_rdbg_select")
        rd.n_members = n_members
        rd.n_slots_used = n_slots
        if rd.overflowed():
            raise PgError("rdBG table overflow")
        return rd

    def rdbg_export(self, n_members=None, sort=True):
        """Members (keys u64, vals u16) of an rdBG table, reference convention."""
        n = self.n_members if n_members is None else n_members
        dev = self.slots.device
        keys = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
        vals = torch.empty(max(n, 1), dtype=torch.int16, device=dev)
        d_n = torch.zeros(1, dtype=torch.int64, device=dev)
        check(self.L.pg_rdbg_export(ctypes.byref(self.c), _ptr(keys), _ptr(vals), n, _ptr(d_n), _stream()), "pg_rdbg_export")
        got = int(d_n.item())
        if got != n:
            raise PgError("pg_rdbg_export produced %d members, expected %d" % (got, n))
        k = keys[:n].cpu().numpy().view(np.uint64)
        v = vals[:n].cpu().numpy().view(np.uint16)
        if sort:
            o = np.argsort(k, kind="stable")
            k, v = k[o], v[o]
        return k, v


def build_dbg(packed, k, rc=True, Ns=2 ** 63, mode=None, capacity=None, max_grow=6):
    """K2+K3 over a PackedSeqs: returns (DbgTable, n_rec_used).  Table capacity
    defaults to next_pow2(positions / 0.5); on overflow it is doubled and the
    build repeated (the GPU table never rehashes in place)."""
    k = int(min(max(1, k), 27))
    if mode is None:
        mode = _lib.PG_MODE_CANONICAL if rc else _lib.PG_MODE_LITERAL
    if (mode == _lib.PG_MODE_LITERAL) == bool(rc):
        raise PgError("mode %d does not match rc=%s" % (mode, rc))
    n_rec = packed.record_prefix(Ns, 2 if rc else 1)
    npos = packed.n_positions(k, n_rec)
    keys_per_pos = 2 if mode == _lib.PG_MODE_LITERAL_RC else 1
    cap = next_pow2(max(1024, capacity or int(npos * keys_per_pos / _DEFAULT_LOAD) + 1))
    for _ in range(max_grow):
        t = DbgTable(cap, k, mode, device=packed.pk2.device)
        t.insert(packed, n_rec)
        if not t.overflowed():
            return t, n_rec
        cap *= 2
    raise PgError("dBG table kept overflowing up to capacity %d" % cap)


class RecordBuckets:
    """Output of K2a (pg_kmer_partition): 2^(owner_bits+sub_bits) buckets of 16-byte update
    records, ``part_cap`` records apart, with the per-bucket counts on the device."""

    def __init__(self, n_parts, part_cap, device):
        self.n_parts, self.part_cap = n_parts, part_cap
        self.records = torch.empty(2 * n_parts * part_cap, dtype=torch.int64, device=device)
        self.counts = torch.zeros(n_parts, dtype=torch.int64, device=device)
        self.seg_off = torch.arange(n_parts, dtype=torch.int64, device=device) * part_cap


class KeySampler:
    """The 1/256 key-space sample K2a can collect to estimate the number of distinct keys, i.e. how
    big the table has to be, before the table is cleared and filled (pg_kmer_partition)."""
    RATE = 256

    def __init__(self, n_positions, device):
        self.cap = next_pow2(max(1024, n_positions // self.RATE * 2 + 1024))
        self.keys = torch.empty(self.cap, dtype=torch.int64, device=device)
        self.count = torch.zeros(1, dtype=torch.int64, device=device)

    def reset(self):
        self.keys.fill_(-1)
        self.count.zero_()

    def estimate(self):
        """Estimated distinct keys, or None if the sample set overflowed (synchronises)."""
        c = int(self.count.item())
        return None if c >= (1 << 40) else c * self.RATE


def capacity_for(est_keys, upper, load=0.35, margin=1.05):
    """Power-of-two capacity for an estimated number of keys (load ends up in (load/2, load])."""
    if est_keys is None:
        return upper
    return min(upper, next_pow2(max(1024, int(est_keys * margin / load) + 1)))


def partition_kmers(packed, k, mode, n_rec, owner_bits, sub_bits, g_begin=None, g_end=None, slack=1.25, buckets=None,
                    sampler=None):
    """K2a over records [0, n_rec): returns RecordBuckets (no synchronisation)."""
    L = _lib.load()
    n_parts = 1 << (owner_bits + sub_bits)
    g_begin = int(packed.seq_off[0]) if g_begin is None else g_begin
    g_end = int(packed.seq_off[n_rec]) if g_end is None else g_end
    per_pos = 2 if mode == _lib.PG_MODE_LITERAL_RC else 1
    part_cap = int((g_end - g_begin) * per_pos / n_parts * slack) + 4096
    if buckets is None or buckets.n_parts != n_parts or buckets.part_cap < part_cap:
        buckets = RecordBuckets(n_parts, part_cap, packed.pk2.device)
    desc = PgTable(None, 2, None, mode, k, 1, 0)    # only mode and k are read by K2a
    if sampler is not None:
        sampler.reset()
    check(L.pg_kmer_partition(ctypes.byref(desc), _ptr(packed.pk2), _ptr(packed.amb), _ptr(packed.d_seq_off), n_rec,
                              g_begin, g_end, owner_bits, sub_bits, _ptr(buckets.records), buckets.part_cap,
                              _ptr(buckets.counts), _ptr(sampler.keys) if sampler else None, sampler.cap if sampler else 0,
                              _ptr(sampler.count) if sampler else None, _stream()), "pg_kmer_partition")
    return buckets


def sub_bits_for(capacity, sub_bytes=32 << 20):
    """Enough hash-prefix buckets that one bucket's table region (capacity*16/2^bits bytes) fits L2."""
    bits = 0
    while (capacity * 16) >> bits > sub_bytes and bits < 10:
        bits += 1
    return bits


def build_dbg_partitioned(packed, k, rc=True, Ns=2 ** 63, mode=None, capacity=None, sub_bytes=8 << 20, buckets=None,
                          table=None):
    """Two-phase build (K2a + K3).  K2a runs first and samples the key space, so the table is sized
    from an estimate of the distinct keys (load 0.18-0.35) instead of the positions upper bound.
    Falls back to the fused kernel when a bucket overflows (pathological hash skew, e.g. one k-mer
    making up most of the input)."""
    k = int(min(max(1, k), 27))
    if mode is None:
        mode = _lib.PG_MODE_CANONICAL if rc else _lib.PG_MODE_LITERAL
    n_rec = packed.record_prefix(Ns, 2 if rc else 1)
    npos = packed.n_positions(k, n_rec)
    per_pos = 2 if mode == _lib.PG_MODE_LITERAL_RC else 1
    upper = next_pow2(max(1024, int(npos * per_pos / _DEFAULT_LOAD) + 1))
    L = _lib.load()
    dev = packed.pk2.device
    if n_rec == 0:
        return DbgTable(capacity or 1024, k, mode, device=dev), n_rec, buckets
    sub_bits = sub_bits_for(capacity or upper, sub_bytes)
    # sparse tables are faster for K3 (see TwoPhaseBuilder); estimate only when the upper bound is expensive
    want_estimate = capacity is None and upper * 16 > 0.35 * torch.cuda.mem_get_info(dev)[0]
    sampler = KeySampler(npos * per_pos, dev) if want_estimate else None
    buckets = partition_kmers(packed, k, mode, n_rec, 0, sub_bits, buckets=buckets, sampler=sampler)
    cap = next_pow2(capacity) if capacity else (capacity_for(sampler.estimate(), upper) if sampler else upper)
    g_begin, g_end = int(packed.seq_off[0]), int(packed.seq_off[n_rec])
    for _ in range(6):
        t = DbgTable(cap, k, mode, device=dev)
        check(L.pg_count_short(ctypes.byref(t.c), _ptr(packed.d_seq_off), n_rec, g_begin, g_end, _stream()), "pg_count_short")
        check(L.pg_insert_records(ctypes.byref(t.c), _ptr(buckets.records), _ptr(buckets.seg_off), _ptr(buckets.counts),
                                  buckets.n_parts, 1, buckets.part_cap, _stream()), "pg_insert_records")
        worst = int(buckets.counts.max().item())           # synchronises
        if worst > buckets.part_cap:
            t2, n_rec = build_dbg(packed, k, rc=rc, Ns=Ns, mode=mode, capacity=cap)
            return t2, n_rec, buckets
        if not t.overflowed():
            return t, n_rec, buckets
        cap *= 2
    raise PgError("dBG table kept overflowing up to capacity %d" % cap)


class TwoPhaseBuilder:
    """Reusable buffers for repeated two-phase builds of same-sized inputs (bench / serving loop):
    the table and the record buckets stay resident in HBM between calls and the table is emptied by an
    epoch bump.  By default the table is sized from the positions upper bound, which allows the fully
    asynchronous build_async(); with ``estimate=True`` (or when that table would take a large part of the
    free HBM) K2a also samples the key space and build() sizes the table from the estimate - a small D2H."""

    def __init__(self, k, mode, n_positions, device="cuda", capacity=None, sub_bytes=8 << 20, owner_bits=0, estimate=None):
        self.L = _lib.load()
        self.k, self.mode = int(min(max(1, k), 27)), int(mode)
        per_pos = 2 if mode == _lib.PG_MODE_LITERAL_RC else 1
        cap = next_pow2(max(1024, capacity or int(n_positions * per_pos / _DEFAULT_LOAD) + 1))
        self.cap_max = cap
        self.table = DbgTable(cap, self.k, self.mode, device=device)
        self.sub_bits = sub_bits_for(cap, sub_bytes)
        self.owner_bits = owner_bits
        n_parts = 1 << (self.sub_bits + owner_bits)
        part_cap = int(n_positions * per_pos / n_parts * 1.25) + 4096
        self.buckets = RecordBuckets(n_parts, part_cap, device)
        # K3 is fastest on a sparse table (measured on config 2: load 0.125 -> 1.02 ms, 0.25 -> 1.10 ms, 0.5 -> 1.33 ms)
        # and emptying a table costs nothing (epoch bump), so the positions upper bound is used while it is affordable; the
        # estimator takes over when that table would eat a large part of the free HBM (config-5 scale)
        if estimate is None:
            free = torch.cuda.mem_get_info(device)[0] if torch.cuda.is_available() else 0
            estimate = cap * 16 > 0.35 * free
        self.sampler = KeySampler(n_positions * per_pos, device) if (estimate and not capacity) else None
        self.launches_per_build = 3          # k2a_partition, count_short, k3_insert_records (the reset is a 64-byte memset)
        self.last_estimate = None

    def begin(self):
        """Empty the table for the next build (an epoch bump, DbgTable.clear).  With the estimator the
        capacity is only known after K2a, so build() resets there instead."""
        if self.sampler is not None:
            return
        self.table.clear()
        self._begun = True

    def build(self, packed, n_rec, ev=None):
        """K2a, (estimate -> capacity), clear, K3.  ``ev`` = optional dict receiving CUDA event pairs
        around the kernels."""
        t, b, L = self.table, self.buckets, self.L
        st = torch.cuda.current_stream()
        if self.sampler is None and not getattr(self, "_begun", False):
            self.begin()
        self._begun = False
        if n_rec == 0:
            if self.sampler is not None:
                t.clear()
            return t
        g_begin, g_end = int(packed.seq_off[0]), int(packed.seq_off[n_rec])
        if ev is not None:
            e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            e[0].record(st)
        self.buckets = b = partition_kmers(packed, self.k, self.mode, n_rec, self.owner_bits, self.sub_bits, buckets=b,
                                           sampler=self.sampler)
        if ev is not None:
            e[1].record(st)
        if self.sampler is not None:
            self.last_estimate = self.sampler.estimate()            # 8-byte D2H, synchronises
            t.set_capacity(capacity_for(self.last_estimate, self.cap_max))
            t.clear()
        check(L.pg_count_short(ctypes.byref(t.c), _ptr(packed.d_seq_off), n_rec, g_begin, g_end, _stream()), "pg_count_short")
        if ev is not None:
            e[2].record(st)
        check(L.pg_insert_records(ctypes.byref(t.c), _ptr(b.records), _ptr(b.seg_off), _ptr(b.counts), b.n_parts, 1, b.part_cap, _stream()),
              "pg_insert_records")
        if ev is not None:
            e[3].record(st)
            ev.setdefault("partition", []).append((e[0], e[1]))
            ev.setdefault("size+clear", []).append((e[1], e[2]))
            ev.setdefault("insert", []).append((e[2], e[3]))
        return t

    def build_async(self, packed, ev=None):
        """K2a + K3 over ALL records of ``packed`` with device-side arguments: nothing is read back
        from K1, so pack -> partition -> insert is enqueued back to back (PackedSeqs(lazy=True)).
        Needs the upper-bound table (no estimator) and a record index that fits ``cap_records``
        (otherwise verify() raises and the caller uses build())."""
        if self.sampler is not None:
            raise PgError("build_async sizes the table before K2a: construct the builder with estimate=False")
        t, b, L = self.table, self.buckets, self.L
        st = torch.cuda.current_stream()
        if not getattr(self, "_begun", False):
            self.begin()
        self._begun = False
        if ev is not None:
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record(st)
        desc = PgTable(None, 2, None, self.mode, self.k, 1, 0)
        check(L.pg_kmer_partition_dev(ctypes.byref(desc), _ptr(packed.pk2), _ptr(packed.amb), _ptr(packed.d_seq_off),
                                      _ptr(packed.d_counts), packed.cap_records, packed.nbytes, self.owner_bits, self.sub_bits,
                                      _ptr(b.records), b.part_cap, _ptr(b.counts), _stream()), "pg_kmer_partition_dev")
        check(L.pg_count_short_dev(ctypes.byref(t.c), _ptr(packed.d_seq_off), _ptr(packed.d_counts), packed.cap_records, _stream()),
              "pg_count_short_dev")
        if ev is not None:
            e[1].record(st)
        check(L.pg_insert_records(ctypes.byref(t.c), _ptr(b.records), _ptr(b.seg_off), _ptr(b.counts), b.n_parts, 1, b.part_cap, _stream()),
              "pg_insert_records")
        if ev is not None:
            e[2].record(st)
            ev.setdefault("partition", []).append((e[0], e[1]))
            ev.setdefault("insert", []).append((e[1], e[2]))
        return t

    def verify(self):
        """After a synchronise: raise if a bucket or the table overflowed."""
        if int(self.buckets.counts.max().item()) > self.buckets.part_cap:
            raise PgError("record bucket overflow (hash skew) or truncated record index: use build_dbg()")
        if self.table.overflowed():
            raise PgError("dBG table overflow")
