"""The streaming dBG builder: one code path for a single GPU and for the hash-partitioned multi-GPU build
(replaces oakht + seq2dbg_jit_, kmer_numba.py:340-679, 1202-1230; the split is SURVEY.md 8e).

A build is cut into ROUNDS of stream positions.  Per round and rank (default: COMPACT 8-byte update records,
csrc/compact_build.cu - canonical mode, 4096-slot regions; the same pipeline runs on 16-byte records for the literal
modes, 256-slot regions and inputs whose wide spill overflows):

    stream A   K2a-c  k-mer extraction -> 8-byte records for interior positions, 16-byte wide records for the rest
                      world 1 : straight into the 2^sub_bits hash-prefix buckets of a local set (+ its wide spill)
                      world N : bucketed by OWNER only and stored into the owners' receive buffers over NVLink
                                (CUDA IPC peer memory) - 8192-position tiles give 8 KB runs per peer at 8 GPUs
    stream B   [N>1] all-to-all of the 2 W record counts (NCCL) - also the barrier that orders the peer stores
               [N>1] K2b-c  what arrived (one segment per source) -> hash-prefix buckets
                     K2c-c  every hash-prefix bucket -> one bucket per table region (one or two levels),
                     K3s-c  one CTA per region builds it in SHARED MEMORY from the 2-bit codes and writes it to HBM once
                            (base-5 keys in the last round), then the wide records are upserted with L2 atomics
               or, for tables beyond 2^18 regions: plan (clamped counts, PG_STAT_LOST), K3 region sweep with L2 atomics
               on 16-byte records

Two record buffers alternate, so K2a of round r+1 runs while K2b/K2c/K3s of round r drain the other buffer: the
extraction (and its NVLink write-out) overlaps the table build.
Nothing is read back inside a build; verify() looks at the table's statistics block afterwards (overflow /
lost-record flags) and the callers fall back to a safer configuration (16-byte records, more rounds, larger table)
when it trips.

Memory: a round holds round_len x 8 (or 16) B x slack per buffer, the table 16 B per slot; both are sized for the
HBM that is actually free (180 GB on a B200), so inputs far larger than one round stream through.
"""
import ctypes
import os

import torch
import torch.distributed as dist

from . import _lib, engine
from ._lib import PgBucketSet, PgCBuckets, PgError, check

_TILE = 8192


class LostRecords(PgError):
    """update records were dropped (bucket + spill overflow): rebuild with more rounds"""


class TableFull(PgError):
    """the hash table ran out of probe room: rebuild with a larger capacity"""


def log2_exact(n):
    b = n.bit_length() - 1
    if n < 1 or (1 << b) != n:
        raise ValueError("world size must be a power of two (1, 2, 4, 8), got %d" % n)
    return b


class LocalBuckets:
    """2^sub_bits buckets of ``part_cap`` update records + one spill bucket (include/pgdbg.h pg_bucket_set)."""

    def __init__(self, sub_bits, part_cap, spill_cap, device):
        self.sub_bits, self.n_parts, self.part_cap, self.spill_cap = sub_bits, 1 << sub_bits, int(part_cap), int(spill_cap)
        n = self.n_parts
        self.records = torch.empty(2 * (n * self.part_cap + self.spill_cap), dtype=torch.int64, device=device)
        self.counts = torch.zeros(n + 1, dtype=torch.int64, device=device)
        self.seg_off = torch.arange(n + 1, dtype=torch.int64, device=device) * self.part_cap      # the spill follows the last bucket
        self.seg_cnt = torch.zeros(n + 1, dtype=torch.int64, device=device)
        self.c = PgBucketSet(self.records.data_ptr(), None, self.counts.data_ptr(), self.part_cap, self.spill_cap, 0, sub_bits, 0, 0)

    def bytes(self):
        return self.records.numel() * 8


class CompactBuckets:
    """The buffers of a compact (8-byte record) build, include/pgdbg.h pg_cbuckets: the level-0 buckets K2a-c fills and the
    wide spill every level of the round shares (16-byte records the compact form cannot hold + bucket surplus)."""

    def __init__(self, bits, part_cap, wide_cap, device):
        self.bits, self.n_parts, self.part_cap, self.wide_cap = bits, 1 << bits, int(part_cap) + (int(part_cap) & 1), int(wide_cap)
        self.records = torch.empty(self.n_parts * self.part_cap, dtype=torch.int64, device=device)
        self.counts = torch.zeros(self.n_parts, dtype=torch.int64, device=device)
        self.wide = torch.empty(2 * self.wide_cap, dtype=torch.int64, device=device)
        self.wide_count = torch.zeros(1, dtype=torch.int64, device=device)
        self.c = self.view(self.records, self.counts, bits, self.part_cap)

    def view(self, records, counts, bits, part_cap):
        """A pg_cbuckets over ``records`` / ``counts`` (another partition level) sharing this set's wide spill."""
        return PgCBuckets(records.data_ptr(), counts.data_ptr(), int(part_cap), int(bits), 0, self.wide.data_ptr(), self.wide_count.data_ptr(),
                          self.wide_cap)

    def bytes(self):
        return self.records.numel() * 8 + self.wide.numel() * 8


def exchange_record_counts(send_counts, recv, world):
    """The one collective on the compact multi-GPU data path.  ``send_counts``: [compact count per owner rank | wide count
    per owner rank] as K2a-c left them (2 * world int64); ``recv``: a (world, 2) int64 buffer that ends up holding, per
    SOURCE rank, (compact records, wide records) that rank stored into this rank's receive buffers.  Also the barrier
    that orders the peer stores before they are read.  Returns (compact counts, wide counts), contiguous."""
    dist.all_to_all_single(recv, send_counts.view(2, world).t().contiguous())
    return recv[:, 0].contiguous(), recv[:, 1].contiguous()


def plan_rounds(n_bases_max, rounds=None, round_len=None, tile=_TILE):
    """(n_rounds, round_len): the stream [0, n_bases_max) in equal rounds, a whole number of K2a tiles each."""
    n_bases_max = max(1, int(n_bases_max))
    if round_len is None:
        rounds = max(1, int(rounds or 1))
        round_len = (n_bases_max + rounds - 1) // rounds
    round_len = max(tile, (int(round_len) + tile - 1) // tile * tile)
    return (n_bases_max + round_len - 1) // round_len, round_len


def plan_levels(region_log, world, max_bits=8):
    """Fan-out bits of the partition levels that take a record down to one bucket per table region (2^region_log of
    them).  Level 0 is K2a's (one GPU) or K2b's (what arrived over the wire) and goes through the bucket-set API (<= 2^10
    buckets); every further level is a sliced re-split (pg_records_resplit, <= 2^8 ways, input <= 2^13 buckets).  As few
    levels as the fan-out limits allow: on BASELINE config 4 at 2 GPUs (2^18 regions per rank) [10, 8], [5, 6, 7] and the
    older tile sort measured 104 / 107 / 101 ms per step - a pass costs its 32 B per record whatever its fan-out, so the
    third pass eats what the longer runs of the first two win."""
    env = os.environ.get("PG_LEVELS")
    if env:                                  # experiment switch: "6,6,6"
        try:
            lv = [int(x) for x in env.split(",")]
            if sum(lv) == region_log and all(1 <= x <= 10 for x in lv):
                return lv
        except ValueError:
            pass
    if region_log <= 8:
        return [region_log]
    first = 8 if world == 1 else min(10, max(6, region_log - 8))
    rest = region_log - first
    if rest <= max_bits:          # compact records take one 2^9-way pass (config 3: 11.7 ms against 13.3 ms for [4, 5])
        return [first, rest]
    a = rest // 2
    return [first, a, rest - a]


def table_capacity_for(n_keys_upper, free_bytes, load=0.5, max_fraction=0.55):
    """Power-of-two slot count for at most ``n_keys_upper`` keys, never more than ``max_fraction`` of the free HBM."""
    cap = engine.next_pow2(max(1024, int(n_keys_upper / load) + 1))
    while cap > 1024 and cap * 16 > max_fraction * free_bytes:
        cap //= 2
    return cap


class RoundBuilder:
    """See the module docstring.  ``n_bases_max``: upper bound of this rank's stream length per build (the file size
    will do).  ``rounds`` / ``round_len``: how the stream is cut.  Default: ONE round whenever its records fit
    (PG_ROUNDS overrides) in the free HBM next to the table: every K3 launch re-reads and writes back
    the table sectors of all the keys its round touches, and in a pangenome every round touches nearly all of them -
    measured on config 2, K3 takes 1.01 / 1.86 / 2.55 ms in 1 / 2 / 4 rounds (profiles/r2c_*), more than the overlap of
    K2a with K3 wins back.  Rounds are for inputs whose records do not fit, not for speed."""

    MAX_ROUND = 1 << 31          # K3 indexes the records of one region with 32 bits

    REGION_BITS = 12             # slots per shared-memory table region (64 KB); PG_REGION_BITS=0 selects the L2-atomic K3
    MAX_REGION_LOG = 18          # 2^10 coarse buckets (K2a) x 2^8 fine ones each (K2c)

    def __init__(self, k, mode, n_bases_max, world=1, rank=0, device="cuda", capacity=None, rounds=None, round_len=None,
                 sub_bytes=None, slack=1.25, spill_frac=1.0 / 16, region_bits=None, sample=False, compact=None):
        engine._require_cuda()
        self.L = _lib.load()
        self.k, self.mode = int(min(max(1, k), 27)), int(mode)
        self.world, self.rank, self.device = int(world), int(rank), torch.device(device)
        self.owner_bits = log2_exact(self.world)
        if self.world > 1 and self.mode == _lib.PG_MODE_LITERAL_RC:
            raise PgError("the multi-GPU build runs in PG_MODE_CANONICAL (both strands) or PG_MODE_LITERAL (one strand)")
        per_pos = 2 if self.mode == _lib.PG_MODE_LITERAL_RC else 1
        dev = self.device
        n_max, n_sum = int(n_bases_max), int(n_bases_max)
        if self.world > 1:
            t = torch.tensor([n_max, n_max], dtype=torch.int64, device=dev)
            tm = t.clone()
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            n_max, n_sum = int(tm[0].item()), int(t[1].item())
        self.n_bases_max = n_max
        # ---- the table: every key lives on exactly one rank; sized for the worst case (all positions distinct, evenly
        # spread) while that is affordable, else for what the free HBM allows (the overflow flag reports a table too small)
        free = torch.cuda.mem_get_info(dev)[0]
        W = self.world
        if W > 1:       # every rank must plan the same rounds: agree on the smallest free HBM
            f = torch.tensor([free], dtype=torch.int64, device=dev)
            dist.all_reduce(f, op=dist.ReduceOp.MIN)
            free = int(f.item())
        per_rank_keys = (n_sum * per_pos + W - 1) // W
        cap = engine.next_pow2(capacity) if capacity else table_capacity_for(per_rank_keys, free)
        # ---- rounds: as few as the free HBM allows (see the class docstring).  Bytes of record buffers per stream position:
        # one local set when a single round suffices, two alternating ones otherwise; across GPUs two receive buffers
        # (peer-written) plus the local set K2b fills
        spill = 1.0 + spill_frac
        # shared-memory region build: the table is a whole number of 2^region_bits-slot regions, K2a / K2b bucket by the top
        # ``sub_bits`` hash bits and K2c refines every bucket down to one per region (one more record buffer)
        if region_bits is None:
            region_bits = int(os.environ.get("PG_REGION_BITS", str(self.REGION_BITS)))
        self._region_pref = region_bits if region_bits in (8, 12) else 0
        # compact 8-byte update records (csrc/compact_build.cu): one GPU, canonical mode, 4096-slot regions; PG_COMPACT=0 keeps
        # the 16-byte records.  verify() switches it off for good when an input overflows the wide spill (many short records
        # or long ambiguity runs: positions the compact form cannot hold).
        if compact is None:
            compact = os.environ.get("PG_COMPACT", "1") != "0"
        self._compact_pref = bool(compact) and self.mode == _lib.PG_MODE_CANONICAL and self._region_pref == 12
        self.compact = False
        cap_log = cap.bit_length() - 1
        region_now = bool(self._region_pref) and 0 <= cap_log - self._region_pref <= self.MAX_REGION_LOG
        if W == 1:
            rec_b = 8.0 if (self._compact_pref and region_now) else 16.0
            fine = rec_b * per_pos * slack * spill if region_now else 0.0
            bpp1, bppn = rec_b * per_pos * slack * spill + fine, 2 * rec_b * per_pos * slack * spill + fine
        else:
            bpp1 = bppn = 16.0 * slack * (2 + slack * spill)
        if rounds is None and round_len is None:
            rounds = int(os.environ.get("PG_ROUNDS", "0"))
            if not rounds:
                room = max(0.85 * free - cap * 16, 0.05 * free)
                rounds = 1 if n_max * bpp1 <= room else max(2, int(-(-n_max * bppn // room)))
            rounds = max(rounds, (n_max + self.MAX_ROUND - 1) // self.MAX_ROUND)
        self.n_rounds, self.round_len = plan_rounds(n_max, rounds, round_len)
        R = self.round_len
        if sub_bytes is None:
            sub_bytes = int(os.environ.get("PG_SUB_MB", "8")) << 20
        self._sub_bytes, self._per_pos, self._slack, self._spill_frac = sub_bytes, per_pos, slack, spill_frac
        self.table, self.sets, self.sub_bits, self.region_bits = None, None, None, 0
        self.fine_records = self.fine_counts = None
        self.adaptive = bool(self._region_pref) and not capacity
        self.sampler = None
        # ---- record buffers
        if W == 1:
            self._arriving = R * per_pos
            self.wire = None
        else:
            self.cap_wire = cw = (int(R / W * slack) + 8192) & ~1
            self.wire_bytes = W * cw * 16
            self.own, self._opened, self.peer_tables, self.wire_sets = [], [], [], []
            for _ in range(2):
                ptr = ctypes.c_void_p()
                handle = ctypes.create_string_buffer(64)
                check(self.L.pg_peer_alloc(self.wire_bytes, ctypes.byref(ptr), handle), "pg_peer_alloc")
                handles = [None] * W
                dist.all_gather_object(handles, handle.raw)
                addrs = []
                for r in range(W):
                    if r == rank:
                        addrs.append(ptr.value)
                    else:
                        q = ctypes.c_void_p()
                        check(self.L.pg_peer_open(handles[r], ctypes.byref(q)), "pg_peer_open")
                        self._opened.append(q)
                        addrs.append(q.value)
                self.own.append(ptr)
                self.peer_tables.append(torch.tensor(addrs, dtype=torch.int64, device=dev))
            self.send_counts = [torch.zeros(W + 1, dtype=torch.int64, device=dev) for _ in range(2)]
            self.recv_counts = [torch.zeros(W, dtype=torch.int64, device=dev) for _ in range(2)]
            for i in range(2):      # bucket (owner) of source `rank` lands at [rank][cap_wire] of the owner's buffer
                self.wire_sets.append(PgBucketSet(None, self.peer_tables[i].data_ptr(), self.send_counts[i].data_ptr(), cw, 0,
                                                  self.owner_bits, 0, rank, 0))
            self.wire_seg_off = torch.arange(W, dtype=torch.int64, device=dev) * cw
            self.sent_total = torch.zeros(W, dtype=torch.int64, device=dev)
            # per source: the most records one round of this build sent to this rank, surplus over cap_wire included
            self.wire_peak = torch.zeros(W, dtype=torch.int64, device=dev)
            self._arriving = W * cw
            # the same receive buffers under compact records: W segments of cw 8-byte records, then W segments of cw / 2
            # wide (16-byte) records; counters [W compact | W wide]
            self.cap_wide_wire = cw // 2
            self.wide_peer_tables = [pt + W * cw * 8 for pt in self.peer_tables]
            self.csend_counts = [torch.zeros(2 * W, dtype=torch.int64, device=dev) for _ in range(2)]
            self.crecv = [torch.zeros((W, 2), dtype=torch.int64, device=dev) for _ in range(2)]
            self.cwire_sets = [PgCBuckets(None, self.csend_counts[i].data_ptr(), cw, self.owner_bits, 0, None,
                                          self.csend_counts[i].data_ptr() + 8 * W, self.cap_wide_wire, self.peer_tables[i].data_ptr(),
                                          self.wide_peer_tables[i].data_ptr(), rank, 0) for i in range(2)]
        self._configure(cap)
        if self.region_bits and W == 1 and sample and self.n_rounds == 1 and not capacity:
            self.sampler = engine.KeySampler(n_max * per_pos, dev)
        if W > 1:
            dist.barrier()
        self.sA, self.sB = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        self._round = 0                     # global round counter: buffer parity carries over from build to build
        self._ev_free = [None, None]        # world 1: K3 finished reading local set i
        self._ev_a2a = None                 # world N: the previous round's count exchange (= every peer drained buffer i)
        self._begun = False
        self._next_capacity = None
        self._reconfigure = False
        self.desc = _lib.PgTable(None, 2, None, self.mode, self.k, 1, 0, 0)      # K2a reads mode and k only

    @property
    def launches_per_round(self):
        """Kernels of this library per round: K2a, (K2b,) then plan + K3, or K2c + K3s + spill upserts."""
        n = 1 + (1 if self.world > 1 else 0)
        if self.compact and self.world > 1:
            n += self.world                      # one wide-record upsert per source rank
        return n + ((len(self.levels) - 1 + 2) if self.region_bits else 2)

    @property
    def launches_per_build(self):
        return 1 + self.n_rounds * self.launches_per_round       # + count_short

    def _configure(self, cap):
        """(Re)build everything that depends on the table capacity: the table itself (a table at least 4x larger than
        needed is released), whether it is built in shared-memory regions, how many hash-prefix buckets K2a / K2b
        produce, and the fine bucket set of K2c.  Called at construction and, between builds, by begin() after verify()
        retuned the capacity."""
        dev, rb = self.device, self._region_pref
        cap = engine.next_pow2(cap)
        cap_log = cap.bit_length() - 1
        region = bool(rb) and 0 <= cap_log - rb <= self.MAX_REGION_LOG
        self._level_bits = 9 if (region and self._compact_pref) else 8        # widest re-split level (K2c-c: 9, K2c: 8)
        if region:
            self.levels = plan_levels(cap_log - rb, self.world, self._level_bits)
            sub_bits = self.levels[0]
        else:
            self.levels = None
            sub_bits = engine.sub_bits_for(cap, self._sub_bytes)
        if self.table is None:
            self.table = engine.DbgTable(cap, self.k, self.mode, device=dev)
        else:
            have = self.table.slots.numel() // 2
            if have < cap or have >= 4 * cap:
                self.table.reallocate(cap)                       # in place: callers keep their reference to the table
            else:
                self.table.set_capacity(cap)
        self.region_bits = rb if region else 0
        self.table.c.region_bits = self.region_bits
        self.compact = bool(region and self._compact_pref)
        self.table.c.hash_kind = 1 if self.compact else 0
        n_sub = 1 << sub_bits
        part_cap = int(self._arriving / n_sub * self._slack) + 2048
        spill_cap = max(1 << 16, int(self._arriving * self._spill_frac))
        if self.compact:
            if self.sets is None or sub_bits != self.sub_bits or not isinstance(self.sets[0], CompactBuckets):
                n_sets = 2 if (self.world == 1 and self.n_rounds > 1) else 1
                self.sets = None
                self.sets = [CompactBuckets(sub_bits, part_cap, spill_cap, dev) for _ in range(n_sets)]
                self._ev_free = [None, None]
            self.sub_bits = sub_bits
            if len(self.levels) > 1:
                n_regions = cap >> rb
                need = int(self._arriving * self._slack) + n_regions * 256
                if self.fine_records is None or self.fine_records.numel() < need:
                    self.fine_records = None
                    torch.cuda.empty_cache()
                    self.fine_records = torch.empty(need, dtype=torch.int64, device=dev)
                if self.fine_counts is None or any(c.numel() < n_regions + 1 for c in self.fine_counts) or len(self.fine_counts) < len(self.levels) - 1:
                    self.fine_counts = [torch.zeros(n_regions + 1, dtype=torch.int64, device=dev) for _ in self.levels[1:]]
            self.min_capacity = 1 << (sub_bits + rb)
            return
        if self.sets is not None and isinstance(self.sets[0], CompactBuckets):
            self.sets, self.fine_records, self.fine_counts = None, None, None       # left the compact path: 16-byte buffers from scratch
        if self.sets is None or sub_bits != self.sub_bits:
            n_sets = 2 if (self.world == 1 and self.n_rounds > 1) else 1
            self.sets = None
            self.sets = [LocalBuckets(sub_bits, part_cap, spill_cap, dev) for _ in range(n_sets)]
            self._ev_free = [None, None]
        self.sub_bits = sub_bits
        if region and len(self.levels) > 1:
            # the re-split levels ping-pong between a second record buffer and the memory of the level-0 set; every level has
            # its own counters.  Buckets of a level share its buffer evenly (laid out per build for the capacity in use).
            n_regions = cap >> rb
            self.fine_spill_cap = spill_cap
            need = 2 * (int(self._arriving * self._slack) + n_regions * 256 + spill_cap)
            if self.fine_records is None or self.fine_records.numel() < need:
                self.fine_records = None
                torch.cuda.empty_cache()                         # what the old table held goes back to the driver first
                room = torch.cuda.mem_get_info(dev)[0] + torch.cuda.memory_reserved(dev) - torch.cuda.memory_allocated(dev)
                if need * 8 > 0.97 * room:
                    # no room for the second record buffer: keep the L2-atomic K3 for this builder
                    self._region_pref = 0
                    return self._configure(cap)
                self.fine_records = torch.empty(need, dtype=torch.int64, device=dev)
            n_max = n_regions
            if self.fine_counts is None or any(c.numel() < n_max + 1 for c in self.fine_counts) or len(self.fine_counts) < len(self.levels) - 1:
                self.fine_counts = [torch.zeros(n_max + 1, dtype=torch.int64, device=dev) for _ in self.levels[1:]]
        # a sampled build fills K2a's buckets before the capacity is known: it must keep at least one region per bucket
        self.min_capacity = (1 << (sub_bits + rb)) if region else 1024

    # ------------------------------------------------------------------------------------------------
    def begin(self):
        """Empty the table for the next build: an epoch bump (DbgTable.clear), no HBM traffic."""
        if (self._next_capacity and self._next_capacity != self.table.capacity) or self._reconfigure:
            torch.cuda.synchronize(self.device)          # buffers may be replaced: nothing of the last build may be in flight
            self._configure(self._next_capacity or self.table.capacity)
        self._next_capacity, self._reconfigure = None, False
        self.table.clear()
        if self.world > 1:
            self.wire_peak.zero_()
        self._begun = True

    def build_async(self, packed, n_rec=None, ev=None):
        """Enqueue one build of records [0, n_rec) of ``packed`` (``None``: ALL records, bounds read on the device -
        nothing K1 produced has to reach the host, PackedSeqs(lazy=True)).  Returns the table; verify() checks it.
        ``ev``: dict receiving (start, end) CUDA event pairs per stage."""
        L, t, W = self.L, self.table, self.world
        P, byref = engine._ptr, ctypes.byref
        cur = torch.cuda.current_stream()
        if not self._begun:
            self.begin()
        self._begun = False
        A, B = self.sA, self.sB
        A.wait_stream(cur)
        B.wait_stream(cur)
        dev_mode = n_rec is None
        if dev_mode:
            d_counts, cap_records, max_bases, g0, g1 = P(packed.d_counts), packed.cap_records, packed.nbytes, 0, None
            n_rec_arg = 1
        else:
            d_counts, cap_records, max_bases = None, 0, 0
            g0 = int(packed.seq_off[0]) if n_rec > 0 else 0
            g1 = int(packed.seq_off[n_rec]) if n_rec > 0 else 0
            n_rec_arg = n_rec
        def stamp(stream):
            if ev is None:
                return None
            e = torch.cuda.Event(enable_timing=True)
            e.record(stream)
            return e

        with torch.cuda.stream(B):
            if dev_mode:
                check(L.pg_count_short_dev(byref(t.c), P(packed.d_seq_off), d_counts, cap_records, engine._stream()), "pg_count_short_dev")
            elif n_rec > 0:
                check(L.pg_count_short(byref(t.c), P(packed.d_seq_off), n_rec, g0, g1, engine._stream()), "pg_count_short")
        for r in range(self.n_rounds):
            lo, hi = r * self.round_len, (r + 1) * self.round_len
            if not dev_mode:
                lo, hi = min(g0 + lo, g1), min(g0 + hi, g1)
            i = self._round & 1
            self._round += 1
            # ---- stream A: extraction (+ NVLink write-out) into buffer i
            with torch.cuda.stream(A):
                if W == 1:
                    si = i % len(self.sets)
                    bs = self.sets[si]
                    if self._ev_free[si] is not None:
                        A.wait_event(self._ev_free[si])           # K3 of the round that last used this set has drained it
                    out = bs.c
                else:
                    if self._ev_a2a is not None:
                        A.wait_event(self._ev_a2a)          # every peer has drained buffer i (its K2b of two rounds ago)
                    out = self.cwire_sets[i] if self.compact else self.wire_sets[i]
                e0 = stamp(A)
                smp = self.sampler if (self.sampler is not None and r == 0) else None
                if smp is not None:
                    smp.reset()
                part = L.pg_kmer_partition_c if self.compact else L.pg_kmer_partition_to
                check(part(byref(self.desc), P(packed.pk2), P(packed.amb), P(packed.d_seq_off), n_rec_arg, lo, hi,
                           d_counts, cap_records, max_bases, byref(out), P(smp.keys) if smp else None, smp.cap if smp else 0,
                           P(smp.count) if smp else None, engine._stream()),
                      "pg_kmer_partition_c" if self.compact else "pg_kmer_partition_to")
                e1 = stamp(A)
                if smp is not None:
                    # size the table from K2a's 1/256 key-space sample before anything is inserted: one 8-byte read-back
                    self.last_estimate = smp.estimate()
                    want = engine.capacity_for(self.last_estimate, t.slots.numel() // 2, load=0.5, margin=1.02)
                    t.set_capacity(max(self.min_capacity, want))
                if ev is not None and W > 1:     # measurement only: records really sent to every owner
                    self.sent_total += self.csend_counts[i][:W] if self.compact else self.send_counts[i][:W]
                done = torch.cuda.Event()
                done.record(A)
            # ---- stream B: (exchange barrier, split,) plan, table sweep
            with torch.cuda.stream(B):
                B.wait_event(done)
                if W > 1 and self.compact:
                    bs = self.sets[0]
                    x0 = stamp(B)
                    # one all-to-all for both counters: [owner][compact, wide] -> [source][compact, wide]
                    recv_c, recv_w = exchange_record_counts(self.csend_counts[i], self.crecv[i], W)
                    torch.maximum(self.wire_peak, recv_c, out=self.wire_peak)
                    self._ev_a2a = torch.cuda.Event()
                    self._ev_a2a.record(B)
                    x1 = stamp(B)
                    own = self.own[i].value
                    arrived = PgCBuckets(own, recv_c.data_ptr(), self.cap_wire, self.owner_bits, 0, bs.wide.data_ptr(), bs.wide_count.data_ptr(),
                                         bs.wide_cap, None, None, 0, 0)
                    bs.wide_count.zero_()               # K2b-c / K2c-c bucket surplus of this round
                    check(L.pg_records_split_c(byref(arrived), byref(bs.c), self.k, P(t.stats), engine._stream()), "pg_records_split_c")
                    self._wide_segments = (own + W * self.cap_wire * 8, recv_w)
                    x2 = stamp(B)
                elif W > 1:
                    bs = self.sets[0]
                    x0 = stamp(B)
                    dist.all_to_all_single(self.recv_counts[i], self.send_counts[i][:W])
                    torch.maximum(self.wire_peak, self.recv_counts[i], out=self.wire_peak)
                    self._ev_a2a = torch.cuda.Event()
                    self._ev_a2a.record(B)
                    x1 = stamp(B)
                    check(L.pg_records_split(self.own[i], P(self.wire_seg_off), P(self.recv_counts[i]), W, self.cap_wire, byref(bs.c),
                                             P(t.stats), engine._stream()), "pg_records_split")
                    x2 = stamp(B)
                else:
                    x2 = stamp(B)
                if self.compact:
                    # K2c-c: 8-byte records level by level down to one bucket per region, then K3s-c (+ the wide spill)
                    region_log = (t.capacity >> self.region_bits).bit_length() - 1
                    levels = [self.sub_bits] + plan_levels(region_log, W, self._level_bits)[1:] if region_log > self.sub_bits else [self.sub_bits]
                    if sum(levels) != region_log:              # sampled capacity: one or two even levels below K2a's buckets
                        rest = region_log - self.sub_bits
                        levels = [self.sub_bits] + ([rest] if rest <= self._level_bits else [rest // 2, rest - rest // 2])
                    cur_c, bits = bs.c, self.sub_bits
                    bufs = [self.fine_records, bs.records]
                    for li, lb in enumerate(levels[1:]):
                        out_rec, ocnt = bufs[li % 2], self.fine_counts[li]
                        n_out = 1 << (bits + lb)
                        ocap = (out_rec.numel() // n_out) & ~1
                        nxt_c = bs.view(out_rec, ocnt, bits + lb, ocap)
                        check(L.pg_records_resplit_c(byref(cur_c), lb, byref(nxt_c), self.k, P(t.stats), engine._stream()), "pg_records_resplit_c")
                        cur_c, bits = nxt_c, bits + lb
                    x2c = stamp(B)
                    last = 1 if r == self.n_rounds - 1 else 0
                    check(L.pg_region_build_c(byref(t.c), byref(cur_c), 1 if r == 0 else 0, last, engine._stream()), "pg_region_build_c")
                    if W > 1:       # the wide records the other ranks sent for keys this rank owns: one segment per source
                        base, recv_w = self._wide_segments
                        for src in range(W):
                            check(L.pg_wide_insert(byref(t.c), ctypes.c_void_p(base + src * self.cap_wide_wire * 16),
                                                   ctypes.c_void_p(recv_w.data_ptr() + 8 * src), self.cap_wide_wire, last, engine._stream()), "pg_wide_insert")
                    if ev is not None:
                        ev.setdefault("k2c", []).append((x2, x2c))
                        x2 = x2c
                elif self.region_bits:
                    # K2c: re-split level by level down to one bucket per region (the capacity may have been set from the
                    # key sample after K2a ran: the levels after the first follow the capacity in use)
                    region_log = (t.capacity >> self.region_bits).bit_length() - 1
                    levels = [self.sub_bits] + plan_levels(region_log, W)[1:] if region_log > self.sub_bits else [self.sub_bits]
                    if sum(levels) != region_log:              # sampled capacity: one or two even levels below K2a's buckets
                        rest = region_log - self.sub_bits
                        levels = [self.sub_bits] + ([rest] if rest <= 8 else [rest // 2, rest - rest // 2])
                    recs, cnts, bits, pcap, scap = bs.records, bs.counts, self.sub_bits, bs.c.part_cap, bs.c.spill_cap
                    bufs = [self.fine_records, bs.records]
                    for li, lb in enumerate(levels[1:]):
                        out, ocnt = bufs[li % 2], self.fine_counts[li]
                        n_out = 1 << (bits + lb)
                        ocap = (out.numel() // 2 - self.fine_spill_cap) // n_out
                        check(L.pg_records_resplit(P(recs), P(cnts), bits, pcap, scap, lb, P(out), P(ocnt), ocap, self.fine_spill_cap,
                                                   P(t.stats), engine._stream()), "pg_records_resplit")
                        recs, cnts, bits, pcap, scap = out, ocnt, bits + lb, ocap, self.fine_spill_cap
                    x2c = stamp(B)
                    check(L.pg_region_build(byref(t.c), P(recs), P(cnts), pcap, scap, 1 if r == 0 else 0, engine._stream()), "pg_region_build")
                    if ev is not None:
                        ev.setdefault("k2c", []).append((x2, x2c))
                        x2 = x2c
                else:
                    check(L.pg_buckets_plan(byref(bs.c), P(bs.seg_cnt), P(t.stats), engine._stream()), "pg_buckets_plan")
                    check(L.pg_insert_records(byref(t.c), P(bs.records), P(bs.seg_off), P(bs.seg_cnt), bs.n_parts + 1, 1, 0, engine._stream()),
                          "pg_insert_records")
                x3 = stamp(B)
                if W == 1:
                    self._ev_free[si] = torch.cuda.Event()
                    self._ev_free[si].record(B)
            if ev is not None:
                ev.setdefault("k2a", []).append((e0, e1))
                if W > 1:
                    ev.setdefault("count_exchange", []).append((x0, x1))
                    ev.setdefault("k2b", []).append((x1, x2))
                ev.setdefault("k3", []).append((x2, x3))
        cur.wait_stream(B)
        cur.wait_stream(A)
        return t

    # ------------------------------------------------------------------------------------------------
    def flags(self):
        """(table full, records lost) after a synchronise; agreed on by all ranks."""
        s = self.table.stats_host()
        f = torch.tensor([int(s[_lib.PG_STAT_OVERFLOW] != 0), int(s[_lib.PG_STAT_LOST] != 0), int(s[_lib.PG_STAT_USED])], dtype=torch.int64,
                         device=self.device)
        if self.world > 1:
            # a truncated record index poisons the wire counts: the receiver flags PG_STAT_LOST, so it is covered here
            dist.all_reduce(f, op=dist.ReduceOp.MAX)
        f = f.cpu()
        self._last_used = int(f[2])             # the fullest rank's distinct keys: every rank retunes to the same capacity
        return bool(f[0]), bool(f[1])

    def verify(self):
        full, lost = self.flags()
        if lost and self.compact:
            # the wide spill overflowed (many short records, long ambiguity runs): this input is not one for compact records
            self._compact_pref = False
            self._reconfigure = True               # begin() re-configures: 16-byte buffers, hash_kind 0
            raise LostRecords("the compact build's wide spill overflowed; the builder is back on 16-byte records")
        if lost:
            raise LostRecords("update records were dropped (bucket/spill overflow or a truncated record index) on some rank")
        if full:
            raise TableFull("dBG table overflow (capacity %d slots per rank)" % self.table.capacity)
        if self.adaptive:
            self.retune()

    def wire_records_peak(self):
        """The most records one source sent to one owner in one round of the last build, over all ranks (a collective).
        Above cap_wire, the records past the owner's receive segment were lost on the wire (or, on compact records,
        went to its wide segment)."""
        p = self.wire_peak.max().reshape(1)
        dist.all_reduce(p, op=dist.ReduceOp.MAX)
        return int(p.item())

    def retune(self, load=0.5):
        """Shared-memory region build: size the table for the NEXT build of this builder from the distinct keys the last one
        found (load <= ``load``; a serving loop sees inputs of one kind).  A K3s launch writes every slot of the table it
        is given and the stages after it scan every slot, so a table 4x too large costs 4x their HBM traffic; a table
        too small shows as TableFull and the caller rebuilds larger.  Never below one region per K2a bucket."""
        used = self._last_used
        want = engine.next_pow2(max(1024, int(used / load) + 1))
        limit = 1 << (self._region_pref + self.MAX_REGION_LOG)
        if want > limit and used <= 0.7 * limit:              # a denser table (load <= 0.7) that can still be built in regions
            want = limit
        self._next_capacity = want                            # applied by begin(): the table just built keeps its size

    def close(self):
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
            for q in self._opened:
                self.L.pg_peer_close(q)
            for p_ in self.own:
                self.L.pg_peer_free(p_)
            self._opened, self.own = [], []

    def describe(self):
        d = {"rounds": self.n_rounds, "round_len": self.round_len, "table_slots": self.table.capacity, "regions": 1 << self.sub_bits,
             "insert": ("K2c + K3s: %d shared-memory regions of %d slots, partition levels (bits) %r"
                        % (self.table.capacity >> self.region_bits, 1 << self.region_bits, self.levels))
                       if self.region_bits else "K3: L2 atomics over %d hash-prefix regions" % (1 << self.sub_bits),
             "records": "compact: 8 bytes per interior position, 16-byte wide records for the rest" if self.compact else "16 bytes",
             "record_buffers_bytes": sum(s.bytes() for s in self.sets) + (2 * self.wire_bytes if self.world > 1 else 0)}
        if self.world > 1:
            d["wire_bucket_records"] = self.cap_wire
        return d


def global_record_prefix(packed, Ns, strands, world=1):
    """How many of THIS rank's records a stage processes under ``-n`` when the file is split across ranks: the
    running base count (kmer_numba.py:1227, 1820, 1847) continues from the ranks before this one."""
    if world == 1:
        return packed.record_prefix(Ns, strands)
    mine = torch.tensor([int(packed.seq_lengths.sum()) * strands], dtype=torch.int64, device=packed.pk2.device)
    parts = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(parts, mine)
    before = sum(int(p.item()) for p in parts[:dist.get_rank()])
    if Ns - before < 0:
        return 0
    return packed.record_prefix(Ns - before, strands)


def build_table(packed, k, rc=True, Ns=2 ** 63, mode=None, world=1, rank=0, capacity=None, rounds=None, max_attempts=4,
                region_bits=None, sample=True, compact=None):
    """The product's stage-1 build: RoundBuilder with automatic recovery - more rounds (smaller buckets relative
    to their capacity) after lost records, a larger table after an overflow.  On one GPU the table is built in
    shared-memory regions and, for a single-round build, sized from K2a's key-space sample (``sample``) instead of the
    positions upper bound: the stages after it scan every slot.  Returns (DbgTable, n_rec, builder)."""
    k = int(min(max(1, k), 27))
    if mode is None:
        mode = _lib.PG_MODE_CANONICAL if rc else _lib.PG_MODE_LITERAL
    strands = 1 if mode == _lib.PG_MODE_LITERAL else 2
    n_rec = global_record_prefix(packed, Ns, strands, world)
    n_bases = int(packed.seq_off[n_rec] - packed.seq_off[0]) if n_rec > 0 else 0
    spill_frac, slack = 1.0 / 16, 1.25
    err = None
    for _ in range(max_attempts + 1):
        b = RoundBuilder(k, mode, max(n_bases, 1), world=world, rank=rank, device=packed.pk2.device, capacity=capacity, rounds=rounds,
                         slack=slack, spill_frac=spill_frac, region_bits=region_bits, sample=sample, compact=compact)
        b.adaptive = False              # one build: nothing to retune for
        b.begin()
        b.build_async(packed, n_rec)
        torch.cuda.synchronize()
        try:
            b.verify()
            return b.table, n_rec, b
        except LostRecords as e:
            err = e
            if b.compact:           # positions the compact records cannot hold overflowed the wide spill: 16-byte records
                compact = False
            elif world > 1:
                # across GPUs: a wire bucket (R / W * slack + 8192 records per source and owner) overflows when one owner
                # takes more than its share of a round - a hot key such as a long poly-A - and a local bucket when one
                # hash prefix does.  Either share stays the same however the stream is cut into rounds, so more rounds do
                # not help; a wider wire bucket (at slack W it holds a whole round) or a larger local spill does
                peak = b.wire_records_peak()
                if peak > b.cap_wire and slack < world:
                    slack = min(float(world), max(2 * slack, 1.05 * (peak - 8192) * world / b.round_len))
                else:
                    spill_frac = min(1.0, spill_frac * 4)
            else:
                rounds, spill_frac = 4 * b.n_rounds, min(1.0, spill_frac * 4)
        except TableFull as e:
            err = e
            capacity = 2 * b.table.capacity
            sample = False
        b.close()
        del b
    raise PgError("dBG build failed after %d attempts: %s" % (max_attempts, err))
