"""The hash-partitioned multi-GPU build with W ranks on ONE device: W processes on cuda:0 that talk over gloo.  NCCL
refuses two ranks on one device; gloo does not, and the builder cannot tell the difference - the peer stores go through
CUDA IPC between processes of one device, and a gloo collective on CUDA tensors reads its input after the current
stream's work and returns only when every rank's input has arrived, so the count exchange still orders the peer stores.
This runs the world > 1 kernels (K2a-c / K2a in their PEER form, the compact overflow-to-owner path, K2b-c / K2b, one
wide upsert per source rank) and the host choreography around them on a one-GPU machine.

Every table is compared with oracle.run on the whole file, bit for bit, through the merged export, and checked for
the partition's invariants: the ranks' exports are pairwise disjoint, every rank's claim counter (PG_STAT_USED) equals
its slot scan, and the claims summed over ranks equal the oracle's distinct keys.

The ranks are started with torch.multiprocessing.spawn and joined: a rank that fails ends the others, and a
collective that waits for a failed rank times out."""
import ctypes
import datetime
import os
import socket

import numpy as np
import pytest

import oracle
from conftest import load_small_cases

pytestmark = pytest.mark.gpu
CASES = load_small_cases()
_SENTINEL = np.uint64(0xFFFFFFFFFFFFFFFF)


def _compute_mode_default():
    """True when device 0 runs in the Default compute mode (read through the CUDA runtime; nothing is changed): under
    an exclusive mode a second context on the device cannot exist."""
    import torch
    torch.cuda.init()                   # the runtime torch loaded answers to its soname
    lib = ctypes.CDLL("libcudart.so.12")
    mode = ctypes.c_int(-1)
    cuda_dev_attr_compute_mode = 20     # cudaDevAttrComputeMode; 0 = cudaComputeModeDefault
    rc = lib.cudaDeviceGetAttribute(ctypes.byref(mode), cuda_dev_attr_compute_mode, 0)
    return rc == 0 and mode.value == 0


@pytest.fixture(scope="module")
def launch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    if not _compute_mode_default():
        pytest.skip("device 0 is not in the Default compute mode: no second process can use it")
    from pangenome_b200 import _lib
    _lib.load()                 # build the library here, so the ranks never run nvcc at the same time

    def run(fn, world, *args):
        import torch.multiprocessing as mp
        with socket.socket() as s:          # a free rendezvous port
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        mp.spawn(_rank_main, args=(world, port, fn, args), nprocs=world, join=True)
    return run


def _rank_main(rank, world, port, fn, args):
    import torch
    import torch.distributed as dist
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=600))
    try:
        fn(rank, world, *args)
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------------
# helpers, run inside the ranks

def _mods():
    from pangenome_b200 import _lib, builder, engine, multigpu, shard
    return _lib, builder, engine, multigpu, shard


def _rank_input(data, world, rank):
    """this rank's record-aligned byte range of the file, packed; and its number of bases"""
    _, _, engine, _, shard = _mods()
    cuts = shard.cut_points(data, world)
    mine = data[cuts[rank]:cuts[rank + 1]]
    packed = engine.PackedSeqs(engine.to_device_bytes(mine))
    n_bases = int(packed.seq_off[packed.n_rec] - packed.seq_off[0]) if packed.n_rec else 0
    return packed, n_bases


def _rc_codes(keys, k):
    x, r = keys.copy(), np.zeros_like(keys)
    for _ in range(k):
        d = x % np.uint64(5)
        x //= np.uint64(5)
        r = r * np.uint64(5) + np.where(d == 4, d, np.uint64(3) - d)
    return r


def _distinct_keys(keys, k, canonical):
    keys = keys[keys != _SENTINEL]
    if canonical:
        keys = np.minimum(keys, _rc_codes(keys, k))
    return int(np.unique(keys).size)


def _check(t, want, k, canonical, world, rank, where):
    """The merged export equals the oracle's dBG ``want``; the ranks' key sets are disjoint; every rank's claim counter
    equals its slot scan; the claims add up to the oracle's distinct keys.  A collective: every rank calls it.
    Returns the per-rank (claimed, scanned, short records) on rank 0."""
    import torch.distributed as dist
    _lib, _, _, multigpu, _ = _mods()
    claimed = t.n_keys()                    # the inserts' own count; count() replaces it by the slot scan
    scanned, _ = t.count()
    ks, _, _ = t.export(sort=False)
    short = int(t.stats_host()[_lib.PG_STAT_SHORT])
    parts = [None] * world
    dist.all_gather_object(parts, (claimed, scanned, short, ks[ks != _SENTINEL]))
    merged = multigpu.gather_export(t, world, rank)
    if rank != 0:
        return None
    allk = np.concatenate([p[3] for p in parts])
    n = _distinct_keys(want[0], k, canonical)
    per_rank = [(p[0], p[1]) for p in parts]
    assert allk.size == np.unique(allk).size, "%s: %d keys live on more than one rank (or twice on one)" % (where, allk.size - np.unique(allk).size)
    assert all(c == s for c, s in per_rank), "%s: claim counters differ from the slot scans: %r" % (where, per_rank)
    assert sum(c for c, _ in per_rank) == n, "%s: claims %r add up to %d, oracle %d distinct keys" % (where, per_rank, sum(c for c, _ in per_rank), n)
    ks, vs, cs = merged
    same = np.array_equal(ks, want[0]) and np.array_equal(vs, want[1]) and np.array_equal(cs, want[2])
    assert same, "%s: merged export (%d entries) differs from the oracle's (%d)" % (where, ks.size, want[0].size)
    return [(p[0], p[1], p[2]) for p in parts]


def _oracle_dbg(rank, data, k, c=2, Ns=2 ** 63):
    return oracle.run(data, k, c=c, Ns=Ns, stages=1)["dbg"] if rank == 0 else None


def _round_build(data, k, mode, world, rank, builds=1, **kw):
    """RoundBuilder on this rank's range, ``builds`` builds (no recovery: a wrong configuration raises)"""
    import torch
    _, builder, _, _, _ = _mods()
    packed, n_bases = _rank_input(data, world, rank)
    b = builder.RoundBuilder(k, mode, max(n_bases, 1), world=world, rank=rank, **kw)
    for _ in range(builds):
        b.begin()
        t = b.build_async(packed, packed.n_rec)
        torch.cuda.synchronize()
        b.verify()
    return b, t


# ---------------------------------------------------------------------------------------------------------------------
# inputs

def _rng_seq(rng, n):
    from pangenome_b200.synth import _ACGT
    return _ACGT[rng.integers(0, 4, n, dtype=np.uint8)]


def _revcomp(s):
    return s[::-1].translate(bytes.maketrans(b"ACGT", b"TGCA"))


def _mixed_input(world, seed=1):
    """diverged copies of one ancestor, one of them with N runs and lower-case bases; records that hold palindromes of
    even length (20: the fold bit at k 20); a poly-A; and 120 records per rank shorter than any k here, spread evenly
    through the file.  The short-record sentinel counts a short record once per strand: 240 per rank in canonical mode,
    below the clamp at 255 on every rank and above it only once the ranks' counts are summed"""
    from pangenome_b200 import synth
    rng = np.random.default_rng(seed)
    anc = rng.integers(0, 4, 12000, dtype=np.uint8)
    recs = []
    for g in range(2 * world):
        s = bytes(synth._ACGT[synth._snp_copy(np.random.default_rng(100 + g), anc, 0.03)])
        if g == 1:
            s = s[:3000] + b"N" * 40 + s[3040:6000].lower() + b"NNRYN" + s[6005:]
        recs.append((b"g%d" % g, s))
        for j in range(60):
            recs.append((b"s%d_%d" % (g, j), b"ACG"))
        h = bytes(_rng_seq(rng, 10))
        recs.append((b"pal%d" % g, bytes(_rng_seq(rng, 7)) + h + _revcomp(h) + bytes(_rng_seq(rng, 9)) + h + _revcomp(h)))
    recs.append((b"polyA", b"A" * 3000))
    return synth.fasta_bytes(recs, width=70)


def _small_input(world, n_per_rank=900, copies=1, seed=7):
    """about ``n_per_rank`` distinct bases per rank in 6 records per rank, with an ambiguity run and a short record;
    the whole set ``copies`` times over (the keys stay, the stream grows: several rounds over a small table)"""
    from pangenome_b200 import synth
    rng = np.random.default_rng(seed)
    recs = []
    for i in range(6 * world):
        s = bytes(_rng_seq(rng, n_per_rank // 6))
        if i == 2:
            s = s[:40] + b"NN" + s[42:]
        recs.append((b"r%d" % i, s))
    recs.append((b"short", b"ACGT"))
    return synth.fasta_bytes([(b"%s_%d" % (h, c), s) for c in range(copies) for h, s in recs], width=60)


# ---------------------------------------------------------------------------------------------------------------------
# 1. mg_check.py's checks (checksum over repeated builds, dBG, rdBG / .xyz / rows, CLI, CLI --cluster mcl) at W ranks

def _mg_check(rank, world):
    import mg_check
    mg_check.main(["--one-device"])


@pytest.mark.parametrize("world", [2, 4, 8])
def test_mg_check_one_device(launch, world):
    launch(_mg_check, world)


# ---------------------------------------------------------------------------------------------------------------------
# 2. every K2a-c flavour (k 27 / 21 compile-time, 15 / 20 runtime; 20 is even: palindromes) on both record forms

_FORMS = [("compact", 2, None, True), ("16-byte", 2, False, False), ("literal -c 0", 0, None, False)]


def _flavours(rank, world):
    _lib = _mods()[0]
    data = _mixed_input(world)
    for k in (27, 21, 15, 20):
        for form, c, compact, want_compact in _FORMS:
            mode = _lib.PG_MODE_CANONICAL if c & 2 else _lib.PG_MODE_LITERAL
            want = _oracle_dbg(rank, data, k, c)
            for rounds in (1, 3):
                b, t = _round_build(data, k, mode, world, rank, builds=2, rounds=rounds, compact=compact)
                assert b.compact == want_compact and b.region_bits == 12
                parts = _check(t, want, k, bool(c & 2), world, rank, "k %d %s rounds %d" % (k, form, rounds))
                if rank == 0:
                    shorts = [p[2] for p in parts]
                    assert max(shorts) < 255 and min(shorts) > 0, shorts
                    assert sum(shorts) > 255 or not c & 2, shorts      # literal mode (one strand) clamps from W = 4
                b.close()


@pytest.mark.parametrize("world", [2, 4])
def test_k2a_flavours_and_record_forms(launch, world):
    launch(_flavours, world)


# ---------------------------------------------------------------------------------------------------------------------
# 3. the edges of the partition

def _golden(rank, world):
    _, builder, _, _, _ = _mods()
    for case in CASES:
        data = case["input_latin1"].encode("latin-1")
        k, c, Ns = case["k"], case["c"], case.get("Ns", 2 ** 63)
        packed, _ = _rank_input(data, world, rank)
        t, _, b = builder.build_table(packed, k, rc=bool(c & 2), Ns=Ns, world=world, rank=rank, max_attempts=0)
        _check(t, _oracle_dbg(rank, data, k, c, Ns), k, bool(c & 2), world, rank,
               "%s (compact %s, %d slots, region_bits %d)" % (case["name"], b.compact, t.capacity, b.region_bits))
        b.close()


@pytest.mark.parametrize("world", [2, 4])
def test_golden_small_cases(launch, world):
    """75 B - 2.1 kB inputs: per-rank tables of 1024-4096 slots (below one region: the L2-atomic K3 on 16-byte records;
    one region: K2b-c into a single bucket), and ranks that receive no record at all"""
    launch(_golden, world)


# (capacity, region_bits, compact) -> (b.compact, b.region_bits, b.levels)
_SWEEP = [
    ((2048, None, None), (False, 0, None)),            # below one region: K3 with L2 atomics
    ((4096, None, None), (True, 12, [0])),             # one region
    ((4096, None, False), (False, 12, [0])),
    ((8192, None, None), (True, 12, [1])),             # two regions
    ((8192, None, False), (False, 12, [1])),
    ((1 << 20, None, None), (True, 12, [8])),          # plan_levels(8, W): one level; 9: two
    ((1 << 21, None, None), (True, 12, [6, 3])),
    ((1 << 21, None, False), (False, 12, [6, 3])),
    ((2048, 8, None), (False, 8, [3])),                # 256-slot regions
    ((1 << 16, 8, None), (False, 8, [8])),
    ((1 << 17, 8, None), (False, 8, [6, 3])),
]


def _sweep(rank, world):
    _lib = _mods()[0]
    data, k = _small_input(world, copies=24), 21          # about 21 kb per rank: three rounds of 8192 positions
    want = _oracle_dbg(rank, data, k)
    for (cap, rb, compact), geo in _SWEEP:
        for rounds in (1, 3):
            b, t = _round_build(data, k, _lib.PG_MODE_CANONICAL, world, rank, builds=2, capacity=cap, region_bits=rb,
                                compact=compact, rounds=rounds)
            where = "capacity %d region_bits %s compact %s rounds %d" % (cap, rb, compact, rounds)
            assert (b.compact, b.region_bits, b.levels) == geo and t.capacity == cap and b.n_rounds == rounds, (
                where, b.compact, b.region_bits, b.levels, b.n_rounds)
            _check(t, want, k, True, world, rank, where)
            b.close()


@pytest.mark.parametrize("world", [2, 4])
def test_geometry_sweep(launch, world):
    launch(_sweep, world)


def _sizing_one_region(rank, world):
    import torch
    _lib, builder, _, _, _ = _mods()
    data, k = _small_input(world, n_per_rank=1440), 21
    want = _oracle_dbg(rank, data, k)
    # the sizing reaches one region on its own: about 1.4 kB per rank
    packed, n_bases = _rank_input(data, world, rank)
    t, _, b = builder.build_table(packed, k, world=world, rank=rank, max_attempts=0)
    assert (b.compact, t.capacity, b.region_bits, b.levels) == (True, 4096, 12, [0])
    _check(t, want, k, True, world, rank, "build_table, one region from the positions bound")
    b.close()
    # retune(): a builder sized for 40 kb per rank finds 1024-2047 keys per rank and moves to 4096 slots
    b = builder.RoundBuilder(k, _lib.PG_MODE_CANONICAL, 40000, world=world, rank=rank)
    assert b.table.capacity > 4096
    for it in range(3):
        b.begin()
        t = b.build_async(packed, packed.n_rec)
        torch.cuda.synchronize()
        b.verify()
        if it > 0:
            assert (b.compact, t.capacity, b.region_bits, b.levels) == (True, 4096, 12, [0])
        _check(t, want, k, True, world, rank, "retuned builder, build %d (%d slots)" % (it, t.capacity))
    b.close()


def test_one_region_from_sizing_and_retune(launch):
    launch(_sizing_one_region, 2)


def _wire_overflow(rank, world):
    """rank 0's range is mostly one poly-A: its wire bucket for that key's owner overflows and the surplus travels as
    compact-in-wide records into the owner's wide segment (wide_emit_compact_owner).  The table stays exact."""
    import torch.distributed as dist
    _lib = _mods()[0]
    from pangenome_b200 import synth
    rng = np.random.default_rng(5)
    data = synth.fasta_bytes([(b"hot", b"A" * 60000 + bytes(_rng_seq(rng, 4000))), (b"cold", bytes(_rng_seq(rng, 64000)))], width=80)
    k = 21
    b, t = _round_build(data, k, _lib.PG_MODE_CANONICAL, world, rank, rounds=1)
    assert b.compact and b.n_rounds == 1
    sent = b.csend_counts[0].cpu().numpy()           # one build of one round: buffer 0; [compact | wide] per owner
    parts = [None] * world
    dist.all_gather_object(parts, (sent, b.cap_wire))
    _check(t, _oracle_dbg(rank, data, k), k, True, world, rank, "wire bucket overflow")
    if rank == 0:
        s0, cw = parts[0]
        owner = int(np.argmax(s0[:world]))
        assert s0[owner] > cw, "rank 0 sent %d compact records to rank %d, its bucket holds %d: no overflow" % (s0[owner], owner, cw)
        assert s0[world + owner] >= s0[owner] - cw, "the surplus did not go to the owner's wide segment: %r" % (s0,)
    b.close()


def test_wire_bucket_overflow_compact(launch):
    launch(_wire_overflow, 2)


def _short_records(rank, world):
    """16384 records of 16 bases at k 3: no 16-position group is interior, so every k-mer travels as a wide record and
    the wide wire segment (cap_wire / 2) overflows.  verify() raises LostRecords; build_table recovers on 16-byte records."""
    _lib, builder, _, _, _ = _mods()
    from pangenome_b200 import synth
    rng = np.random.default_rng(11)
    data = synth.fasta_bytes([(b"%d" % i, bytes(_rng_seq(rng, 16))) for i in range(16384)], width=80)
    k = 3
    with pytest.raises(builder.LostRecords):
        _round_build(data, k, _lib.PG_MODE_CANONICAL, world, rank, rounds=1)
    packed, _ = _rank_input(data, world, rank)
    t, _, b = builder.build_table(packed, k, world=world, rank=rank)
    assert not b.compact
    _check(t, _oracle_dbg(rank, data, k), k, True, world, rank, "many short records")
    b.close()


def test_short_records_overflow_wide_wire(launch):
    launch(_short_records, 2)


def _owner_skew(rank, world):
    """rank 0's 2 Mbp range is 60 % poly-A: one owner takes far more than 1.25 / W of it in every round however the
    stream is cut, so 16-byte records lose records on the wire at 1 and at 16 rounds; build_table widens the wire
    bucket and returns the oracle's table"""
    _lib, builder, _, _, _ = _mods()
    from pangenome_b200 import synth
    rng = np.random.default_rng(13)
    recs = [(b"hot", bytes(_rng_seq(rng, 800_000)) + b"A" * 1_200_000)]
    recs += [(b"cold%d" % i, bytes(_rng_seq(rng, 2_000_000))) for i in range(world - 1)]
    data = synth.fasta_bytes(recs, width=80)
    k = 21
    for rounds in (1, 16):
        with pytest.raises(builder.LostRecords):
            _round_build(data, k, _lib.PG_MODE_CANONICAL, world, rank, rounds=rounds, compact=False)
    packed, _ = _rank_input(data, world, rank)
    t, _, b = builder.build_table(packed, k, world=world, rank=rank)
    _check(t, _oracle_dbg(rank, data, k), k, True, world, rank, "owner skew (slack %.2f, %d rounds)" % (b._slack, b.n_rounds))
    b.close()


def test_owner_skew_recovers(launch):
    launch(_owner_skew, 4)
