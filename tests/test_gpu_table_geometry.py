"""GPU parity of the streaming dBG builder at the edges of its table geometry, against the oracle: the product defaults
on the golden small cases (1-2 kb inputs land on a compact table of exactly one 4096-slot region), an explicit sweep of
region sizes and counts across the plan_levels boundaries and the K3 fallback, later upserts into one-region tables,
sampled capacities below the planned one, and retune() walking one builder across geometries.

Every table is checked three ways: its export equals the oracle's dBG, the unsorted export has unique keys, and the
inserts' claim counter (n_keys, read before count()) equals the slot scan (count()[0]) and the oracle's number of
distinct keys (canonical pairs under -c 2/3, literal keys under -c 0/1).  A key placed twice shows in all three."""
import numpy as np
import pytest

import oracle
from conftest import load_small_cases
from pangenome_b200.synth import _ACGT, fasta_bytes, pangenome

pytestmark = pytest.mark.gpu
CASES = load_small_cases()
_BY_NAME = {c["name"]: c for c in CASES}
_SENTINEL = np.uint64(0xFFFFFFFFFFFFFFFF)          # the short-record entry of an export
_REF = {}


@pytest.fixture(scope="module")
def mods():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pangenome_b200 import _lib, builder, engine, graph, stages
    return engine, builder, _lib, stages, graph


def ref(data, k, c=2, Ns=2 ** 63, stages=1):
    """oracle.run, once per input within this module"""
    key = (data, k, c, Ns, stages)
    if key not in _REF:
        _REF[key] = oracle.run(data, k, c=c, Ns=Ns, stages=stages)
    return _REF[key]


def golden_dbg(case):
    d = case["dbg"]
    return (np.array([e[0] for e in d], dtype=np.uint64), np.array([e[1] for e in d], dtype=np.uint16),
            np.array([e[2] for e in d], dtype=np.uint8))


def rc_codes(keys, k):
    """reverse complement of base-5 codes (digit i weighs 5^i; complement 3 - d, the ambiguity digit 4 stays)"""
    x, r = keys.copy(), np.zeros_like(keys)
    for _ in range(k):
        d = x % np.uint64(5)
        x //= np.uint64(5)
        r = r * np.uint64(5) + np.where(d == 4, d, np.uint64(3) - d)
    return r


def distinct_keys(keys, k, canonical):
    keys = keys[keys != _SENTINEL]
    if canonical:
        keys = np.minimum(keys, rc_codes(keys, k))
    return int(np.unique(keys).size)


def check_table(t, want, k, canonical, where):
    """the three checks of the module docstring against the oracle's (keys, vals, cnts)"""
    claimed = t.n_keys()                 # the inserts' own count; count() below replaces it by the slot scan
    scanned, _ = t.count()
    ks, vs, cs = t.export(sort=False)
    dup = ks.size - np.unique(ks).size
    o = np.argsort(ks, kind="stable")
    same = np.array_equal(ks[o], want[0]) and np.array_equal(vs[o], want[1]) and np.array_equal(cs[o], want[2])
    n = distinct_keys(want[0], k, canonical)
    assert dup == 0 and same and claimed == scanned == n, (
        "%s: %d duplicate keys in the export, export %s the oracle's (%d entries, oracle %d); claimed %d, slots %d, "
        "oracle %d distinct keys" % (where, dup, "equals" if same else "differs from", ks.size, want[0].size, claimed, scanned, n))


# ---------------------------------------------------------------------------------------------------------------------
# 1. the product defaults on the golden small cases

def _n_bases(case):
    r = ref(case["input_latin1"].encode("latin-1"), case["k"], case["c"], case.get("Ns", 2 ** 63))
    return int(r["seq_off"][-1] - r["seq_off"][0]) if r["n_records"] else 0


def _one_region_case(case):
    return bool((case["c"] >> 1) & 1) and 1024 <= _n_bases(case) < 2048


def test_golden_set_reaches_one_region_tables():
    """The canonical-mode cases of 1024-2047 bases get a 4096-slot table from the positions bound: one region of the
    compact build.  The golden set must keep holding such cases, or the next test stops covering that geometry."""
    names = [c["name"] for c in CASES if _one_region_case(c)]
    assert len(names) >= 9, names


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_product_defaults_golden(mods, case):
    eng, bld, _lib, stages, graph = mods
    data = case["input_latin1"].encode("latin-1")
    k, c, Ns = case["k"], case["c"], case.get("Ns", 2 ** 63)
    rc0, rc1 = bool((c >> 1) & 1), bool(c & 1)
    packed = eng.PackedSeqs(eng.to_device_bytes(data))
    t, n_rec, b = bld.build_table(packed, k, rc=rc0, Ns=Ns)
    if _one_region_case(case):
        assert (b.compact, t.capacity, b.region_bits) == (True, 4096, 12)
    check_table(t, golden_dbg(case), k, rc0, "build_table defaults (compact %s, %d slots, region_bits %d)"
                % (b.compact, t.capacity, b.region_bits))
    # the stage API on the same input: seq2rdbg -> rdBG -> seq2graph_device
    full = ref(data, k, c, Ns, stages=4)
    h = stages.seq2rdbg(None, kmer=k, Ns=Ns, rc=rc0, brkpt=None, data=np.frombuffer(data, dtype=np.uint8))
    assert h.table.capacity == t.capacity and h.builder.compact == b.compact
    rd = h.table.select_rdbg()
    rk, _ = rd.rdbg_export()
    assert np.array_equal(rk, full["rdbg"])
    res = graph.seq2graph_device(h.packed, rd, k, Ns=Ns, rc=rc1)
    assert res.xyz_lines() == full["xyz"]                  # same edges, weights and file order
    assert res.rows(h.packed, data) == full["rows"]


# ---------------------------------------------------------------------------------------------------------------------
# 2. an explicit sweep of region size, record form, region count and rounds

def mixed_records(seed=21, copies=15, block=1200):
    """Copies of one random block (about 2000 distinct 21-mers in all) with N runs, lowercase, IUPAC codes, and records
    of 0, k-1, k and k+2 bases: record edges and ambiguous positions travel as wide records (compact build) and the
    input spans three 8192-base rounds."""
    rng = np.random.default_rng(seed)
    base = _ACGT[rng.integers(0, 4, block)].tobytes()
    recs = []
    for i in range(copies):
        s = bytearray(base)
        a = int(rng.integers(0, block - 60))
        n = int(rng.integers(1, 30))
        s[a:a + n] = b"N" * n
        a = int(rng.integers(0, block - 60))
        s[a:a + 40] = bytes(s[a:a + 40]).lower()
        s[int(rng.integers(0, block))] = ord("RYKMSW"[i % 6])
        recs.append((b"m%d" % i, bytes(s)))
        n = (0, 20, 21, 23)[i % 4]
        a = int(rng.integers(0, block - n))
        recs.append((b"s%d" % i, base[a:a + n]))
    return fasta_bytes(recs, width=70)


def _sweep_input(name):
    if name == "golden":
        case = _BY_NAME["rand13_k15_c2"]                   # 1563 bases
        return case["input_latin1"].encode("latin-1"), case["k"]
    if name == "pangenome":
        return pangenome(3, 20_000), 21
    return mixed_records(), 21


# region counts (log2) per (region_bits, compact): 1 and 2 regions, either side of each plan_levels boundary, and the
# region_bits 8 table past MAX_REGION_LOG that must fall back to the L2-atomic K3
_SWEEP = {(12, True): [0, 1, 8, 9, 17, 18], (12, False): [0, 1, 8, 9], (8, False): [0, 1, 8, 9, 16, 17, 18, 19]}
_LEVELS = {(True, 17): [8, 9], (True, 18): [8, 5, 5], (False, 8): [8], (False, 9): [8, 1], (False, 16): [8, 8],
           (False, 17): [8, 4, 5], (False, 18): [8, 5, 5]}


@pytest.mark.parametrize("rb,compact", list(_SWEEP), ids=["%d-%s" % (rb, "compact" if c else "16B") for rb, c in _SWEEP])
@pytest.mark.parametrize("inp", ["golden", "pangenome", "mixed"])
def test_capacity_sweep(mods, inp, rb, compact):
    import torch
    eng, bld, _lib, _, _ = mods
    data, k = _sweep_input(inp)
    r = ref(data, k)
    assert r["ub_count"] == 0
    want = r["dbg"]
    n_keys = distinct_keys(want[0], k, True)
    packed = eng.PackedSeqs(eng.to_device_bytes(data))
    ran = []
    for rl in _SWEEP[(rb, compact)]:
        cap = 1 << (rb + rl)
        if cap < 1.5 * n_keys:                             # keep the load below 2/3: the input does not fit this table
            continue
        if compact and rl >= 17:                           # 8 and 16 GiB tables
            torch.cuda.empty_cache()
            if torch.cuda.mem_get_info()[0] < 2 * 16 * cap:
                continue
        for rounds in (1, 3):
            where = "%s: region_bits %d, %s records, 2^%d regions, %d rounds" % (inp, rb, "compact" if compact else "16-byte", rl, rounds)
            t, n_rec, b = bld.build_table(packed, k, capacity=cap, rounds=rounds, region_bits=rb, compact=compact, sample=False)
            assert t.capacity == cap, where
            if rl <= bld.RoundBuilder.MAX_REGION_LOG:
                assert (b.region_bits, b.compact, t.c.region_bits) == (rb, compact, rb), where
                if (compact, rl) in _LEVELS:
                    assert b.levels == _LEVELS[(compact, rl)], where
            else:
                assert b.region_bits == 0 and not b.compact and t.c.region_bits == 0, where
            assert b.n_rounds == (1 if inp == "golden" else rounds), where          # rounds are whole 8192-base tiles
            if compact and inp == "mixed":
                assert max(int(s.wide_count.item()) for s in b.sets) > 0, where
            check_table(t, want, k, True, where)
            ran.append(rl)
            del t, b
    torch.cuda.empty_cache()
    assert ran, "no geometry fits this input"


# ---------------------------------------------------------------------------------------------------------------------
# 3. one-region tables take later writes

@pytest.mark.parametrize("rb,compact,cap,name", [(12, True, 4096, "rand13_k15_c2"), (12, False, 4096, "rand13_k15_c2"),
                                                 (8, False, 256, "rand17_k4_c2")])
def test_one_region_table_takes_later_upserts(mods, rb, compact, cap, name):
    """The fused insert (pg_kmer_insert) into a table K3s / K3s-c built as one region probes from the same home: adding
    the same records again only doubles the counts."""
    eng, bld, _, _, _ = mods
    case = _BY_NAME[name]
    data, k = case["input_latin1"].encode("latin-1"), case["k"]
    assert data.startswith(b">") and data.endswith(b"\n")
    packed = eng.PackedSeqs(eng.to_device_bytes(data))
    t, n_rec, b = bld.build_table(packed, k, capacity=cap, region_bits=rb, compact=compact, sample=False)
    assert (t.capacity, b.region_bits, b.compact, t.c.region_bits, b.levels) == (cap, rb, compact, rb, [0])
    check_table(t, ref(data, k)["dbg"], k, True, "%s: one region, build" % name)
    t.insert(packed, n_rec)
    check_table(t, ref(data + data.replace(b">", b">x"), k)["dbg"], k, True, "%s: one region, build + insert" % name)


def test_one_region_spill_upserts(mods):
    """A 16-byte one-region build whose bucket overflows: the surplus goes through the spill's L2-atomic upserts into
    the region K3s built, and must meet the keys already there."""
    import torch
    eng, bld, _lib, _, _ = mods
    case = _BY_NAME["rand13_k15_c2"]
    data, k = case["input_latin1"].encode("latin-1"), case["k"]
    packed = eng.PackedSeqs(eng.to_device_bytes(data))
    b = bld.RoundBuilder(k, _lib.PG_MODE_CANONICAL, len(data), capacity=4096, region_bits=12, compact=False, slack=1.0, spill_frac=1.0)
    assert b.region_bits == 12 and not b.compact and b.levels == [0] and b.sets[0].n_parts == 1
    b.sets[0].c.part_cap = b.sets[0].part_cap = 256          # far below the input's 1563 positions
    b.sets[0].seg_off.copy_(torch.arange(b.sets[0].n_parts + 1, device="cuda") * 256)
    b.begin()
    t = b.build_async(packed, packed.n_rec)
    torch.cuda.synchronize()
    b.verify()
    assert int(b.sets[0].counts[-1].item()) > 0               # the spill really was used
    check_table(t, ref(data, k)["dbg"], k, True, "one region + spill")


# ---------------------------------------------------------------------------------------------------------------------
# 4. a sampled capacity below the planned one

def repetitive(block, copies, rate=0.0005, seed=3):
    """``copies`` copies of one random block, each with substitutions at ``rate``: about ``block`` distinct keys over
    ``block * copies`` positions"""
    rng = np.random.default_rng(seed)
    anc = rng.integers(0, 4, block, dtype=np.uint8)
    recs = []
    for i in range(copies):
        s = anc.copy()
        m = rng.random(block) < rate
        s[m] = (s[m] + rng.integers(1, 4, int(m.sum()), dtype=np.uint8)) % 4
        recs.append((b"c%d" % i, _ACGT[s]))
    return fasta_bytes(recs)


@pytest.mark.parametrize("compact", [True, False], ids=["compact", "16B"])
@pytest.mark.parametrize("block,copies,regions", [(100_000, 30, (1 << 8,)), (750_000, 4, (1 << 9, 1 << 10))],
                         ids=["no-K2c", "one-K2c-level"])
def test_sampled_capacity_below_planned(mods, block, copies, regions, compact):
    """3 Mbp plan 2^23 slots (2^11 regions, K2a into 2^8 buckets + one K2c level of 2^3).  The key sample then shrinks
    the table after K2a ran: to 2^8 regions, one per K2a bucket (no K2c pass), or to 2^9 / 2^10 regions (one K2c level
    the plan did not have)."""
    eng, bld, _, _, _ = mods
    data = repetitive(block, copies)
    packed = eng.PackedSeqs(eng.to_device_bytes(data))
    t, n_rec, b = bld.build_table(packed, 21, compact=compact)
    planned = (t.slots.numel() // 2) >> 12
    assert 1 << 11 <= planned <= 1 << 13 and b.sub_bits == 8 and b.sampler is not None
    assert (b.region_bits, b.compact) == (12, compact)
    assert t.capacity >> 12 in regions, "sampled capacity %d slots" % t.capacity
    check_table(t, ref(data, 21)["dbg"], 21, True, "sampled %d slots of %d planned regions" % (t.capacity, planned))


# ---------------------------------------------------------------------------------------------------------------------
# 5. retune() walks one builder across geometries

def test_retune_across_geometries(mods):
    """One adaptive builder, inputs of about 6000, 1500, 700 and 300 distinct keys, each built twice: the capacity walks
    16384 -> 4096 (one region, compact) -> 2048 -> 1024 (16-byte records, L2-atomic K3) and every table is exact."""
    import torch
    eng, bld, _lib, _, _ = mods
    rng = np.random.default_rng(8)
    inputs = [fasta_bytes([(b"r%d" % n, _ACGT[rng.integers(0, 4, n)])]) for n in (6000, 1500, 700, 300)]
    b = bld.RoundBuilder(21, _lib.PG_MODE_CANONICAL, max(len(d) for d in inputs))
    assert b.adaptive
    seen = []
    for i, data in enumerate(inputs):
        packed = eng.PackedSeqs(eng.to_device_bytes(data))
        for rep in range(2):
            b.begin()
            t = b.build_async(packed, packed.n_rec)
            torch.cuda.synchronize()
            b.verify()
            seen.append((t.capacity, b.compact, b.region_bits, type(b.sets[0]).__name__))
            check_table(t, ref(data, 21)["dbg"], 21, True, "input %d build %d: %r" % (i, rep, seen[-1]))
    assert seen == [(16384, True, 12, "CompactBuckets")] * 3 + [(4096, True, 12, "CompactBuckets")] * 2 + \
        [(2048, False, 0, "LocalBuckets")] * 2 + [(1024, False, 0, "LocalBuckets")], seen
