"""CPU check of the kernels' per-thread integer logic (tests/host_emul.cu runs the
same host+device functions the CUDA kernels call) against the oracle and the
reference's golden vectors.  No GPU needed."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import oracle
from conftest import ROOT, load_small_cases
from pangenome_b200.synth import survey_4x1m

CASES = load_small_cases()
_SO = os.path.join(ROOT, "tests", "_host_emul.so")


@pytest.fixture(scope="module")
def emul():
    src = os.path.join(ROOT, "tests", "host_emul.cu")
    deps = [src] + [os.path.join(ROOT, "pangenome_b200", "csrc", f) for f in
                    ("fasta_chunk.cuh", "kmer_core.cuh", "common.cuh")]
    if not os.path.isfile(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps):
        # compiled under a private name and renamed into place: parallel test workers never load a half-written library
        tmp = "%s.%d.so" % (_SO[:-3], os.getpid())
        subprocess.check_call(["nvcc", "-O2", "-std=c++17", "--shared", "-Xcompiler", "-fPIC", "-o", tmp, src])
        os.replace(tmp, _SO)
    L = ctypes.CDLL(_SO)
    L.emul_pack.restype = ctypes.c_int64
    L.emul_pack2.restype = ctypes.c_int64
    L.emul_pack3.restype = ctypes.c_int64
    L.emul_dbg.restype = ctypes.c_int64
    return L


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def run_pack(L, data, fn="emul_pack"):
    n = len(data)
    buf = np.frombuffer(data, dtype=np.uint8) if n else np.zeros(1, np.uint8)
    nw = n // 16 + 64
    pk2 = np.zeros(nw, np.uint32)
    amb = np.zeros(nw, np.uint32)
    cap = max(16, data.count(b">") + 1)
    hdr = np.zeros(cap + 1, np.int64)
    so = np.zeros(cap + 2, np.int64)
    counts = np.zeros(4, np.int64)
    rc = getattr(L, fn)(_p(buf), ctypes.c_int64(n), _p(pk2), _p(amb), ctypes.c_int64(nw), _p(hdr), _p(so),
                        ctypes.c_int64(cap), _p(counts))
    assert rc >= 0, "tile summary disagrees with the final pass in tile %d" % (-rc - 1000)
    nrec = int(counts[0])
    return pk2, amb, hdr[:nrec], so[:nrec + 1], counts


def unpack_syms(pk2, amb, n):
    i = np.arange(n)
    d = (pk2[i >> 4] >> (2 * (i & 15)).astype(np.uint32)) & 3
    a = (amb[i >> 5] >> (i & 31).astype(np.uint32)) & 1
    return np.where(a == 1, 4 + d, d).astype(np.uint8)


def syms_of_bytes(seq):
    lut = np.full(256, 5, np.uint8)
    for ch, v in ((b"Aa", 0), (b"Gg", 1), (b"Cc", 2), (b"Tt", 3), (b"Nn", 4)):
        for c in ch:
            lut[c] = v
    return lut[seq]


def run_dbg(L, pk2, amb, so, k, mode):
    nrec = so.size - 1
    cap = int(2 * max(1, so[-1]) + 8)
    keys = np.zeros(cap, np.uint64)
    vals = np.zeros(cap, np.uint16)
    cnts = np.zeros(cap, np.uint8)
    rkeys = np.zeros(cap, np.uint64)
    rvals = np.zeros(cap, np.uint16)
    nr = np.zeros(1, np.int64)
    n = L.emul_dbg(_p(pk2), _p(amb), ctypes.c_int64(pk2.size), _p(so), ctypes.c_int64(nrec), ctypes.c_int(k),
                   ctypes.c_int(mode), _p(keys), _p(vals), _p(cnts), ctypes.c_int64(cap), _p(rkeys), _p(rvals),
                   ctypes.c_int64(cap), _p(nr))
    o = np.argsort(keys[:n], kind="stable")
    ro = np.argsort(rkeys[:int(nr[0])], kind="stable")
    return (keys[:n][o], vals[:n][o], cnts[:n][o]), rkeys[:int(nr[0])][ro]


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_emul_matches_golden(emul, case):
    if "Ns" in case:
        pytest.skip("-n prefix selection is host logic, tested with the host module")
    data = case["input_latin1"].encode("latin-1")
    ref = oracle.run(data, case["k"], c=case["c"], stages=2)
    pk2, amb, hdr, so, counts = run_pack(emul, data)
    assert so.tolist() == ref["seq_off"].tolist()
    assert hdr.tolist() == ref["hdr_off"].tolist()
    junk = int(so[0]) if so.size else 0
    got = unpack_syms(pk2, amb, int(counts[1]))[junk:]
    assert got.tolist() == syms_of_bytes(ref["seq"]).tolist()
    rc0 = (case["c"] >> 1) & 1
    modes = (1, 2) if rc0 else (0,)
    for mode in modes:
        (ks, vs, cs), rk = run_dbg(emul, pk2, amb, so, case["k"], mode)
        got = [[int(a), int(b), int(c)] for a, b, c in zip(ks, vs, cs)]
        assert got == case["dbg"], "mode %d" % mode
        assert rk.tolist() == case["rdbg"], "mode %d" % mode


def test_emul_header_offsets(emul):
    data = b"junk\n>s1 desc\nACGT\nAC\n>s2\n\n>s3\nGGGTT"
    pk2, amb, hdr, so, counts = run_pack(emul, data)
    assert hdr.tolist() == [5, 22, 27]
    assert so.tolist() == [4, 10, 10, 14]          # 'junk' occupies [0,4) and belongs to no record
    assert counts[0] == 3 and counts[1] == 14
    # a file without any newline yields no line at all
    pk2, amb, hdr, so, counts = run_pack(emul, b">x ACGT")
    assert counts[0] == 0 and counts[1] == 0


def test_emul_big(emul, big_facts):
    data = survey_4x1m()
    pk2, amb, hdr, so, counts = run_pack(emul, data)
    assert counts[0] == 4 and int(so[-1]) == 4_000_000
    (ks, vs, cs), rk = run_dbg(emul, pk2, amb, so, 27, 2)
    assert ks.size == big_facts["dbg_entries"]
    assert int(cs.astype(np.int64).sum()) == big_facts["dbg_count_sum"]
    ref = oracle.run(data, 27, stages=2)
    assert np.array_equal(ks, ref["dbg"][0]) and np.array_equal(vs, ref["dbg"][1]) and np.array_equal(cs, ref["dbg"][2])
    assert np.array_equal(rk, ref["rdbg"])
    assert oracle.table_checksum(ks, vs, cs) == oracle.table_checksum(*ref["dbg"])


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_emul_single_pass_pack_matches_golden(emul, case):
    """the single-pass K1 formulation (states from the last newline, tile_sum3) == the oracle's parse"""
    data = case["input_latin1"].encode("latin-1")
    ref = oracle.run(data, case["k"], c=case["c"], stages=1)
    for fn in ("emul_pack2", "emul_pack3"):
        pk2, amb, hdr, so, counts = run_pack(emul, data, fn)
        assert so.tolist() == ref["seq_off"].tolist(), fn
        assert hdr.tolist() == ref["hdr_off"].tolist(), fn
        assert unpack_syms(pk2, amb, int(counts[1])).tolist() == syms_of_bytes(ref["seq"]).tolist(), fn


def test_emul_single_pass_pack_hostile_layouts(emul):
    rng = np.random.default_rng(5)
    alph = np.frombuffer(b"ACGTNacgtRY>\n\n\r", dtype=np.uint8)
    for it in range(300):
        n = int(rng.integers(0, 70000 if it % 10 == 0 else 3000))
        body = bytes(rng.choice(alph, size=n, p=[.2, .2, .2, .2, .02, .01, .01, .01, .01, .01, .01, .03, .04, .03, .02]).tolist())
        data = (b">h\n" if it % 3 else b"") + body
        ref = oracle.run(data, 5, stages=1)
        a = run_pack(emul, data, "emul_pack")
        nb = int(a[4][1])
        assert (a[3] - a[3][0]).tolist() == ref["seq_off"].tolist(), data[:80]      # bases before the first header stay in the stream
        for fn in ("emul_pack2", "emul_pack3"):      # the single-pass and the 32-byte-chunk / local-header formulations
            b = run_pack(emul, data, fn)
            assert a[3].tolist() == b[3].tolist() and a[2].tolist() == b[2].tolist() and a[4][:3].tolist() == b[4][:3].tolist(), (fn, data[:80])
            assert np.array_equal(unpack_syms(a[0], a[1], nb), unpack_syms(b[0], b[1], nb)), (fn, data[:80])


@pytest.mark.parametrize("case", [c for c in CASES if (c["c"] >> 1) & 1 and "Ns" not in c], ids=lambda c: c["name"])
def test_emul_compact_records_match_golden(emul, case):
    """compact 8-byte records (compact_build.cu): interior positions through pg_interior_visit_c -> pg_crec_pack -> the
    expansion K3s-c applies; the table must equal the reference's, and the 2-bit <-> base-5 conversions and the
    hash_kind-1 placement hash must agree for every record"""
    data = case["input_latin1"].encode("latin-1")
    pk2, amb, hdr, so, counts = run_pack(emul, data)
    emul.emul_compact_bad.restype = ctypes.c_int64
    emul.emul_set_compact(1)
    try:
        (ks, vs, cs), rk = run_dbg(emul, pk2, amb, so, case["k"], 2)
        assert emul.emul_compact_bad() == 0
    finally:
        emul.emul_set_compact(0)
    assert [[int(a), int(b), int(c)] for a, b, c in zip(ks, vs, cs)] == case["dbg"]
    assert rk.tolist() == case["rdbg"]


@pytest.mark.parametrize("k,form", [(4, 1), (12, 1), (21, 1), (26, 1), (27, 1), (17, 2), (21, 2), (26, 2), (27, 2)])
def test_emul_compact_records_big(emul, k, form):
    """1 Mbp x 4 with every k parity (even k: palindromes take the fold-and-count-twice bit); form 2 = the compile-time-k
    extraction (pg_interior_visit_ck: funnel shifts of three digit words, no rolling state)"""
    data = survey_4x1m()[:600_000]
    data = data[:data.rfind(b"\n") + 1]
    pk2, amb, hdr, so, counts = run_pack(emul, data)
    emul.emul_compact_bad.restype = ctypes.c_int64
    emul.emul_set_compact(form)
    try:
        (ks, vs, cs), rk = run_dbg(emul, pk2, amb, so, k, 2)
        assert emul.emul_compact_bad() == 0
    finally:
        emul.emul_set_compact(0)
    ref = oracle.run(data, k, stages=2)
    assert np.array_equal(ks, ref["dbg"][0]) and np.array_equal(vs, ref["dbg"][1]) and np.array_equal(cs, ref["dbg"][2])
    assert np.array_equal(rk, ref["rdbg"])


def test_emul_compact_records_random_inputs(emul):
    """seeded random multi-record inputs (N runs, lowercase, IUPAC, records shorter than k, poly-A, palindromic repeats)
    through the compact-record logic, rolling and compile-time-k forms, against the oracle"""
    rng = np.random.default_rng(77)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    emul.emul_compact_bad.restype = ctypes.c_int64
    for it in range(24):
        k = int(rng.choice([17, 20, 21, 26, 27, 11, 5]))
        recs = []
        for r in range(int(rng.integers(1, 6))):
            n = int(rng.choice([0, k - 1, k, k + 2, int(rng.integers(200, 4000))]))
            s = bytearray(acgt[rng.integers(0, 4, n)].tobytes())
            if n > 300 and rng.random() < 0.5:
                a = int(rng.integers(0, n - 100)); s[a:a + int(rng.integers(1, 60))] = b"N" * len(s[a:a + int(rng.integers(1, 60))])
            if n > 300 and rng.random() < 0.4:
                a = int(rng.integers(0, n - 100)); s[a:a + 50] = bytes(s[a:a + 50]).lower()
            if n > 300 and rng.random() < 0.3:
                a = int(rng.integers(0, n - 100)); s[a] = ord("R")
            if n > 300 and rng.random() < 0.4:
                a = int(rng.integers(0, n - 120)); s[a:a + 90] = b"A" * 90
            if n > 300 and rng.random() < 0.4:
                a = int(rng.integers(0, n - 120)); s[a:a + 64] = b"ACGT" * 16        # palindromic at every even k
            recs.append(b">r%d\n" % r + bytes(s) + b"\n")
        data = b"".join(recs)
        ref = oracle.run(data, k, stages=1)
        if ref["ub_count"]:
            continue
        pk2, amb, hdr, so, counts = run_pack(emul, data, "emul_pack3")
        for form in (1, 2):
            emul.emul_set_compact(form)
            try:
                (ks, vs, cs), _ = run_dbg(emul, pk2, amb, so, k, 2)
                assert emul.emul_compact_bad() == 0
            finally:
                emul.emul_set_compact(0)
            assert np.array_equal(ks, ref["dbg"][0]) and np.array_equal(vs, ref["dbg"][1]) and np.array_equal(cs, ref["dbg"][2]), (it, k, form)
