"""FASTQ input on the CPU: format detection, the FASTQ rule for multi-GPU cut points (plain and over BGZF members), and
the FASTQ pack's per-chunk line-role logic (pangenome_b200/csrc/fastq_chunk.cuh, built for the host through
tests/fastq_emul.cu) against a Python parse at random tile boundaries.  No GPU needed."""
import ctypes
import gzip
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from pangenome_b200 import seqfile, shard, stages, synth

_SO = os.path.join(ROOT, "tests", "_fastq_emul.so")


def random_fastq(rng, n_rec, crlf=False, max_len=40, trailing_blank=0):
    """Valid four-line FASTQ: empty sequences, quality lines starting with '@' or '+', N and lower-case bases."""
    eol = b"\r\n" if crlf else b"\n"
    out = []
    for r in range(n_rec):
        n = int(rng.integers(0, max_len + 1)) if rng.random() < 0.9 else 0
        seq = bytes(rng.choice(list(b"ACGTNacgt"), n, p=[.22, .22, .22, .22, .04, .02, .02, .02, .02]).astype(np.uint8))
        qual = bytearray(rng.integers(33, 75, n).astype(np.uint8))
        if n and rng.random() < 0.3:
            qual[0] = ord("@") if rng.random() < 0.6 else ord("+")
        sep = b"+" if rng.random() < 0.7 else b"+r%d" % r
        # with CRLF the '\r' is the last byte of every line: a base of the sequence line, so the quality line has one too
        out.append(b"@r%d len=%d" % (r, n) + eol + seq + eol + sep + eol + bytes(qual) + eol)
    return b"".join(out) + b"\n" * trailing_blank


def parse_starts(data):
    """Record starts of a valid FASTQ by parsing it four lines at a time (blank trailing lines are no records)."""
    starts, pos, line = [], 0, 0
    while pos < len(data):
        nl = data.find(b"\n", pos)
        end = len(data) if nl < 0 else nl + 1
        if line % 4 == 0 and data[pos:end].strip(b"\n"):
            starts.append(pos)
        pos, line = end, line + 1
    return starts


def test_detect():
    assert seqfile.detect(b"@r1\nACGT\n+\nIIII\n") == "fastq"
    assert seqfile.detect(b"@r\nAC\n+\n>>\n@r2\nAC\n+\nII\n") == "fastq"       # a '>' quality line in the first 40 bytes
    assert seqfile.detect(b">g1\nACGT\n") == "fasta"
    assert seqfile.detect(b"junk\n>g1\nACGT\n") == "fasta"
    assert seqfile.detect(b"junk\n@r\nAC\n") == "fastq"
    assert seqfile.detect(b"ACGT\n") is None
    assert seqfile.detect(b"") is None


def test_seq_chk_reads_the_decompressed_head(tmp_path):
    fq = b"@r\nAC\n+\n>>\n" * 4
    (tmp_path / "a.fq").write_bytes(fq)
    (tmp_path / "a.fq.gz").write_bytes(gzip.compress(fq))
    (tmp_path / "a.fa").write_bytes(b">g\nACGT\n")
    assert stages.seq_chk(str(tmp_path / "a.fq")) == "fastq"
    assert stages.seq_chk(str(tmp_path / "a.fq.gz")) == "fastq"
    assert stages.seq_chk(str(tmp_path / "a.fa")) == "fasta"


@pytest.mark.parametrize("crlf", [False, True])
def test_fastq_cut_rule_against_a_parse(crlf):
    """Every nominal offset, so the offsets land on every line role: the first record start at or after it."""
    rng = np.random.default_rng(5 + crlf)
    for trial in range(12):
        data = random_fastq(rng, int(rng.integers(1, 40)), crlf=crlf, trailing_blank=int(rng.integers(0, 3)))
        starts = parse_starts(data)
        for nominal in range(len(data) + 1):
            j = next((s for s in starts if s >= nominal), len(data))
            assert shard._first_fastq_start(data, len(data), nominal) == j, (trial, nominal)
        for world in (1, 2, 3, 5, 8):
            assert shard.cut_points(data, world, "fastq") == shard.cut_points_from_starts(starts, len(data), world)


def test_fastq_cut_rule_quality_line_at_the_nominal_offset():
    data = b"@a\nACGT\n+\n@III\n@b\nACGT\n+\n+III\n@c\nACGT\n+\nIIII\n"
    q = data.index(b"@III")
    assert shard._first_fastq_start(data, len(data), q) == data.index(b"@b")
    assert shard._first_fastq_start(data, len(data), data.index(b"+III")) == data.index(b"@c")


def test_fastq_cut_rule_over_members():
    """member_rank_range over members of many sizes gives the cuts and bytes of cut_points on the whole stream."""
    rng = np.random.default_rng(9)
    for trial in range(20):
        data = random_fastq(rng, int(rng.integers(1, 60)), crlf=trial % 3 == 0, trailing_blank=trial % 2)
        block = int(rng.integers(1, 60))
        out_off = np.array(list(range(0, len(data), block)) + [len(data), len(data)], dtype=np.int64)   # + an empty EOF member
        for world in (2, 3, 4, 7):
            cuts = shard.cut_points(data, world, "fastq")
            for rank in range(world):
                got, (a, b), size = shard.member_rank_range(out_off, world, rank,
                                                            lambda i0, i1: data[out_off[i0]:out_off[i1]], "fastq")
                assert (a, b, size) == (cuts[rank], cuts[rank + 1], len(data)) and got == data[a:b], (trial, world, rank)


def test_plain_rank_range_fastq(tmp_path):
    rng = np.random.default_rng(3)
    data = random_fastq(rng, 50)
    p = tmp_path / "r.fq"
    p.write_bytes(data)
    for world in (2, 3):
        cuts = shard.cut_points(data, world, "fastq")
        for rank in range(world):
            got, (a, b), size = shard.read_rank_range(str(p), world, rank)
            assert (a, b) == (cuts[rank], cuts[rank + 1]) and got == data[a:b] and size == len(data)
            assert not got or got[:1] == b"@"


# ---- the pack's line-role logic on the host ------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emul():
    src = os.path.join(ROOT, "tests", "fastq_emul.cu")
    deps = [src] + [os.path.join(ROOT, "pangenome_b200", "csrc", f) for f in ("fastq_chunk.cuh", "fasta_chunk.cuh", "common.cuh")]
    if not os.path.isfile(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps):
        tmp = "%s.%d.so" % (_SO[:-3], os.getpid())
        subprocess.check_call(["nvcc", "-O2", "-std=c++17", "--shared", "-Xcompiler", "-fPIC", "-o", tmp, src])
        os.replace(tmp, _SO)
    L = ctypes.CDLL(_SO)
    L.emul_fq_pack.restype = ctypes.c_int64
    return L


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def model(data):
    """Python parse: symbols of the sequence lines (digit A0 G1 C2 T3, N/n 0, other 1; | ambiguity << 2), and per group
    of four lines the starts of lines 0, 2, 3 and the bases before it."""
    starts = [0] + [i + 1 for i, b in enumerate(data) if b == 10 and i + 1 < len(data)]
    syms, seq_off = [], []
    dig = {ord(c): d for c, d in zip("AGCTagct", [0, 1, 2, 3, 0, 1, 2, 3])}
    for li, s in enumerate(starts):
        if li % 4 == 0:
            seq_off.append(len(syms))
        if li % 4 == 1:
            end = starts[li + 1] - 1 if li + 1 < len(starts) else len(data) - 1     # the line's last byte ends it
            for b in data[s:end]:
                syms.append(dig[b] if b in dig else ((0 if b in b"Nn" else 1) | 4))
    return np.array(syms, np.uint8), starts[0::4], seq_off + [len(syms)], starts[2::4], starts[3::4], len(starts)


@pytest.mark.parametrize("crlf", [False, True])
def test_emulated_pack_at_random_tile_boundaries(emul, crlf):
    rng = np.random.default_rng(11 + crlf)
    for trial in range(25):
        data = random_fastq(rng, int(rng.integers(1, 80)), crlf=crlf, max_len=int(rng.choice([5, 40, 300])),
                            trailing_blank=int(rng.integers(0, 3)))
        if trial % 5 == 4:
            data = data[:int(rng.integers(1, len(data)))]         # a cut file: the line logic must still hold
        n = len(data)
        tile = 32 * int(rng.integers(1, 12))
        buf = np.frombuffer(data, np.uint8).copy()
        cap = data.count(b"\n") + 2
        sym = np.zeros(n + 1, np.uint8)
        hdr, so, sep, qual = (np.full(cap + 1, -1, np.int64) for _ in range(4))
        counts = np.zeros(4, np.int64)
        assert emul.emul_fq_pack(_p(buf), ctypes.c_int64(n), ctypes.c_int64(tile), _p(sym), _p(hdr), _p(so), _p(sep), _p(qual),
                                 ctypes.c_int64(cap), _p(counts)) == 0, "tile aggregates disagree with the second pass"
        m_sym, m_hdr, m_so, m_sep, m_qual, n_lines = model(data)
        n_rec, n_bases = int(counts[0]), int(counts[1])
        assert n_rec == len(m_hdr) and n_bases == len(m_sym) and int(counts[2]) == n_lines, trial
        assert np.array_equal(sym[:n_bases], m_sym), trial
        assert list(hdr[:n_rec]) == m_hdr and list(so[:n_rec + 1]) == m_so, trial
        assert list(sep[:len(m_sep)]) == m_sep and list(qual[:len(m_qual)]) == m_qual, trial
        assert int(counts[3]) == max((i + 1 for i, b in enumerate(data) if b != 10), default=0)


def test_fastq_to_fasta_is_the_reads_fasta():
    fq = synth.reads(synth.pangenome(2, 3000), 20, length=150)
    fa = synth.fastq_to_fasta(fq)
    assert fa.count(b">") == 20 and len(fa.split(b"\n")[1]) == 150
    assert synth.fastq_to_fasta(fq + b"\n\n") == fa
