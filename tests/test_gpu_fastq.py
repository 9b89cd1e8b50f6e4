"""FASTQ input on the GPU: the FASTQ pack (pg_fastq_scan_pack) against K1 on the FASTA equivalent, and the whole
pipeline on FASTQ against the same records as FASTA - golden cases, config 2, a short-read set, compressed, several
ranks on one device - plus the malformed-input reports."""
import datetime
import gzip
import io
import json
import os
import socket

import numpy as np
import pytest

from conftest import GOLDEN, load_small_cases
from pangenome_b200 import synth

pytestmark = pytest.mark.gpu
CASES = load_small_cases()


@pytest.fixture(scope="module")
def eng():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pangenome_b200 import engine
    return engine


def random_fastq(rng, n_rec, max_len=300, crlf=False, trailing_blank=0):
    """Valid FASTQ: random lengths (empty ones too), N / lower-case / other bytes, quality lines starting with '@' or '+'."""
    eol = b"\r\n" if crlf else b"\n"
    recs = []
    for r in range(n_rec):
        n = int(rng.integers(0, max_len + 1)) if rng.random() < 0.95 else 0
        seq = bytes(rng.choice(list(b"ACGTNacgtRY"), n).astype(np.uint8))
        qual = bytearray(rng.integers(33, 75, n).astype(np.uint8))
        if n and rng.random() < 0.3:
            qual[0] = ord("@") if rng.random() < 0.5 else ord("+")
        recs.append(b"@read%d extra" % r + eol + seq + eol + b"+" + eol + bytes(qual) + eol)
    return b"".join(recs) + b"\n" * trailing_blank


def fastq_to_fasta(fq):
    return synth.fastq_to_fasta(fq)


def _unpack(p, n):
    i = np.arange(n)
    pk2, amb = p.pk2.cpu().numpy().view(np.uint32), p.amb.cpu().numpy().view(np.uint32)
    return ((pk2[i >> 4] >> (2 * (i & 15)).astype(np.uint32)) & 3), ((amb[i >> 5] >> (i & 31).astype(np.uint32)) & 1)


def _pack_pair(eng, fq):
    a = eng.PackedSeqs(eng.to_device_bytes(fq), fmt="fastq")
    b = eng.PackedSeqs(eng.to_device_bytes(fastq_to_fasta(fq)))
    return a, b


# ---------------------------------------------------------------------------------------------------------------------
# 1. the pack against K1 on fasta(F)

@pytest.mark.parametrize("n_rec,crlf,blank", [(1, False, 0), (37, True, 2), (500, False, 1), (5000, False, 0), (20000, True, 3)])
def test_pack_parity_with_k1(eng, n_rec, crlf, blank):
    rng = np.random.default_rng(n_rec)
    fq = random_fastq(rng, n_rec, max_len=300 if n_rec < 10000 else 60, crlf=crlf, trailing_blank=blank)
    a, b = _pack_pair(eng, fq)
    assert (a.n_rec, a.n_bases) == (b.n_rec, b.n_bases) == (n_rec, b.n_bases)
    assert np.array_equal(a.seq_off, b.seq_off)
    assert all(fq[h:h + 1] == b"@" and (h == 0 or fq[h - 1:h] == b"\n") for h in a.hdr_off.tolist())
    assert a.hdr_off.tolist() == [i for i in range(len(fq)) if fq[i:i + 5] == b"@read" and (i == 0 or fq[i - 1] == 10)]
    n = int(a.n_bases)
    for x, y in zip(_unpack(a, n), _unpack(b, n)):
        assert np.array_equal(x, y)
    assert a.n_newlines == fq.count(b"\n")


def test_pack_empty_and_blank(eng):
    for data in (b"", b"\n", b"\n\n\n\n\n"):
        p = eng.PackedSeqs(eng.to_device_bytes(data), fmt="fastq")
        assert (p.n_rec, p.n_bases) == (0, 0)


def test_pack_index_growth(eng):
    """more records than the first record-index capacity (4096): the pack runs again with room for all of them"""
    rng = np.random.default_rng(2)
    fq = random_fastq(rng, 9000, max_len=20)
    a, b = _pack_pair(eng, fq)
    assert a.n_rec == 9000 and np.array_equal(a.seq_off, b.seq_off)


# ---------------------------------------------------------------------------------------------------------------------
# 2. golden cases rewritten as FASTQ

def golden_as_fastq(data):
    """(FASTQ bytes, None) holding each record's base bytes as one sequence line, or (None, reason) for the inputs the
    rewrite cannot express."""
    if b"\n" not in data:
        return None, "no line end: the FASTA reader yields no line at all"
    if data[:1] != b">":
        return None, "bytes before the first header belong to no record"
    lines, pos = [], 0
    while pos < len(data):
        nl = data.find(b"\n", pos)
        end = len(data) if nl < 0 else nl + 1
        lines.append(data[pos:end])
        pos = end
    recs = []
    for l in lines:
        if l[:1] == b">":
            if not l.endswith(b"\n"):
                return None, "a header line without a line end: its last byte is dropped, FASTQ keeps it"
            recs.append([l, b""])
        else:
            recs[-1][1] += l[:-1]             # the last byte of every line is dropped (Q8)
    return b"".join(b"@" + h[1:] + s + b"\n+\n" + b"I" * len(s) + b"\n" for h, s in recs), None


def _cli(path, k, c, ns=None, extra=()):
    from pangenome_b200 import cli
    out = io.StringIO()
    args = ["prog", "-i", path, "-k", str(k), "-c", str(c)] + (["-n", str(int(ns))] if ns is not None else [])
    cli.entry_point(args + list(extra), out=out)
    lines = out.getvalue().split("\n")
    rows = [l for l in lines if l and not l.startswith("#")]
    banners = [l if not l.startswith("# finished in") else "# finished" for l in lines if l.startswith("# ")]

    def side(ext):
        p = path + ext
        return open(p).read() if os.path.isfile(p) else None
    db = None
    if os.path.isfile(path + "_db.npz"):
        # the content of the saved table: its parameters and its slots as a multiset (where a key sits in the image
        # depends on the order the table's export hands the entries over, which the build does not fix)
        z = np.load(path + "_db.npz")
        o = np.lexsort((z["counts"], z["values"], z["keys"]))
        db = (z["parameters"].tolist(), z["keys"][o].tobytes(), z["values"][o].tobytes(), z["counts"][o].tobytes())
    return rows, banners, side("_rdbg_weight.xyz"), side("_rdbg_weight.xyz.mcl"), db


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_cli_on_golden_cases_as_fastq(eng, case, tmp_path):
    data = case["input_latin1"].encode("latin-1")
    fq, why = golden_as_fastq(data)
    if fq is None:
        pytest.skip(why)
    fa = tmp_path / "in.fa"
    fa.write_bytes(data)
    q = tmp_path / "in.fq"
    q.write_bytes(fq)
    want = _cli(str(fa), case["k"], case["c"], case.get("Ns"))
    got = _cli(str(q), case["k"], case["c"], case.get("Ns"))
    assert got[0] == ["%s\t%d\t%d\t%s\t%d" % tuple(r) for r in case["rows"]]
    assert got[2].split("\n")[:-1] == case["xyz"]
    assert got == want
    from pangenome_b200 import stages
    h = stages.seq2rdbg(str(q), int(case["k"]), 5, case.get("Ns", 2 ** 63), brkpt="", chunk=2 ** 33, rc=int(case["c"]) >> 1 == 1)
    keys, vals, cnts = h.table.export()
    assert [[int(a), int(b), int(c)] for a, b, c in zip(keys, vals, cnts)] == case["dbg"]
    rk, _ = stages.dbg2rdbg(h).table.rdbg_export()
    assert [int(x) for x in rk] == case["rdbg"]


# ---------------------------------------------------------------------------------------------------------------------
# 3. config 2 as a 10-record FASTQ

def test_cfg2_as_fastq_checksum(eng, tmp_path):
    from pangenome_b200 import stages
    facts = json.load(open(os.path.join(GOLDEN, "cfg2_oracle_facts.json")))
    data = synth.pangenome(10, 5_000_000)
    fq = b"".join(b"@" + r.split(b"\n", 1)[0] + b"\n" + r.split(b"\n", 1)[1].replace(b"\n", b"") + b"\n+\n" + b"F" * 5_000_000 + b"\n"
                  for r in data[1:].split(b"\n>"))
    p = tmp_path / "cfg2.fq"
    p.write_bytes(fq)
    h = stages.seq2rdbg(str(p), 27, 5, 2 ** 63, brkpt="", chunk=2 ** 33, rc=True)
    assert h.n_rec == 10 and list(h.table.checksum()) == facts["dbg_checksum"]


# ---------------------------------------------------------------------------------------------------------------------
# 4./5. a short-read set, plain and compressed, against its FASTA equivalent

@pytest.fixture(scope="module")
def reads_fq():
    return synth.reads(synth.pangenome(10, 200_000, seed=5), 100_000, length=150, n_rate=0.0005)


def _write(tmp_path, fq, kinds):
    """the read set as FASTQ, as its FASTA equivalent, as BGZF and as gzip FASTQ; each test writes its own copies, so no
    side file of another test (an existing .xyz.mcl wins over clustering) is in the way"""
    blobs = {"fq": fq, "fa": synth.fastq_to_fasta(fq), "bgzf": synth.bgzf_bytes(fq, block=30011), "gzip": gzip.compress(fq)}
    names = {"fq": "r.fq", "fa": "r.fa", "bgzf": "r.fq.gz", "gzip": "rz.fq.gz"}
    out = {}
    for k in kinds:
        (tmp_path / names[k]).write_bytes(blobs[k])
        out[k] = str(tmp_path / names[k])
    return out


def test_reads_against_fasta(eng, reads_fq, tmp_path):
    from pangenome_b200 import stages
    f = _write(tmp_path, reads_fq, ("fq", "fa"))
    hs = {k: stages.seq2rdbg(f[k], 27, 5, 2 ** 63, brkpt="", chunk=2 ** 33, rc=True) for k in ("fq", "fa")}
    assert hs["fq"].n_rec == hs["fa"].n_rec == 100_000
    assert list(hs["fq"].table.checksum()) == list(hs["fa"].table.checksum())
    # the record form the build ended on, so a change is visible: this 150 bp read set ends on 16-byte records, FASTQ and
    # FASTA alike (DESIGN.md 6c item 6: compact records for inputs of short records)
    assert hs["fq"].builder.compact is False and hs["fa"].builder.compact is False
    out = {k: _cli(f[k], 27, 2, extra=["--cluster", "mcl"]) for k in ("fq", "fa")}
    assert out["fq"] == out["fa"] and out["fq"][0] and out["fq"][3] and out["fq"][4]


def test_reads_compressed(eng, reads_fq, tmp_path):
    f = _write(tmp_path, reads_fq, ("fq", "bgzf", "gzip"))
    want = _cli(f["fq"], 27, 2, extra=["--min-edge-weight", "2"])
    for k in ("bgzf", "gzip"):
        assert _cli(f[k], 27, 2, extra=["--min-edge-weight", "2"]) == want, k


def test_reads_db_reload_and_prefix(eng, reads_fq, tmp_path):
    """-d from the _db.npz written on the FASTQ, and -n, give what they give on the FASTA"""
    f = _write(tmp_path, reads_fq, ("fq", "fa"))
    res = []
    for k in ("fq", "fa"):
        _cli(f[k], 27, 2, extra=["--no-mcl-file"])
        db = str(tmp_path / (k + ".db.npz"))
        os.replace(f[k] + "_db.npz", db)
        res.append((_cli(f[k], 27, 2, extra=["-d", db, "--no-mcl-file", "--no-dump-db"])[0],
                    _cli(f[k], 21, 3, ns=2_000_000, extra=["--no-mcl-file", "--no-dump-db"])[0]))
    assert res[0] == res[1] and res[0][0] and res[0][1]


# ---------------------------------------------------------------------------------------------------------------------
# 6. several ranks on one device (gloo)

def _rank_main(rank, world, port, paths, n_rec, ref_rows, ref_xyz):
    import torch
    import torch.distributed as dist
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=600))
    try:
        from pangenome_b200 import engine, shard, stages
        ranges = [shard.read_rank_range(p, world, rank) for p in paths]
        assert all(r[1:] == ranges[0][1:] and bytes(r[0]) == bytes(ranges[0][0]) for r in ranges), [r[1:] for r in ranges]
        data = bytes(ranges[0][0])
        p = engine.PackedSeqs(engine.to_device_bytes(data), fmt="fastq")        # every rank's range is whole records
        counts = [None] * world
        dist.all_gather_object(counts, p.n_rec)
        assert sum(counts) == n_rec, counts
        if world & (world - 1) == 0:            # the hash-partitioned build takes 2, 4 or 8 ranks
            for path in paths:
                out = io.StringIO()
                h = stages.seq2rdbg(path, 27, 5, 2 ** 63, brkpt="", chunk=2 ** 33, rc=True)
                stages.seq2graph(path, kmer=27, Ns=2 ** 63, rdbg_dict=stages.dbg2rdbg(h), rc=True, out=out, write_mcl=False)
                if rank == 0:
                    assert [l for l in out.getvalue().split("\n") if l] == ref_rows, path
                    assert open(path + "_rdbg_weight.xyz").read() == ref_xyz, path
                dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_multi_rank_fastq_one_device(eng, world, tmp_path):
    import torch.multiprocessing as mp
    from pangenome_b200 import shard
    from test_gpu_multi_one_device import _compute_mode_default
    if not _compute_mode_default():
        pytest.skip("device 0 is not in the Default compute mode: no second process can use it")
    fq = synth.reads(synth.pangenome(4, 50_000, seed=6), 3000, length=150)
    # rank 1's nominal cut lands exactly on a quality line that starts with '@' (blank lines at the end set the size)
    q = fq.find(b"\n+\n", len(fq) // world) + 3
    fq = fq[:q] + b"@" + fq[q + 1:] + b"\n" * (world * q - len(fq))
    assert len(fq) // world == q and fq[q:q + 1] == b"@"
    assert shard.cut_points(fq, world, "fastq")[1] == fq.index(b"\n@SIM", q) + 1
    paths = [tmp_path / "m.fq", tmp_path / "m.fq.gz"]
    paths[0].write_bytes(fq)
    paths[1].write_bytes(synth.bgzf_bytes(fq, block=7001))
    one = _cli(str(paths[0]), 27, 3, extra=["--no-mcl-file", "--no-dump-db"])
    os.remove(str(paths[0]) + "_rdbg_weight.xyz")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_rank_main, args=(world, port, [str(p) for p in paths], 3000, one[0], one[2]), nprocs=world, join=True)


# ---------------------------------------------------------------------------------------------------------------------
# 7. malformed input

GOOD = b"@a\nACGT\n+\nIIII\n@b\nGGCC\n+x\nJJJJ\n@c\nTTAA\n+\nKKKK\n"


@pytest.mark.parametrize("bad,offset,kind", [
    (GOOD.replace(b"@b\n", b"Xb\n"), GOOD.index(b"@b"), "'@'"),                       # a header line without '@'
    (GOOD.replace(b"+x\n", b"-x\n"), GOOD.index(b"@b"), "'\\+'"),                     # a separator line without '+'
    (GOOD.replace(b"KKKK", b"KKK"), GOOD.index(b"@c"), "quality length"),            # quality shorter than the sequence
    (GOOD.replace(b"JJJJ", b"JJJJJ"), GOOD.index(b"@b"), "quality length"),          # ... or longer
    (GOOD[:-8], GOOD.index(b"@c"), "truncated"),                                      # a truncated last record
    (GOOD + b"@d\nAC\nGT\n+\nIIII\n", len(GOOD), "quality length|separator"),         # wrapped (multi-line) FASTQ
    (GOOD + b"\n\n@d\nAC\n+\nII\n", len(GOOD), "'@'"),                                # a blank line inside the file
    (b"@a\nACGT", 0, "truncated"),                                                     # no line end at all
])
def test_malformed_fastq(eng, tmp_path, bad, offset, kind):
    from pangenome_b200 import _lib, engine, stages
    with pytest.raises(engine.FastqError, match=kind) as e:
        engine.PackedSeqs(engine.to_device_bytes(bad), fmt="fastq")
    assert e.value.offset == offset
    p = tmp_path / "bad.fq"
    p.write_bytes(bad)
    with pytest.raises(SystemExit, match="at byte %d" % offset):
        _cli(str(p), 5, 2)
    assert sorted(os.listdir(tmp_path)) == ["bad.fq"]                 # no side file
    assert isinstance(e.value, _lib.PgError)
    with pytest.raises(SystemExit, match="at byte %d" % offset):
        stages.seq2rdbg(str(p), 5, 5, 2 ** 63, brkpt="", chunk=2 ** 33, rc=True)


def test_trailing_blank_lines_are_allowed(eng):
    for tail in (b"\n", b"\n\n\n\n\n\n"):
        a, b = _pack_pair(eng, GOOD + tail)
        assert a.n_rec == 3 and np.array_equal(a.seq_off, b.seq_off)


def test_r_is_refused_on_fastq(eng, tmp_path):
    p = tmp_path / "a.fq"
    p.write_bytes(GOOD)
    with pytest.raises(SystemExit, match="-r"):
        _cli(str(p), 3, 2, extra=["-r", str(tmp_path / "a.fq_db_brkpt.npz")])
