"""BGZF / gzip input on the GPU: pg_bgzf_inflate against zlib, its error reports on damaged members, and the whole
pipeline on compressed inputs against the same inputs uncompressed (CLI rows, side files and banners; config 2 table
checksum; chunked build; ``-d``; the hash-partitioned build with several ranks on one device)."""
import datetime
import gzip
import io
import os
import socket
import struct
import zlib

import numpy as np
import pytest

from conftest import load_small_cases
from pangenome_b200 import synth

pytestmark = pytest.mark.gpu
CASES = load_small_cases()
STRATEGIES = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED]


@pytest.fixture(scope="module")
def sf():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pangenome_b200 import seqfile
    return seqfile


def _inflate(sf, gz):
    """the whole BGZF image inflated on the GPU, as host bytes"""
    buf = np.frombuffer(gz, dtype=np.uint8)
    member_off, out_off = sf.bgzf_index(buf)
    return sf.inflate_members(buf, member_off, out_off, 0, len(member_off) - 1).cpu().numpy().tobytes()


def test_inflate_matches_zlib_matrix(sf):
    """levels 0-9 x the five zlib strategies (subsampled) on pangenome text, the golden inputs, random bytes (stored
    blocks), a poly-A (overlapping distance-1 copies) and blocks of 0, 1, 65280 bytes; all in ONE file, one launch"""
    rng = np.random.default_rng(3)
    inputs = [synth.pangenome(3, 60000, seed=3), "".join(c["input_latin1"] for c in CASES).encode("latin-1"),
              rng.integers(0, 256, 150000, dtype=np.uint8).tobytes(), b"A" * 200000, b"", b"G",
              synth.pangenome(2, 40000, seed=4)[:65280]]
    parts, want = [], []
    for i, data in enumerate(inputs):
        for level in range(10):
            for s, strategy in enumerate(STRATEGIES):
                if (level + s + i) % 3:
                    continue
                block = 65280 if (level + i) % 2 else 7919
                parts.append(synth.bgzf_bytes(data, block=block, level=level, strategy=strategy))
                want.append(data)
    assert _inflate(sf, b"".join(parts)) == b"".join(want)


def test_inflate_one_member_file(sf):
    data = b">one\nACGTNacgtn\nRYKM\n"
    assert _inflate(sf, synth.bgzf_member(data)) == data          # no EOF member either
    assert _inflate(sf, synth.BGZF_EOF) == b""


def test_inflate_large_file(sf):
    """>= 200 MB inflated in one launch: >= 3000 members, several per SM"""
    import torch
    data = synth.pangenome(40, 5_000_000, seed=8)
    gz = synth.bgzf_bytes(data, level=1)
    buf = np.frombuffer(gz, dtype=np.uint8)
    member_off, out_off = sf.bgzf_index(buf)
    assert len(data) >= 200_000_000 and len(member_off) - 1 >= 3000
    d = sf.inflate_members(buf, member_off, out_off, 0, len(member_off) - 1)
    assert torch.equal(d, torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).cuda())


def _member_starts(gz):
    buf = np.frombuffer(gz, dtype=np.uint8)
    from pangenome_b200 import seqfile
    return seqfile.bgzf_index(buf)[0]


def test_damaged_members_raise_naming_the_member(sf, tmp_path):
    from pangenome_b200 import _lib, stages
    data = synth.pangenome(2, 30000, seed=6)
    gz = synth.bgzf_bytes(data, block=4000)
    starts = _member_starts(gz)
    m = 5
    a, b = int(starts[m]), int(starts[m + 1])
    bad_crc = bytearray(gz)
    bad_crc[b - 8] ^= 0x10
    bad_isize = bytearray(gz)
    bad_isize[b - 4:b] = struct.pack("<I", 3999)
    bad_data = bytearray(gz)
    bad_data[a + 18 + (b - a - 26) // 2] ^= 0x04
    for bad, what in ((bad_crc, "CRC-32 mismatch"), (bad_isize, None), (bad_data, None)):
        with pytest.raises(_lib.PgError, match="BGZF member %d at byte %d" % (m, a)) as e:
            _inflate(sf, bytes(bad))
        if what:
            assert what in str(e.value)
        p = tmp_path / "bad.fa.gz"
        p.write_bytes(bytes(bad))
        with pytest.raises(_lib.PgError, match="member %d at byte %d" % (m, a)):      # nothing is built on it
            stages.seq2rdbg(str(p), 27, 5, 2 ** 63, brkpt="", chunk=2 ** 33, rc=True)


# ---------------------------------------------------------------------------------------------------------------------
# the pipeline on compressed inputs

def _variants(data):
    """the input as written by bgzip (one member), as 7-byte BGZF members, and by gzip"""
    return {"bgzf1": synth.bgzf_bytes(data), "bgzf7": synth.bgzf_bytes(data, block=7), "gzip": gzip.compress(data)}


def _cli(path, case, extra=()):
    from pangenome_b200 import cli
    out = io.StringIO()
    args = ["prog", "-i", path, "-k", str(case["k"]), "-c", str(case["c"])]
    if "Ns" in case:
        args += ["-n", str(int(case["Ns"]))]
    cli.entry_point(args + list(extra), out=out)
    lines = out.getvalue().split("\n")
    rows = [l for l in lines if l and not l.startswith("#")]
    banners = [l if not l.startswith("# finished in") else "# finished" for l in lines if l.startswith("# ")]

    def side(ext):
        p = path + ext
        return open(p).read() if os.path.isfile(p) else None
    return rows, banners, side("_rdbg_weight.xyz"), side("_rdbg_weight.xyz.mcl")


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_cli_on_compressed_golden_inputs(sf, case, tmp_path):
    data = case["input_latin1"].encode("latin-1")
    plain = tmp_path / "in.fa"
    plain.write_bytes(data)
    want = _cli(str(plain), case)
    assert want[0] == ["%s\t%d\t%d\t%s\t%d" % tuple(r) for r in case["rows"]]
    assert want[2].split("\n")[:-1] == case["xyz"]
    for name, blob in _variants(data).items():
        p = tmp_path / ("in_%s.fa.gz" % name)
        p.write_bytes(blob)
        got = _cli(str(p), case)
        assert got == want, name
        assert os.path.isfile(str(p) + "_db.npz")       # side files keep the input's name as given


def test_cfg2_bgzf_checksum(sf, tmp_path):
    """config 2 (10 x 5 Mbp) as BGZF: the same dBG checksum as the plain file and as the oracle's facts"""
    import json
    from conftest import GOLDEN
    from pangenome_b200 import stages
    facts = json.load(open(os.path.join(GOLDEN, "cfg2_oracle_facts.json")))
    data = synth.pangenome(10, 5_000_000)
    plain, gz = tmp_path / "cfg2.fa", tmp_path / "cfg2.fa.gz"
    plain.write_bytes(data)
    gz.write_bytes(synth.bgzf_bytes(data))
    sums = [list(stages.seq2rdbg(str(p), 27, 5, 2 ** 63, brkpt="", chunk=2 ** 33, rc=True).table.checksum()) for p in (plain, gz)]
    assert sums[0] == sums[1] == facts["dbg_checksum"]


def test_chunked_build_and_db_reload_on_bgzf(sf, tmp_path):
    """the chunked build (checkpoints every 2^21 bases: offsets in the decompressed stream) and -d from a _db.npz give
    the same tables and rows on the BGZF file as on the plain one"""
    from pangenome_b200 import stages
    data = synth.pangenome(4, 500_000, seed=12)
    plain, gz = tmp_path / "p.fa", tmp_path / "p.fa.gz"
    plain.write_bytes(data)
    gz.write_bytes(synth.bgzf_bytes(data, block=30011))
    res = []
    for p in (plain, gz):
        h = stages.seq2rdbg(str(p), 27, 5, 2 ** 63, brkpt="", chunk=2 ** 21, rc=True)
        ck = np.load(str(p) + "_db_brkpt.npz")
        res.append((list(h.table.checksum()), int(ck["parameters"][5])))
    assert res[0] == res[1]
    case = {"k": 27, "c": 2}
    rows = []
    for p in (plain, gz):
        _cli(str(p), case, ["--no-mcl-file"])            # writes <input>_db.npz
        os.rename(str(p) + "_db.npz", str(p) + ".db.npz")
        rows.append(_cli(str(p), case, ["-d", str(p) + ".db.npz", "--no-mcl-file"])[0])
    assert rows[0] == rows[1] and rows[0]


# ---------------------------------------------------------------------------------------------------------------------
# several ranks on one device (gloo), as tests/test_gpu_multi_one_device.py: every rank's byte range of the BGZF and
# gzip files equals that of the plain file; where the world size allows the build, so does the merged table

def _rank_main(rank, world, port, paths):
    import torch
    import torch.distributed as dist
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=600))
    try:
        from pangenome_b200 import multigpu, shard, stages
        ranges = [shard.read_rank_range(p, world, rank) for p in paths]
        assert all(r[1:] == ranges[0][1:] and bytes(r[0]) == bytes(ranges[0][0]) for r in ranges), [r[1:] for r in ranges]
        merged = []
        for p in (paths if world & (world - 1) == 0 else ()):       # the hash-partitioned build takes 2, 4 or 8 ranks
            h = stages.seq2rdbg(p, 21, 5, 2 ** 63, brkpt="", chunk=2 ** 33, rc=True)
            merged.append(multigpu.gather_export(h.table, world, rank))
        if rank == 0:
            for m in merged[1:]:
                assert all(np.array_equal(x, y) for x, y in zip(m, merged[0]))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3, 4])
def test_multi_rank_bgzf_one_device(sf, world, tmp_path):
    import torch.multiprocessing as mp
    from test_gpu_multi_one_device import _compute_mode_default, _mixed_input
    if not _compute_mode_default():
        pytest.skip("device 0 is not in the Default compute mode: no second process can use it")
    data = _mixed_input(world)
    paths = [tmp_path / "m.fa", tmp_path / "m1.fa.gz", tmp_path / "m7.fa.gz", tmp_path / "mz.fa.gz"]
    paths[0].write_bytes(data)
    paths[1].write_bytes(synth.bgzf_bytes(data, block=1000))
    paths[2].write_bytes(synth.bgzf_bytes(data, block=7))
    paths[3].write_bytes(gzip.compress(data))
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_rank_main, args=(world, port, [str(p) for p in paths]), nprocs=world, join=True)
