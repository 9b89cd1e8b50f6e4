"""CPU checks of the BGZF input path: the DEFLATE decoder core (pangenome_b200/csrc/inflate.cuh, compiled for the host by
tests/inflate_emul.cu) against zlib, its behaviour on damaged members, the member index (pg_host_bgzf_index) and the
rank cut search over members (shard.member_rank_range) against shard.cut_points.  No GPU needed."""
import ctypes
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from conftest import ROOT, load_small_cases
from pangenome_b200 import shard, synth

_SO = os.path.join(ROOT, "tests", "_inflate_emul.so")
STRATEGIES = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED]
CANARY = 64


@pytest.fixture(scope="module")
def emul():
    src = os.path.join(ROOT, "tests", "inflate_emul.cu")
    deps = [src, os.path.join(ROOT, "pangenome_b200", "csrc", "inflate.cuh"), os.path.join(ROOT, "include", "pgdbg.h")]
    if not os.path.isfile(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps):
        tmp = "%s.%d.so" % (_SO[:-3], os.getpid())       # private name, renamed into place: parallel workers never load half a file
        subprocess.check_call(["nvcc", "-O2", "-std=c++17", "--shared", "-Xcompiler", "-fPIC", "-o", tmp, src])
        os.replace(tmp, _SO)
    L = ctypes.CDLL(_SO)
    L.emul_crc32_segments.restype = ctypes.c_uint32
    L.emul_crc32_segments.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int]
    L.emul_inflate_raw.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]
    L.emul_bgzf_member.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64]
    return L


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _guarded(data):
    """``data`` inside a buffer with canary bytes on both sides: (buffer, view of the data)."""
    buf = np.full(len(data) + 2 * CANARY, 0xA5, dtype=np.uint8)
    buf[CANARY:CANARY + len(data)] = np.frombuffer(data, dtype=np.uint8)
    return buf


def _intact(buf, n):
    return bool((buf[:CANARY] == 0xA5).all() and (buf[CANARY + n:] == 0xA5).all())


def inflate_raw(L, comp, out_len):
    """(error, output bytes, consumed, crc) of the decoder core on raw DEFLATE ``comp`` with an exact ``out_len`` window;
    the canaries around the input copy and the output window are checked."""
    src = _guarded(comp)
    dst = np.full(out_len + 2 * CANARY, 0xA5, dtype=np.uint8)
    info = np.zeros(3, dtype=np.int64)
    err = L.emul_inflate_raw(_p(src[CANARY:]), len(comp), _p(dst[CANARY:]), out_len, _p(info))
    assert _intact(dst, out_len) and _intact(src, len(comp)) and bytes(src[CANARY:CANARY + len(comp)]) == comp
    return err, bytes(dst[CANARY:CANARY + int(info[0])]), int(info[1]), int(info[2]) & 0xFFFFFFFF


def member(L, gz, out_len):
    src = _guarded(gz)
    dst = np.full(out_len + 2 * CANARY, 0xA5, dtype=np.uint8)
    err = L.emul_bgzf_member(_p(src[CANARY:]), len(gz), _p(dst[CANARY:]), out_len)
    assert _intact(dst, out_len) and _intact(src, len(gz))
    return err, bytes(dst[CANARY:CANARY + out_len])


def _deflate(data, level, strategy):
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    return c.compress(data) + c.flush()


def _inputs():
    rng = np.random.default_rng(7)
    cases = load_small_cases()
    return {
        "pangenome": synth.pangenome(3, 40000, seed=3)[:100000],
        "golden": "".join(c["input_latin1"] for c in cases).encode("latin-1"),      # lowercase, IUPAC, CRLF, N runs
        "random": rng.integers(0, 256, 70000, dtype=np.uint8).tobytes(),          # incompressible: stored blocks
        "poly_a": b"A" * 65536,                                                     # distance-1 copies of 258 bytes
        "empty": b"",
        "one": b"G",
        "block_65280": synth.pangenome(2, 40000, seed=4)[:65280],
        "block_65536": synth.pangenome(2, 40000, seed=5)[:65536],
    }


INPUTS = _inputs()


@pytest.mark.parametrize("name", sorted(INPUTS))
def test_decoder_matches_zlib_every_level_and_strategy(emul, name):
    data = INPUTS[name]
    for level in range(10):
        for strategy in STRATEGIES:
            comp = _deflate(data, level, strategy)
            err, out, consumed, crc = inflate_raw(emul, comp, len(data))
            assert err == 0, (name, level, strategy, err)
            assert out == data and consumed == len(comp) and crc == zlib.crc32(data), (name, level, strategy)


def test_decoder_matches_zlib_on_each_golden_case(emul):
    for c in load_small_cases():
        data = c["input_latin1"].encode("latin-1")
        for level in (1, 6, 9):
            comp = _deflate(data, level, zlib.Z_DEFAULT_STRATEGY)
            err, out, consumed, crc = inflate_raw(emul, comp, len(data))
            assert (err, out, consumed, crc) == (0, data, len(comp), zlib.crc32(data)), c["name"]


def test_decoder_rejects_output_past_the_window(emul):
    data = INPUTS["pangenome"][:5000]
    for strategy in STRATEGIES:
        comp = _deflate(data, 6, strategy)
        err, _, _, _ = inflate_raw(emul, comp, len(data) - 1)
        assert err == 8                                  # PG_INF_ERR_OVERFLOW
    err, _, _, _ = inflate_raw(emul, _deflate(b"A" * 1000, 9, zlib.Z_DEFAULT_STRATEGY), 999)
    assert err == 8


def test_crc_combine_of_lane_segments(emul):
    rng = np.random.default_rng(11)
    for n in (0, 1, 31, 32, 33, 1000, 65280, 65536):
        buf = rng.integers(0, 256, max(n, 1), dtype=np.uint8)[:n].copy()
        for lanes in (1, 2, 7, 32):
            assert emul.emul_crc32_segments(_p(buf) if n else None, n, lanes) == zlib.crc32(buf.tobytes()), (n, lanes)


def _members(data, block, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    return [(synth.bgzf_member(data[i:i + block], level, strategy), data[i:i + block]) for i in range(0, len(data), block)]


def test_member_decoder_on_valid_members(emul):
    for level, strategy in ((0, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_RLE), (6, zlib.Z_DEFAULT_STRATEGY), (9, zlib.Z_FIXED)):
        for gz, raw in _members(INPUTS["pangenome"], 65280, level, strategy) + [(synth.BGZF_EOF, b"")]:
            assert member(emul, gz, len(raw)) == (0, raw)


def test_damaged_members_never_decode_silently(emul):
    """Seeded single-bit flips in the deflate data or the CRC-32 / ISIZE trailer, and truncations: every one gives an
    error code unless the damaged member still decodes to the very same bytes.  That happens when the flip lands in the
    final byte's padding bits, which no decoder reads, or turns a back-reference into another one that copies identical
    bytes (repetitive text): no output is ever accepted that differs from the original."""
    rng = np.random.default_rng(2024)
    sources = _members(INPUTS["pangenome"][:40000], 8000) + _members(INPUTS["golden"], 4000, 9, zlib.Z_FIXED) \
        + _members(INPUTS["random"][:9000], 9000, 0) + _members(INPUTS["poly_a"][:20000], 20000, 9, zlib.Z_RLE)
    n_flips = n_same = 0
    for gz, raw in sources:
        body = np.frombuffer(gz, dtype=np.uint8)
        for _ in range(300):
            pos = int(rng.integers(18, len(gz)))             # deflate data and trailer (MTIME, XFL, OS and BC are not read)
            bad = body.copy()
            bad[pos] ^= np.uint8(1 << int(rng.integers(0, 8)))
            err, out = member(emul, bad.tobytes(), len(raw))
            n_flips += 1
            if err == 0:
                assert out == raw, (pos, len(gz))
                n_same += 1
        for cut in sorted(set(int(c) for c in rng.integers(0, len(gz), 40))):
            assert member(emul, gz[:cut], len(raw))[0] != 0, cut
        assert member(emul, gz, len(raw) + 1)[0] == 9       # a window that disagrees with ISIZE
    assert n_flips >= 3000 and n_same < n_flips // 50


def test_member_decoder_error_kinds(emul):
    raw = INPUTS["pangenome"][:3000]
    gz = bytearray(synth.bgzf_member(raw))
    bad = bytearray(gz)
    bad[-8] ^= 1                                            # CRC-32
    assert member(emul, bytes(bad), len(raw))[0] == 10
    bad = bytearray(gz)
    bad[-4:] = struct.pack("<I", len(raw) + 5)              # ISIZE
    assert member(emul, bytes(bad), len(raw) + 5)[0] == 9
    bad = bytearray(gz)
    bad[3] = 0                                              # FLG without FEXTRA
    assert member(emul, bytes(bad), len(raw))[0] == 1
    stored = synth.bgzf_member(b"ACGT" * 10, level=0)
    bad = bytearray(stored)
    bad[18 + 3] ^= 0x40                                     # LEN of the stored block no longer matches NLEN
    assert member(emul, bytes(bad), 40)[0] in (2, 4)
    # a back-reference before the start of the window: fixed block, literal 'A', then length 3 distance 2
    bits = [(1, 1), (1, 2)]                                  # BFINAL, BTYPE=01 (values, widths), codes sent MSB first below

    def code(v, n):
        return [((v >> (n - 1 - i)) & 1, 1) for i in range(n)]
    bits += code(0x30 + ord("A"), 8) + code(1, 7) + code(1, 5) + code(0, 7)       # 'A', len 3 (257), dist 2, end
    acc = nb = 0
    for v, w in bits:
        acc |= v << nb
        nb += w
    comp = acc.to_bytes((nb + 7) // 8, "little")
    assert inflate_raw(emul, comp, 4)[0] == 7                # PG_INF_ERR_DISTANCE
    assert inflate_raw(emul, b"\x07", 4)[0] == 3             # BTYPE = 3


def _lib_built():
    from pangenome_b200 import _lib, build
    build.build()
    return _lib


def _index(data):
    import pangenome_b200.seqfile as seqfile
    return seqfile.bgzf_index(np.frombuffer(data, dtype=np.uint8).copy() if data else np.zeros(0, np.uint8))


def test_index_walks_members_and_concatenations():
    _lib_built()
    data = INPUTS["pangenome"]
    f1 = synth.bgzf_bytes(data, block=7000)
    mo, oo = _index(f1)
    assert len(mo) - 1 == (len(data) + 6999) // 7000 + 1 and oo[-1] == len(data) and mo[-1] == len(f1)
    assert list(oo[:-2]) == list(range(0, len(data), 7000))
    f2 = synth.bgzf_bytes(INPUTS["golden"], block=7)          # tiny members
    cat = f1 + f2                                             # the first file's EOF member sits mid-file
    mo, oo = _index(cat)
    assert oo[-1] == len(data) + len(INPUTS["golden"]) and mo[-1] == len(cat)
    assert len(mo) - 1 == (len(data) + 6999) // 7000 + 1 + (len(INPUTS["golden"]) + 6) // 7 + 1
    assert _index(synth.BGZF_EOF)[1].tolist() == [0, 0]
    # the index grows its arrays when the file has more members than its first guess
    many = synth.bgzf_bytes(INPUTS["golden"][:3000], block=1)
    assert len(_index(many)[0]) == 3002


def test_index_rejects_non_bgzf_and_damaged_files():
    _lib = _lib_built()
    import gzip
    assert _index(gzip.compress(INPUTS["golden"])) is None                  # a plain gzip file: "not BGZF"
    assert _index(INPUTS["golden"]) is None                                 # plain text
    assert _index(b"") is None
    f = synth.bgzf_bytes(INPUTS["pangenome"], block=20000)
    with pytest.raises(_lib.PgError, match="truncated"):
        _index(f[:-28 - 5])                                                 # last data member cut short
    bad = bytearray(f)
    bad[16:18] = struct.pack("<H", len(f) + 100)                            # BSIZE of member 0 past the end of the file
    with pytest.raises(_lib.PgError, match="truncated"):
        _index(bytes(bad))
    with pytest.raises(_lib.PgError, match="no BGZF member header"):
        _index(f[:-28] + gzip.compress(b">x\nACGT\n"))                      # a later member that is not BGZF
    with pytest.raises(_lib.PgError, match="no BGZF member header"):
        _index(f + b"\n")                                                   # trailing garbage


def _zlib_inflater(gz, member_off, calls):
    def inflate(i0, i1):
        calls.append((i0, i1))
        return b"".join(zlib.decompress(gz[member_off[i]:member_off[i + 1]], wbits=31) for i in range(i0, i1))
    return inflate


def _cut_cases():
    rng = np.random.default_rng(5)
    long_rec = synth.fasta_bytes([(b"long one", synth._ACGT[rng.integers(0, 4, 30000)])])
    short = synth.fasta_bytes([(b"s%d" % i, synth._ACGT[rng.integers(0, 4, int(rng.integers(1, 300)))]) for i in range(60)])
    return [(INPUTS["golden"], 7), (short + long_rec + short, 7), (short + long_rec + short, 4096), (long_rec, 1000),
            (b"no header at all\nACGT\n", 5), (INPUTS["pangenome"], 65280), (b">only\n", 7)]


def test_member_cut_search_equals_cut_points():
    """shard.member_rank_range driven by zlib: the same cuts and bytes as shard.cut_points on the decompressed stream,
    with records longer than a rank's share and 7-byte members that split headers and lines."""
    _lib_built()
    for data, block in _cut_cases():
        gz = synth.bgzf_bytes(data, block=block)
        member_off, out_off = _index(gz)
        for world in range(1, 9):
            cuts = shard.cut_points(data, world)
            for rank in range(world):
                calls = []
                got, (a, b), size = shard.member_rank_range(out_off, world, rank, _zlib_inflater(gz, member_off, calls))
                assert (a, b, size) == (cuts[rank], cuts[rank + 1], len(data)), (block, world, rank)
                assert got == data[a:b]
                # the members read are contiguous and start at the one holding nominal_r - 1
                assert all(calls[i][1] == calls[i + 1][0] for i in range(len(calls) - 1))
    assert shard.member_rank_range(np.zeros(2, np.int64), 3, 1, None) == (b"", (0, 0), 0)
