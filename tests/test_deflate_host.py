"""CPU checks of the GPU `_db.npz` writer: the chunk encoder core (pangenome_b200/csrc/deflate.cuh, compiled for the host
by tests/deflate_emul.cu) against zlib and the repo's own decoder, the placement rule of pg_oakht_place stated in numpy,
and the zip container of pangenome_b200.npz built from host-compressed members.  No GPU needed."""
import ctypes
import io
import os
import subprocess
import zipfile
import zlib

import numpy as np
import pytest

from conftest import ROOT, load_small_cases
from test_inflate_host import emul, inflate_raw  # noqa: F401  (the decoder core's harness and its fixture)
from pangenome_b200 import npz

_SO = os.path.join(ROOT, "tests", "_deflate_emul.so")
CHUNK = npz.CHUNK
CASES = {c["name"]: c for c in load_small_cases()}
SENT = np.uint64(0xFFFFFFFFFFFFFFFF)


@pytest.fixture(scope="module")
def denc():
    src = os.path.join(ROOT, "tests", "deflate_emul.cu")
    csrc = os.path.join(ROOT, "pangenome_b200", "csrc")
    deps = [src, os.path.join(csrc, "deflate.cuh"), os.path.join(csrc, "inflate.cuh"), os.path.join(ROOT, "include", "pgdbg.h")]
    if not os.path.isfile(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps):
        tmp = "%s.%d.so" % (_SO[:-3], os.getpid())
        subprocess.check_call(["nvcc", "-O2", "-std=c++17", "--shared", "-Xcompiler", "-fPIC", "-o", tmp, src])
        os.replace(tmp, _SO)
    L = ctypes.CDLL(_SO)
    L.emul_deflate.restype = ctypes.c_int64
    L.emul_deflate.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                               ctypes.c_void_p, ctypes.c_void_p]
    return L


def deflate(L, data, chunk=CHUNK):
    """(raw DEFLATE stream, chunk sizes, CRC-32) of the CPU core on ``data``."""
    src = np.frombuffer(data, dtype=np.uint8) if len(data) else np.zeros(1, dtype=np.uint8)
    n = len(data)
    nc = max(1, -(-n // chunk))
    out = np.zeros(n + 5 * nc + 64, dtype=np.uint8)
    sizes = np.zeros(nc, dtype=np.int64)
    crcs = np.zeros(nc, dtype=np.uint32)
    crc = ctypes.c_uint32()
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    tot = L.emul_deflate(P(src), n, chunk, P(out), P(sizes), P(crcs), ctypes.byref(crc))
    assert tot >= 0
    return out[:tot].tobytes(), sizes, crc.value


def _zlib_inflate(comp):
    d = zlib.decompressobj(-15)
    out = d.decompress(comp) + d.flush()
    assert d.eof and d.unused_data == b""
    return out


def check_roundtrip(denc, emul, data, chunk=CHUNK):  # noqa: F811
    comp, sizes, crc = deflate(denc, data, chunk)
    assert _zlib_inflate(comp) == data
    err, out, consumed, _ = inflate_raw(emul, comp, len(data))
    assert err == 0 and out == data and consumed == len(comp)
    assert crc == zlib.crc32(data)
    # every chunk decodes on its own from its offset (an empty final fixed block, 03 00, ends it for the repo decoder)
    offs = np.concatenate([[0], np.cumsum(sizes)])
    for i in range(len(sizes)):
        piece = comp[offs[i]:offs[i + 1]]
        want = data[i * chunk:(i + 1) * chunk]
        d = zlib.decompressobj(-15)
        assert d.decompress(piece) == want
        if i + 1 < len(sizes):
            err, out, _, _ = inflate_raw(emul, piece + b"\x03\x00", len(want))
            assert err == 0 and out == want
    return comp


def _runs_at_edges(chunk):
    cases = []
    for L in (3, 4, 258, 259, 260, 516):
        for at in (chunk - L // 2, chunk - L, chunk, chunk - 1):
            d = bytearray(b"ab" * chunk)
            d[at:at + L] = b"\x00" * L
            cases.append(bytes(d[:chunk + 600]))
    return cases


def test_roundtrip_sizes_and_edges(denc, emul):  # noqa: F811
    rng = np.random.default_rng(7)
    for n in (0, 1, CHUNK - 1, CHUNK, CHUNK + 1, 3 * CHUNK + 17):
        check_roundtrip(denc, emul, rng.integers(0, 4, n, dtype=np.uint8).tobytes())
    for d in _runs_at_edges(CHUNK):
        check_roundtrip(denc, emul, d)
    check_roundtrip(denc, emul, bytes(range(256)) * 300)
    for chunk in (1, 2, 3, 100, 65535):        # other chunk sizes, down to one byte per chunk
        check_roundtrip(denc, emul, bytes(range(256)) + b"\x00" * 700 + bytes(5), chunk)


def test_run_pieces_match_the_split_rule(denc):
    """A run of L >= 4 is one literal + matches of 3..258 at distance 1; every length in the range decodes."""
    for L in list(range(1, 300)) + [515, 516, 517, 518, 519, 774, 775, 776]:
        d = b"q" + b"z" * L + b"q"
        assert _zlib_inflate(deflate(denc, d)[0]) == d


def test_random_bytes_are_stored(denc, emul):  # noqa: F811
    data = np.random.default_rng(3).integers(0, 256, 10 * CHUNK + 99, dtype=np.uint8).tobytes()
    comp = check_roundtrip(denc, emul, data)
    assert len(comp) <= len(data) + 5 * 11      # at most 5 bytes per chunk


def test_zeros(denc, emul):  # noqa: F811
    data = bytes(11_000_000)
    comp = check_roundtrip(denc, emul, data)
    assert len(comp) < len(data) // 200


def test_deterministic(denc):
    data = np.random.default_rng(5).integers(0, 6, 500_000, dtype=np.uint8).tobytes()
    assert deflate(denc, data)[0] == deflate(denc, data)[0]


def _fnv4(keys):
    a = np.full(keys.shape, 0xcbf29ce484222325, dtype=np.uint64)
    v = keys.astype(np.uint64)
    with np.errstate(over="ignore"):
        for _ in range(4):
            a ^= v & np.uint64(0xFF)
            a *= np.uint64(0x100000001b3)
            v = v >> np.uint64(8)
    return a


def oak_rounds(keys, vals, cnts, cap, max_rounds=4096):
    """The placement rule of pg_oakht_place in numpy: the sentinel first at its first probe slot; then in round s every
    unplaced entry bids for its s-th probe slot of oakht.pointer() (j0, j0, j0+1, j0+4, ...) if no earlier round took
    it, the smallest key wins.  Returns (okeys, ovals, ocnts)."""
    keys = np.asarray(keys, dtype=np.uint64)
    j0 = _fnv4(keys).view(np.int64) % cap                   # signed hash, floor modulo
    ok = np.full(cap, SENT, dtype=np.uint64)
    ov = np.zeros(cap, dtype=np.uint16)
    oc = np.zeros(cap, dtype=np.uint8)
    live_cnt = np.maximum(np.asarray(cnts, dtype=np.uint8), 1)
    s_ = keys == SENT
    ok[j0[s_]], ov[j0[s_]], oc[j0[s_]] = keys[s_], np.asarray(vals)[s_], live_cnt[s_]
    todo = np.flatnonzero(~s_)
    s, rounds = 0, 0
    while todo.size:
        assert rounds < max_rounds, "probe sequence exhausted"
        j = j0[todo] if s == 0 else (j0[todo] + (s - 1) ** 2) % cap
        free = oc[j] == 0
        np.minimum.at(ok, j[free], keys[todo][free])
        won = free & (ok[j] == keys[todo])
        ov[j[won]], oc[j[won]] = np.asarray(vals)[todo[won]], live_cnt[todo[won]]
        todo = todo[~won]
        s = 2 if s == 0 else s + 1
        rounds += 1
    ok[oc == 0] = 0
    return ok, ov, oc


def _probe_finds_all(keys, vals, cnts, ok, ov, oc):
    M = ok.size
    for k_, v_, c_ in zip(keys.tolist(), vals.tolist(), cnts.tolist()):
        h = int(_fnv4(np.array([k_], dtype=np.uint64))[0])
        j = (h - (1 << 64) if h >> 63 else h) % M
        j0, t = j, 0
        while not (int(ok[j]) == k_ or oc[j] == 0):      # oakht.pointer (:521-538)
            j = (j0 + t * t) % M
            t += 1
        assert int(ok[j]) == k_ and ov[j] == v_ and oc[j] == max(c_, 1)


def _triples(case):
    return (np.array([r[0] for r in case["dbg"]], dtype=np.uint64), np.array([r[1] for r in case["dbg"]], dtype=np.uint16),
            np.array([r[2] for r in case["dbg"]], dtype=np.uint8))


@pytest.mark.parametrize("name", ["test_fsa_k5", "test_fsa_k27", "nasty_k11_lf", "rand05_k15_c2"])
def test_placement_rule_is_probeable(name):
    k, v, c = _triples(CASES[name])
    params, hk, _, _ = npz.oakht_image(k, v, c)
    cap = int(params[0])
    ok, ov, oc = oak_rounds(k, v, c, cap)
    assert ok.size == hk.size == cap
    assert int((oc > 0).sum()) == k.size
    _probe_finds_all(k, v, c, ok, ov, oc)
    perm = np.random.default_rng(1).permutation(k.size)      # the image depends only on the set of entries
    ok2, ov2, oc2 = oak_rounds(k[perm], v[perm], c[perm], cap)
    assert np.array_equal(ok, ok2) and np.array_equal(ov, ov2) and np.array_equal(oc, oc2)


def test_placement_rule_dense_with_sentinel_and_phantom():
    rng = np.random.default_rng(11)
    cap = 1048583                                            # pg_host_oakht_capacity at its first step
    n = int(0.75 * cap)
    k = np.unique(rng.integers(0, 5 ** 15, n + 1000, dtype=np.uint64))[:n - 2]
    k = np.concatenate([k, np.array([0, SENT], dtype=np.uint64)])
    v = rng.integers(0, 4096, k.size).astype(np.uint16)
    c = rng.integers(0, 256, k.size).astype(np.uint8)
    ok, ov, oc = oak_rounds(k, v, c, cap)
    sel = rng.choice(k.size, 20000, replace=False)
    _probe_finds_all(k[np.concatenate([sel, [k.size - 2, k.size - 1]])], v[np.concatenate([sel, [k.size - 2, k.size - 1]])],
                     c[np.concatenate([sel, [k.size - 2, k.size - 1]])], ok, ov, oc)
    assert int((oc > 0).sum()) == k.size


def synthetic_image(n_slots=5_000_000, seed=2):
    """Slot arrays shaped like a k = 27 dBG image: ~68 % live slots, random base-5 keys, sparse masks, small counts."""
    rng = np.random.default_rng(seed)
    n = int(0.68 * n_slots)
    keys = np.zeros(n_slots, np.uint64)
    vals = np.zeros(n_slots, np.uint16)
    cnts = np.zeros(n_slots, np.uint8)
    idx = rng.choice(n_slots, n, replace=False)
    keys[idx] = rng.integers(0, 5 ** 27, n, dtype=np.uint64)
    vals[idx] = rng.integers(0, 4096, n) & rng.integers(0, 4096, n)
    cnts[idx] = np.minimum(rng.geometric(0.4, n), 255)
    return keys, vals, cnts


def test_synthetic_image_size_against_zlib(denc, emul):  # noqa: F811
    for a in synthetic_image():
        raw = npz.npy_header(a.dtype, a.size) + a.tobytes()
        comp = check_roundtrip(denc, emul, raw)
        co = zlib.compressobj(6, zlib.DEFLATED, -15, 8, zlib.Z_RLE)
        rle = b"".join(co.compress(raw[i:i + 65536]) + co.flush(zlib.Z_FULL_FLUSH) for i in range(0, len(raw), 65536))
        assert len(comp) <= 1.02 * len(rle)
        assert len(comp) <= 1.05 * len(zlib.compress(raw, 6))


@pytest.mark.parametrize("name", ["test_fsa_k27", "nasty_k11_lf", "rand05_k15_c2"])
def test_golden_images_roundtrip(denc, emul, name):  # noqa: F811
    params, ok, ov, oc = npz.oakht_image(*_triples(CASES[name]))
    for a in (params, ok, ov, oc):
        check_roundtrip(denc, emul, npz.npy_header(a.dtype, a.size) + a.tobytes())


def write_host_npz(denc, path, arrays):
    """The container of npz.write_container with members compressed by the CPU core."""
    def member(a):
        def compress(write):
            raw = npz.npy_header(a.dtype, a.size) + a.tobytes()
            comp, _, crc = deflate(denc, raw)
            write(comp)
            return crc, len(raw)
        return compress
    npz.write_container(path, [(name + ".npy", member(a)) for name, a in arrays.items()])


def test_container_reads_like_savez_compressed(denc, tmp_path):
    k, v, c = _triples(CASES["rand05_k15_c2"])
    params, ok, ov, oc = npz.oakht_image(k, v, c, offset=1234)
    arrays = dict(parameters=params, keys=ok, values=ov, counts=oc)
    ours = str(tmp_path / "ours.npz")
    write_host_npz(denc, ours, arrays)
    theirs = str(tmp_path / "theirs.npz")
    np.savez_compressed(theirs, **arrays)
    with zipfile.ZipFile(ours) as z:
        assert z.testzip() is None
        names = z.namelist()
        assert all(i.compress_type == zipfile.ZIP_DEFLATED for i in z.infolist())
    with zipfile.ZipFile(theirs) as z:
        assert names == z.namelist()
    a, b = np.load(ours, allow_pickle=False), np.load(theirs, allow_pickle=False)
    for name in arrays:
        assert a[name].dtype == b[name].dtype and a[name].shape == b[name].shape
        assert np.array_equal(a[name], b[name])
    write_host_npz(denc, str(tmp_path / "again.npz"), arrays)
    assert open(ours, "rb").read() == open(str(tmp_path / "again.npz"), "rb").read()


def test_container_empty_arrays(denc, tmp_path):
    arrays = dict(parameters=np.zeros(6, np.uint64), keys=np.zeros(0, np.uint64), values=np.zeros(0, np.uint16),
                  counts=np.zeros(0, np.uint8))
    p = str(tmp_path / "e.npz")
    write_host_npz(denc, p, arrays)
    z = np.load(p)
    assert z["keys"].shape == (0,) and z["counts"].dtype == np.uint8
    with zipfile.ZipFile(io.BytesIO(open(p, "rb").read())) as zz:
        assert zz.testzip() is None
