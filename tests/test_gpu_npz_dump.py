"""The `_db.npz` image written on the GPU (pg_oakht_place + pg_deflate_chunks / pg_deflate_compact, through npz.dump):
slot for slot the numpy statement of the placement rule (tests/test_deflate_host.py: oak_rounds), member for member the
bytes of the CPU build of the encoder core, readable by np.load and npz.load, identical from dump to dump, and - under
torchrun - written by rank 0 from a gather to rank 0 alone, byte-identical to the one-GPU file."""
import datetime
import os
import socket
import struct
import zipfile

import numpy as np
import pytest

from conftest import load_small_cases
from test_deflate_host import deflate, denc, oak_rounds  # noqa: F401  (the CPU encoder, its fixture and the placement rule)

pytestmark = pytest.mark.gpu
CASES = {c["name"]: c for c in load_small_cases()}
MEMBERS = [("parameters", np.uint64), ("keys", np.uint64), ("values", np.uint16), ("counts", np.uint8)]


@pytest.fixture(scope="module")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pangenome_b200 import _lib
    _lib.load()
    return torch


def raw_members(path):
    """{name: raw DEFLATE bytes} of the zip members, read at their local headers."""
    out = {}
    blob = open(path, "rb").read()
    with zipfile.ZipFile(path) as z:
        for info in z.infolist():
            off = info.header_offset
            nlen, elen = struct.unpack("<HH", blob[off + 26:off + 30])
            start = off + 30 + nlen + elen
            out[info.filename[:-4]] = blob[start:start + info.compress_size]
    return out


def check_file(denc, path, keys, vals, cnts, offset=0):  # noqa: F811
    """The file holds the numpy rule's image of the entries, and each member is the CPU core's compression of it."""
    from pangenome_b200 import _lib, npz
    z = np.load(path, allow_pickle=False)
    n = keys.size
    cap = int(_lib.load().pg_host_oakht_capacity(n))
    assert z["parameters"].tolist() == [cap, 750000000, n, 1, 1, offset]
    ok, ov, oc = oak_rounds(keys, vals, cnts, cap)
    assert np.array_equal(z["keys"], ok) and np.array_equal(z["values"], ov) and np.array_equal(z["counts"], oc)
    raw = raw_members(path)
    for name, dt in MEMBERS:
        a = z[name]
        assert a.dtype == dt and a.shape == (cap if name != "parameters" else 6,)
        assert raw[name] == deflate(denc, npz.npy_header(a.dtype, a.size) + a.tobytes())[0], name
    with zipfile.ZipFile(path) as zz:
        assert zz.testzip() is None
    return z


def _live(z):
    live = z["counts"] > 0
    o = np.argsort(z["keys"][live], kind="stable")
    return z["keys"][live][o], z["values"][live][o], z["counts"][live][o]


def _roundtrip(cuda, denc, t, tmp_path, k):  # noqa: F811
    from pangenome_b200 import npz
    ks, vs, cs = t.export()
    fn = npz.dump(t, str(tmp_path / "x_db"))
    z = check_file(denc, fn, ks, vs, cs)
    lk, lv, lc = _live(z)
    assert np.array_equal(lk, ks) and np.array_equal(lv, vs) and np.array_equal(lc, cs)
    t2 = npz.load(fn, k)
    k2, v2, c2 = t2.export()
    assert np.array_equal(k2, ks) and np.array_equal(v2, vs) and np.array_equal(c2, cs)
    fn2 = npz.dump(t, str(tmp_path / "y_db"))
    assert open(fn, "rb").read() == open(fn2, "rb").read()
    return fn


@pytest.mark.parametrize("name", ["test_fsa_k5", "test_fsa_k27", "nasty_k11_lf", "rand05_k15_c2", "rand21_k15_c0"])
def test_golden(cuda, denc, name, tmp_path):  # noqa: F811
    from pangenome_b200 import engine
    case = CASES[name]
    packed = engine.PackedSeqs(engine.to_device_bytes(case["input_latin1"].encode("latin-1")))
    t, _ = engine.build_dbg(packed, case["k"], rc=bool((case["c"] >> 1) & 1))
    fn = _roundtrip(cuda, denc, t, tmp_path, case["k"])
    lk, lv, lc = _live(np.load(fn))
    assert [[int(a), int(b), int(c)] for a, b, c in zip(lk, lv, lc)] == case["dbg"]


def test_reference_loader(cuda, tmp_path):
    """Where the reference is installed (oracle/_ref), its own load_on_disk + dbg2rdbg read our file to the golden rdBG."""
    from oracle import refrun
    if not refrun.available():
        pytest.skip("oracle/_ref (the reference) is not installed")
    from pangenome_b200 import engine, npz
    case = CASES["nasty_k11_lf"]
    packed = engine.PackedSeqs(engine.to_device_bytes(case["input_latin1"].encode("latin-1")))
    t, _ = engine.build_dbg(packed, case["k"], rc=bool((case["c"] >> 1) & 1))
    fn = npz.dump(t, str(tmp_path / "ref_db"))
    mod = refrun.load()
    _, kd = mod.load_on_disk(fn)
    assert kd.size == len(case["dbg"])
    rk, _, _ = refrun.table_triples(mod.dbg2rdbg(kd))
    assert rk.tolist() == case["rdbg"]


def test_synthetic_pangenome(cuda, denc, tmp_path):  # noqa: F811
    from pangenome_b200 import engine, synth
    data = synth.pangenome(3, 200_000, seed=9)
    packed = engine.PackedSeqs(engine.to_device_bytes(data))
    t, _ = engine.build_dbg(packed, 27)
    _roundtrip(cuda, denc, t, tmp_path, 27)


def test_config2(cuda, denc, tmp_path):  # noqa: F811
    """Config 2 (10 x 5 Mbp, 1 % SNP) through the CLI's stage API; the compressed size against zlib is printed."""
    import zlib
    from pangenome_b200 import stages, synth
    qry = str(tmp_path / "cfg2.fa")
    with open(qry, "wb") as f:
        f.write(synth.pangenome(10, 5_000_000))
    h = stages.seq2rdbg(qry, 27, 5, 1e18, brkpt="", rc=True)
    ks, vs, cs = h.table.export()
    fn = stages.dump(h, qry + "_db")
    z = check_file(denc, fn, ks, vs, cs)
    raw = raw_members(fn)
    a = z["keys"]
    keys_raw = a.tobytes()
    co = zlib.compressobj(6, zlib.DEFLATED, -15, 8, zlib.Z_RLE)
    rle = sum(len(co.compress(keys_raw[i:i + 65536]) + co.flush(zlib.Z_FULL_FLUSH)) for i in range(0, len(keys_raw), 65536))
    print("config 2: %d entries, file %d bytes; keys member %.4f of raw, %.4f of zlib Z_RLE 64 KiB chunks"
          % (ks.size, os.path.getsize(fn), len(raw["keys"]) / len(keys_raw), len(raw["keys"]) / rle))


def test_chunked_build_checkpoint_is_a_device_image(cuda, denc, tmp_path):  # noqa: F811
    """The chunked build's `_db_brkpt.npz` comes from the same writer, with the resume offset in parameters[5]."""
    from pangenome_b200 import stages, synth
    qry = str(tmp_path / "ck.fa")
    with open(qry, "wb") as f:
        f.write(synth.pangenome(4, 20_000, seed=3))
    h = stages.seq2rdbg(qry, 15, 5, 1e18, chunk=50_000, brkpt="", rc=True)
    ck = qry + "_db_brkpt.npz"
    assert os.path.isfile(ck) and h.table is not None
    z = np.load(ck)
    lk, lv, lc = _live(z)
    check_file(denc, ck, lk, lv, lc, offset=int(z["parameters"][5]))


# ---- ranks on one device (gloo), the spawn pattern of tests/test_gpu_multi_one_device.py -------------------------------

def _rank_main(rank, world, port, qry, want, fallback_out):
    import torch
    import torch.distributed as dist
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world, timeout=datetime.timedelta(seconds=600))
    try:
        from pangenome_b200 import multigpu, stages

        def no_gather_export(*a, **kw):
            raise AssertionError("stages.dump called gather_export")
        multigpu.gather_export = no_gather_export
        h = stages.seq2rdbg(qry, 27, 5, 1e18, brkpt="", rc=True)
        out_dir = os.path.dirname(want)
        fn = stages.dump(h, os.path.join(out_dir, "w%d_db" % world))
        if rank == 0:
            assert open(fn, "rb").read() == open(want, "rb").read()
        else:
            assert fn is None
        fn2 = stages.dump(h, fallback_out, budget=1)             # rank 0 writes on the host
        if rank == 0:
            a, b = np.load(fn2), np.load(want)
            assert a["parameters"].tolist() == b["parameters"].tolist()
            for x, y in zip(_live(a), _live(b)):
                assert np.array_equal(x, y)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])       # the hash-partitioned build takes power-of-two worlds
def test_ranks_on_one_device(cuda, tmp_path, world):
    import torch.multiprocessing as mp
    from pangenome_b200 import stages, synth
    qry = str(tmp_path / "mg.fa")
    with open(qry, "wb") as f:
        f.write(synth.pangenome(3, 100_000, seed=4))
    h = stages.seq2rdbg(qry, 27, 5, 1e18, brkpt="", rc=True)
    want = stages.dump(h, str(tmp_path / "one_db"))
    del h
    cuda.cuda.synchronize()
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_rank_main, args=(world, port, qry, want, str(tmp_path / ("fb%d_db" % world))), nprocs=world, join=True)
