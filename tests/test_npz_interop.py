"""`_db.npz` interop (SURVEY 8 f1).  CPU part: the oakht image written by pangenome_b200.npz is
what the reference's own loader expects - checked by probing like `oakht.pointer`, against the
images the reference itself wrote (its chunk checkpoints in tests/golden/chunk_cases.json), and by
running the reference's load_on_disk + dbg2rdbg on it where oracle/_ref exists.  GPU part:
`-d file.npz` produced by the reference-layout writer round-trips through the GPU table."""
import base64
import io
import json
import os

import numpy as np
import pytest

import oracle
from conftest import GOLDEN, load_small_cases
from oracle import refrun

CASES = {c["name"]: c for c in load_small_cases()}
with open(os.path.join(GOLDEN, "chunk_cases.json")) as f:
    REF_IMAGES = [c for c in json.load(f) if c["brkpt_b64"] is not None]     # written by the reference's dump (:243-261)


def _triples(case):
    k = np.array([r[0] for r in case["dbg"]], dtype=np.uint64)
    v = np.array([r[1] for r in case["dbg"]], dtype=np.uint16)
    c = np.array([r[2] for r in case["dbg"]], dtype=np.uint8)
    return k, v, c


def _fnv4(v):
    a = 0xcbf29ce484222325
    for _ in range(4):
        a ^= v & 0xff
        a = (a * 0x100000001b3) & (2 ** 64 - 1)
        v >>= 8
    return a


def _slot0(key, M):
    """First probe slot of oakht.pointer: the hash is an int64 there and numba's % is Python's floor modulo."""
    h = _fnv4(key)
    return (h - (1 << 64) if h >> 63 else h) % M


@pytest.mark.parametrize("name", ["test_fsa_k5", "test_fsa_k27", "nasty_k11_lf", "rand05_k15_c2"])
def test_oakht_image_is_probeable_like_the_reference(name):
    from pangenome_b200 import npz
    case = CASES[name]
    keys, vals, cnts = _triples(case)
    params, ok, ov, oc = npz.oakht_image(keys, vals, cnts)
    ref = oracle.run(case["input_latin1"].encode("latin-1"), case["k"], c=case["c"], stages=1, image=True)
    assert int(params[0]) == ref["dbg_capacity"] and int(params[2]) == keys.size     # same capacity / size as upstream
    assert params.tolist()[1:] == [750000000, keys.size, 1, 1, 0]
    M = int(params[0])
    for k_, v_, c_ in zip(keys.tolist(), vals.tolist(), cnts.tolist()):
        j = _slot0(k_, M)
        j0, t = j, 0
        while not (int(ok[j]) == k_ or oc[j] == 0):      # oakht.pointer (:521-538)
            j = (j0 + t * t) % M
            t += 1
        assert int(ok[j]) == k_ and ov[j] == v_ and oc[j] == c_


def test_reference_loads_our_image(tmp_path):
    """The image we write for a table is, slot for slot, the one the reference writes for it: compared with every
    checkpoint image the reference wrote (and resumed from) in the golden chunk cases, so its load_on_disk reads back
    its own layout and its pointer() finds every key.  The nasty_k11_lf image read back the way load_on_disk reads it
    (live slots) is the reference's dBG, whose rdBG is the golden one; where oracle/_ref exists the reference's own
    load_on_disk + dbg2rdbg run on that image as well."""
    from pangenome_b200 import npz
    for ref in REF_IMAGES:
        z = np.load(io.BytesIO(base64.b64decode(ref["brkpt_b64"])))
        keys = np.array([e[0] for e in ref["brkpt_live"]], dtype=np.uint64)
        vals = np.array([e[1] for e in ref["brkpt_live"]], dtype=np.uint16)
        cnts = np.array([e[2] for e in ref["brkpt_live"]], dtype=np.uint8)
        ours = npz.oakht_image(keys, vals, cnts, offset=ref["offset"])
        for name, a in zip(("parameters", "keys", "values", "counts"), ours):
            assert np.array_equal(a, z[name]), (ref["name"], name)
    case = CASES["nasty_k11_lf"]
    keys, vals, cnts = _triples(case)
    params, ok, ov, oc = npz.oakht_image(keys, vals, cnts)
    fn = str(tmp_path / "x_db")
    np.savez_compressed(fn, parameters=params, keys=ok, values=ov, counts=oc)
    z = np.load(fn + ".npz")
    live = z["counts"] > 0
    assert int(z["parameters"][2]) == live.sum() == len(case["dbg"])
    o = np.argsort(z["keys"][live], kind="stable")
    assert [[int(a), int(b), int(c)] for a, b, c in zip(z["keys"][live][o], z["values"][live][o], z["counts"][live][o])] == case["dbg"]
    if not refrun.available():
        return
    mod = refrun.load()
    offset, kd = mod.load_on_disk(fn + ".npz")
    assert kd.size == keys.size
    rd = mod.dbg2rdbg(kd)
    rk, _, _ = refrun.table_triples(rd)
    assert rk.tolist() == case["rdbg"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["test_fsa_k5", "nasty_k11_lf", "rand05_k15_c2", "rand21_k15_c0"])
def test_gpu_dump_and_load_roundtrip(name, tmp_path):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pangenome_b200 import engine, graph, npz
    case = CASES[name]
    data = case["input_latin1"].encode("latin-1")
    k, c = case["k"], case["c"]
    rc0, rc1 = bool((c >> 1) & 1), bool(c & 1)
    packed = engine.PackedSeqs(engine.to_device_bytes(data))
    t, _ = engine.build_dbg(packed, k, rc=rc0)
    fn = npz.dump(t, str(tmp_path / "in.fa_db"))
    z = np.load(fn)
    live = z["counts"] > 0
    o = np.argsort(z["keys"][live])
    got = [[int(a), int(b), int(d)] for a, b, d in zip(z["keys"][live][o], z["values"][live][o], z["counts"][live][o])]
    assert got == case["dbg"]
    # -d: load the file into a (literal-key) GPU table and run the remaining stages on it
    t2 = npz.load(fn, k)
    ks, vs, cs = t2.export()
    assert [[int(a), int(b), int(d)] for a, b, d in zip(ks, vs, cs)] == case["dbg"]
    rd = t2.select_rdbg()
    rk, _ = rd.rdbg_export()
    assert rk.tolist() == case["rdbg"]
    res = graph.seq2graph_device(packed, rd, k, rc=rc1)
    assert res.xyz_lines() == case["xyz"]
    assert res.rows(packed, data) == [tuple(r) for r in case["rows"]]
