"""The kernel variants behind the PG_* switches, against the oracle.

The C++ switches are read once per process into a ``static``, so every profile of tests/switch_table.py starts
tests/switch_child.py once with its environment.  Each item of the child's battery must equal the oracle: the sorted
export triples and the table checksum, the claim counter (PG_STAT_USED) equal to the slot scan and to the oracle's
distinct keys, no duplicate key in the unsorted export, no LOST / OVERFLOW flag.  The kernels the profiler saw must
include what the profile selects and none of what it replaces.

The Python switches (PG_LEVELS, PG_REGION_BITS, PG_COMPACT, PG_ROUNDS, PG_SUB_MB) are read per call and are tested
in-process.  The last test checks that every k1* / k2* / k3* / k_table_clear instantiation in libpgdbg.so is
launched by some profile or allowlisted with a reason."""
import os
import shutil
import signal
import subprocess
import sys

import numpy as np
import pytest

import oracle
import switch_table as T
from conftest import ROOT

pytestmark = pytest.mark.gpu
CHILD = os.path.join(ROOT, "tests", "switch_child.py")
_SENTINEL = np.uint64(0xFFFFFFFFFFFFFFFF)
_RESULTS = {}
_PROFILES = {p[0]: p for p in T.PROFILES}


@pytest.fixture(scope="module")
def gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pangenome_b200 import _lib
    _lib.load()


class Oracle:
    """oracle.run once per (input, k, c): the sha of the sorted triples, the checksum, the distinct keys"""

    def __init__(self):
        self.cache, self.inputs = {}, {}

    def data(self, name):
        if name not in self.inputs:
            self.inputs[name] = T.pack_input() if name == "pack" else T.INPUTS[name]()
        return self.inputs[name]

    def __call__(self, name, k, c):
        key = (name, k, c)
        if key not in self.cache:
            import switch_child as C
            r = oracle.run(self.data(name), k, c=c, stages=1)
            ks, vs, cs = r["dbg"]
            keys = ks[ks != _SENTINEL]
            if c & 2:
                distinct = int(np.unique(np.minimum(keys, rc_codes(keys, k))).size)      # canonical pairs
            else:
                distinct = int(np.unique(keys).size)
            self.cache[key] = dict(sha=C.triples_sha(ks, vs, cs), checksum=list(oracle.table_checksum(ks, vs, cs)), distinct=distinct,
                                   literal=int(np.unique(keys).size), ub=int(r["ub_count"]), ref=r)
        return self.cache[key]


def rc_codes(keys, k):
    x, r = keys.copy(), np.zeros_like(keys)
    for _ in range(k):
        d = x % np.uint64(5)
        x //= np.uint64(5)
        r = r * np.uint64(5) + np.where(d == 4, d, np.uint64(3) - d)
    return r


@pytest.fixture(scope="module")
def ref():
    return Oracle()


def run_profile(name, timeout=420):
    """the child's JSON for profile ``name``; one child per profile and module"""
    if name in _RESULTS:
        return _RESULTS[name]
    import json
    _, env, groups, _, _ = _PROFILES[name]
    e = {k: v for k, v in os.environ.items() if not k.startswith("PG_")}
    e.update(env)
    p = subprocess.Popen([sys.executable, CHILD] + list(groups), stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=e, cwd=ROOT,
                         text=True, start_new_session=True)
    try:
        out, err = p.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        os.killpg(p.pid, signal.SIGKILL)            # the child and anything it started
        p.communicate()
        pytest.fail("profile %s: the child did not finish in %d s" % (name, timeout))
    assert p.returncode == 0, "profile %s: the child exited with %d\n%s" % (name, p.returncode, err[-4000:])
    _RESULTS[name] = json.loads(out.strip().splitlines()[-1])
    return _RESULTS[name]


def expected_error(env, item):
    """the one refusal a profile asks for: 512-thread K2a tiles do not fit the literal-rc mode"""
    if env.get("PG_K2A_THREADS") == "512" and item.get("mode") == 1 and item.get("kind") == "table" and item.get("compact") is False:
        return "512-thread tiles do not fit the literal-rc mode"
    return None


def check_item(name, it, env, ref):
    want_err = expected_error(env, it)
    if want_err:
        assert "error" in it and want_err in it["error"], "%s: expected the refusal %r, got %r" % (name, want_err, it.get("error", "a table"))
        return
    assert "error" not in it, "%s: %s" % (name, it["error"])
    if it["kind"] == "pack":
        r = ref("pack", it["k"], 2)["ref"]
        from switch_child import sha
        lut = np.full(256, 5, np.uint8)
        for ch, v in ((b"Aa", 0), (b"Gg", 1), (b"Cc", 2), (b"Tt", 3), (b"Nn", 4)):
            for c in ch:
                lut[c] = v
        got = (it["n_rec"], it["seq_off"], it["hdr_off"], it["syms"])
        want = (int(r["n_records"]), sha(r["seq_off"].astype("<i8")), sha(r["hdr_off"].astype("<i8")), sha(lut[r["seq"]]))
        assert got == want, "%s: K1 differs from the oracle in (n_rec, seq_off, hdr_off, symbols): %r" % (name, [a == b for a, b in zip(got, want)])
        return
    o = ref(it["input"], it["k"], it["c"])
    assert o["ub"] == 0, "%s: the input has records of k + 1 bases, which the reference leaves undefined" % name
    distinct = o["distinct"] if it.get("mode", 2) == 2 else o["literal"]
    got = (it["sha"] == o["sha"], it["checksum"] == o["checksum"], it["dup"], it["claimed"], it["scanned"], it["lost"], it["overflow"])
    assert got == (True, True, 0, distinct, distinct, 0, 0), (
        "%s: (export equals oracle, checksum equals oracle, duplicate keys, claimed, slot scan, LOST, OVERFLOW) = %r; oracle %d distinct keys"
        % (name, got, distinct))
    if it.get("compact"):
        assert it["compact"] and it["region_bits"] == 12, "%s: not built on compact records: %r" % (name, it)
    if it["kind"] == "clear":
        assert it["stale"] > 0 and it["after_clear"] == [0, 0], "%s: %d stale keys before the clear, %r after" % (name, it["stale"], it["after_clear"])
    if it["kind"] == "fused":
        base = 1 << (max(1024, int(it["positions"] / it["load"]) + 1) - 1).bit_length()
        assert it["load"] == float(env.get("PG_TABLE_LOAD", "0.5")) and it["capacity"] in (base, 2 * base, 4 * base), name


@pytest.mark.parametrize("profile", [p[0] for p in T.PROFILES])
def test_profile(gpu, ref, profile):
    name, env, groups, must, must_not = _PROFILES[profile]
    res = run_profile(profile)
    assert res["env"] == env
    items = res["items"]
    assert items, "profile %s ran no item" % profile
    bad = []
    for iname, it in items.items():
        try:
            check_item(iname, it, env, ref)
        except AssertionError as e:
            bad.append(str(e).split("\n")[0])
    assert not bad, "profile %s: %d of %d items wrong:\n%s" % (profile, len(bad), len(items), "\n".join(bad[:40]))
    names = sorted(res["kernels"])
    missing = [p for pat in must for p in T.expand(pat) if not T.matches(names, p)]
    assert not missing, "profile %s did not launch %s; it launched %s" % (profile, missing, names)
    unwanted = {p: T.matches(names, p) for pat in must_not for p in T.expand(pat) if T.matches(names, p)}
    assert not unwanted, "profile %s launched what it replaces: %s" % (profile, unwanted)
    grids, sms = res["kernels"], res["sms"]
    if "pack" in groups and grids.get("k1x_pack"):
        tiles = items["pack"]["tiles"]
        assert tiles > 5 * sms
        for k1 in ("k1x_pack", "k1x_tile_aggs"):
            if env.get("PG_K1_GRID") == "1":        # one CTA per SM, each looping over 5-6 tiles
                assert max(grids[k1]) == sms and tiles not in grids[k1], (k1, grids[k1])
            else:                                   # one CTA per tile
                assert tiles in grids[k1], (k1, grids[k1], tiles)
    if env.get("PG_CLEAR_CTAS_PER_SM") == "1" and grids.get("k_table_clear"):
        assert max(grids["k_table_clear"]) <= sms, grids["k_table_clear"]
    if profile == "split-policy":              # inert: the same kernels as the default
        assert names == sorted(run_profile("default")["kernels"])


# ---------------------------------------------------------------------------------------------------------------------
# the Python switches, read per call

def _build(monkeypatch, env, data, k, **kw):
    from pangenome_b200 import builder, engine
    for name in ("PG_LEVELS", "PG_REGION_BITS", "PG_COMPACT", "PG_ROUNDS", "PG_SUB_MB"):
        monkeypatch.delenv(name, raising=False)
    for name, v in env.items():
        monkeypatch.setenv(name, v)
    packed = engine.PackedSeqs(engine.to_device_bytes(data))
    t, _, b = builder.build_table(packed, k, sample=False, max_attempts=0, **kw)
    return t, b


def _exact(t, o, where):
    import switch_child as C
    claimed = t.n_keys()
    scanned, _ = t.count()
    ks, vs, cs = t.export(sort=False)
    got = (C.triples_sha(ks, vs, cs) == o["sha"], int(ks.size - np.unique(ks).size), claimed, scanned)
    assert got == (True, 0, o["distinct"], o["distinct"]), "%s: %r, oracle %d distinct keys" % (where, got, o["distinct"])


@pytest.mark.parametrize("levels,cap,compact,rb", [("4,4,4", 1 << 24, True, 12), ("2,3,3", 1 << 20, False, 12), ("11,6", 1 << 25, False, 8),
                                                    ("0,17", 1 << 25, False, 8)])
def test_levels_other_than_the_plan(gpu, ref, monkeypatch, levels, cap, compact, rb):
    """PG_LEVELS with a valid list other than the plan is used on both record forms; a list plan_levels rejects
    (a level of 11 or 0 bits) is ignored and the plan is used"""
    from pangenome_b200 import builder
    t, b = _build(monkeypatch, {"PG_LEVELS": levels}, ref.data("pan16"), 21, capacity=cap, compact=compact, region_bits=rb)
    lv = [int(x) for x in levels.split(",")]
    valid = all(1 <= x <= 10 for x in lv)
    assert b.compact == compact and b.region_bits == rb
    assert b.levels == (lv if valid else builder.plan_levels((cap.bit_length() - 1) - rb, 1, 9 if compact else 8)), b.levels
    _exact(t, ref("pan16", 21, 2), "PG_LEVELS=%s" % levels)


@pytest.mark.parametrize("levels,cap,rb,msg", [("8,9", 1 << 25, 8, "pg_records_resplit"), ("10,4,4", 1 << 26, 8, "pg_records_resplit")])
def test_levels_the_kernels_refuse(gpu, ref, monkeypatch, levels, cap, rb, msg):
    """16-byte records re-split at most 8 bits per level, from at most 2^13 buckets: such a list is a clean PgError"""
    from pangenome_b200._lib import PgError
    with pytest.raises(PgError, match=msg):
        _build(monkeypatch, {"PG_LEVELS": levels}, ref.data("pan16"), 21, capacity=cap, compact=False, region_bits=rb)


@pytest.mark.parametrize("env,kw", [({"PG_REGION_BITS": "8"}, dict(region_bits=8)), ({"PG_REGION_BITS": "0"}, dict(region_bits=0)),
                                    ({"PG_COMPACT": "0"}, dict(compact=False)), ({"PG_ROUNDS": "3"}, dict(rounds=3)),
                                    ({"PG_SUB_MB": "1", "PG_REGION_BITS": "0"}, dict(region_bits=0, sub_bytes=1 << 20))],
                         ids=["region_bits-8", "region_bits-0", "compact-0", "rounds-3", "sub_mb-1"])
def test_python_switch_equals_its_argument(gpu, ref, monkeypatch, env, kw):
    """the same table and the same geometry as the explicit argument"""
    from pangenome_b200 import builder, engine
    data, cap = ref.data("pan16"), 1 << 22
    t, b = _build(monkeypatch, env, data, 21, capacity=cap)
    geo = (b.compact, b.region_bits, b.levels, b.n_rounds, b.sub_bits)
    _exact(t, ref("pan16", 21, 2), "%r" % env)
    for name in env:
        monkeypatch.delenv(name)
    packed = engine.PackedSeqs(engine.to_device_bytes(data))
    sub = kw.pop("sub_bytes", None)
    b2 = builder.RoundBuilder(21, 2, len(data), capacity=cap, sample=False, sub_bytes=sub, **kw)
    b2.begin()
    t2 = b2.build_async(packed, packed.n_rec)
    b2.verify()
    assert (b2.compact, b2.region_bits, b2.levels, b2.n_rounds, b2.sub_bits) == geo
    assert geo != (True, 12, [8, 2], 1, 8), "the switch changed nothing: %r" % (geo,)
    _exact(t2, ref("pan16", 21, 2), "explicit %r" % kw)


# ---------------------------------------------------------------------------------------------------------------------

def _tool(name):
    for d in ([os.environ["CUDA_HOME"]] if os.environ.get("CUDA_HOME") else []) + ["/usr/local/cuda"]:
        p = os.path.join(d, "bin", name)
        if os.path.isfile(p):
            return p
    return shutil.which(name)


def test_every_instantiation_is_launched(gpu):
    """The union of the profiles' kernel lists holds every k1* / k2* / k3* / k_table_clear instantiation in
    libpgdbg.so, except the allowlisted ones."""
    from pangenome_b200._lib import LIB_PATH
    cuobjdump, filt = _tool("cuobjdump"), _tool("cu++filt")
    if not cuobjdump or not filt:
        pytest.skip("cuobjdump / cu++filt not found")
    syms = subprocess.run([cuobjdump, "-symbols", LIB_PATH], capture_output=True, text=True, check=True).stdout
    mangled = sorted(set(w for w in syms.split() if w.startswith("_Z")))
    demangled = subprocess.run([filt], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout.splitlines()
    built = {n for n in (T.norm_kernel(d) for d in demangled) if n and n.startswith(("k1", "k2", "k3", "k_table_clear"))}
    assert len(built) > 60, sorted(built)
    seen = set()
    for p in T.PROFILES:
        seen |= set(run_profile(p[0])["kernels"])
    allowed = {x for pat in T.ALLOWLIST for x in T.expand(pat)}
    assert allowed <= built, sorted(allowed - built)
    never = sorted(built - seen - allowed)
    assert not never, "instantiations no profile launches: %s" % never
