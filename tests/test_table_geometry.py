"""CPU check of the dBG table's home-slot rule at every geometry the builder produces (tests/table_geometry_emul.cu runs
table_dev.cuh's make_view / tv_home / tv_next on the host).  The shared-memory region kernels (K3s, K3s-c) place a key
at the first free slot of its group-aligned home group inside its region; every generic upsert and look-up (spill and
wide-record inserts, DbgTable.insert) probes from tv_home.  A key the generic probe cannot find from tv_home is claimed
a second time by the next upsert of it.  No GPU needed."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

_SO = os.path.join(ROOT, "tests", "_table_geometry_emul.so")
_GROUP = 4                                   # PG_REGION_GROUP
_ALL = (1 << 64) - 1


@pytest.fixture(scope="module")
def tg():
    src = os.path.join(ROOT, "tests", "table_geometry_emul.cu")
    deps = [src, os.path.join(ROOT, "include", "pgdbg.h")] + [os.path.join(ROOT, "pangenome_b200", "csrc", f) for f in
                                                              ("table_dev.cuh", "kmer_core.cuh", "common.cuh")]
    if not os.path.isfile(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps):
        # compiled under a private name and renamed into place: parallel test workers never load a half-written library
        tmp = "%s.%d.so" % (_SO[:-3], os.getpid())
        subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-std=c++17", "--shared",
                               "-Xcompiler", "-fPIC", "-o", tmp, src])
        os.replace(tmp, _SO)
    L = ctypes.CDLL(_SO)
    L.tg_place_lookup.restype = ctypes.c_int64
    return L


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def view(L, bits, rb, hk, k):
    out = np.zeros(4, np.uint64)
    L.tg_view(bits, rb, hk, k, _p(out))
    return {n: int(x) for n, x in zip(("capmask", "rmask", "hmask", "shift"), out)}


def homes(L, bits, rb, hk, k, keys):
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    tv, region, flat = (np.zeros(keys.size, np.uint64) for _ in range(3))
    L.tg_homes(bits, rb, hk, k, _p(keys), ctypes.c_int64(keys.size), _p(tv), _p(region), _p(flat))
    return tv, region, flat


def random_keys(rng, n, k, ambiguous=0.1):
    """Base-5 k-mer codes (digit i weighs 5^i; digit 4 = the ambiguity code): ACGT-only keys, and a share with one
    ambiguity digit (keys without a 2-bit form: hash_kind 1 places them by mix64(~key))."""
    d = rng.integers(0, 4, (n, k), dtype=np.uint64)
    amb = rng.random(n) < ambiguous
    d[amb, rng.integers(0, k, int(amb.sum()))] = 4
    keys = d @ (np.uint64(5) ** np.arange(k, dtype=np.uint64))
    _, first = np.unique(keys, return_index=True)
    return keys[np.sort(first)]


# every geometry pg_region_build / pg_region_build_c and RoundBuilder accept: 2^0 .. 2^18 regions of 256 or 4096 slots
@pytest.mark.parametrize("k", [5, 21, 27])
@pytest.mark.parametrize("hk", [0, 1])
@pytest.mark.parametrize("rb", [8, 12])
def test_region_view_home_rule(tg, rb, hk, k):
    rng = np.random.default_rng(rb * 100 + hk * 30 + k)
    keys = random_keys(rng, 4000, k)
    for bits in range(rb, rb + 19):
        v = view(tg, bits, rb, hk, k)
        assert v["capmask"] == (1 << bits) - 1 and v["shift"] == 64 - bits
        assert v["rmask"] == (1 << rb) - 1, "bits %d" % bits
        assert v["hmask"] == _ALL & ~(_GROUP - 1), "bits %d: home not rounded down to a group" % bits
        tv, region, _ = homes(tg, bits, rb, hk, k, keys)
        assert np.all(tv & np.uint64(_GROUP - 1) == 0) and np.all(tv < np.uint64(1 << bits))
        bad = np.flatnonzero(tv != region)
        assert bad.size == 0, "bits %d region_bits %d: tv_home differs from the region kernels' home for %d of %d keys" % (
            bits, rb, bad.size, keys.size)


@pytest.mark.parametrize("hk", [0, 1])
@pytest.mark.parametrize("bits,rb", [(10, 0), (12, 0), (20, 0), (8, 12), (11, 12), (4, 8), (7, 8)])
def test_view_without_regions(tg, bits, rb, hk):
    """region_bits 0 (the L2-atomic K3), or a table smaller than one region: probing wraps around the whole table from
    the unrounded home slot."""
    keys = random_keys(np.random.default_rng(bits), 2000, 21)
    v = view(tg, bits, rb, hk, 21)
    assert v["rmask"] == v["capmask"] == (1 << bits) - 1 and v["hmask"] == _ALL
    tv, _, flat = homes(tg, bits, rb, hk, 21, keys)
    assert np.array_equal(tv, flat)
    assert np.count_nonzero(tv & np.uint64(_GROUP - 1)) > keys.size // 2          # really unrounded


def keys_at_load(L, rng, bits, rb, hk, k, load):
    """Random keys, exactly round(load * 2^rb) of them hashing into each region of a 2^bits-slot table."""
    n_reg, want = 1 << (bits - rb), int(round(load * (1 << rb)))
    keys = random_keys(rng, 3 * n_reg * want + 4096, k)
    _, region, _ = homes(L, bits, rb, hk, k, keys)
    reg = (region >> np.uint64(rb)).astype(np.int64)
    order = np.argsort(reg, kind="stable")
    rank = np.arange(keys.size) - np.searchsorted(reg[order], reg[order])        # position of each key within its region
    pick = np.sort(order[rank < want])
    assert np.array_equal(np.bincount(reg[pick], minlength=n_reg), np.full(n_reg, want))
    return keys[pick]


@pytest.mark.parametrize("load", [0.1, 0.5, 0.9])
@pytest.mark.parametrize("hk", [0, 1])
@pytest.mark.parametrize("rb", [8, 12])
def test_region_placement_found_by_generic_probe(tg, rb, hk, load):
    """Keys placed by the region kernels' rule are all found by the generic probe from tv_home, and upserting them again
    claims nothing: at one region (capacity == 2^region_bits), two, and eight."""
    rng = np.random.default_rng(int(load * 10) + 7 * hk + rb)
    wrapped = 0
    for bits in (rb, rb + 1, rb + 3):
        for k in (21, 27):
            keys = keys_at_load(tg, rng, bits, rb, hk, k, load)
            stats = np.zeros(5, np.int64)
            bad = tg.tg_place_lookup(bits, rb, hk, k, _p(keys), ctypes.c_int64(keys.size), _p(stats))
            where = "bits %d region_bits %d k %d load %.1f" % (bits, rb, k, load)
            assert stats[0] == 0, where
            if load >= 0.5:
                assert stats[1] > 0, where + ": no key left its home group, the probe went untested"
            wrapped += int(stats[2])
            assert stats[3] == 0, "%s: the generic probe misses %d of %d keys" % (where, stats[3], keys.size)
            assert stats[4] == 0, "%s: a later upsert claims %d keys a second time" % (where, stats[4])
            assert bad == 0
    if load >= 0.9:
        assert wrapped > 0, "no probe wrapped at a region's end"
