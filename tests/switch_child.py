"""Runs a fixed battery of builds under whatever PG_* environment it was started with and prints ONE JSON document:
a result per item, and the kernels torch.profiler recorded around the battery (names normalised by
switch_table.norm_kernel, with the grid sizes the trace shows).  tests/test_gpu_switches.py starts it once per profile
and compares every item with the oracle.

    python tests/switch_child.py pack compact b16 split misc

Groups:
  pack     K1 on a ragged 12.8 MB file (switch_table.pack_input)
  compact  build_table on compact 8-byte records: k 27/21/16/15, one region to 2^17 regions (K2c-c fan-outs 2, 64,
           256 and 512), 1 and 3 rounds; sampled builds at k 27/21/15
  b16      build_table on 16-byte records: canonical, literal_rc and literal; region_bits 12, 8 and 0 (the L2-atomic
           K3); one, two and three partition levels (re-split fan-outs 2 to 256); 1 and 3 rounds; one sampled build per mode
  split    the receive-side split K2b (pg_records_split, 2 source segments -> 2^6 and 2^9 buckets) and the coarse ->
           fine refine (pg_records_refine) feeding a region build, through the C ABI
  misc     the fused insert (engine.build_dbg) in all three modes, a build from the device-side record index, and a
           fresh clear of a table full of stale slots

An item that raises records its error and the battery goes on; the process exits 0 unless the battery itself broke."""
import ctypes
import hashlib
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

import switch_table as T  # noqa: E402

_SENTINEL = np.uint64(0xFFFFFFFFFFFFFFFF)


def sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def triples_sha(ks, vs, cs):
    o = np.argsort(ks, kind="stable")
    return sha(ks[o].astype("<u8"), vs[o].astype("<u2"), cs[o].astype("u1"))


class Battery:
    def __init__(self):
        import torch
        from pangenome_b200 import _lib, builder, engine
        self.torch, self.L, self.lib, self.builder, self.engine = torch, _lib.load(), _lib, builder, engine
        self.items = {}
        self._inputs, self._packed = {}, {}

    def data(self, name):
        if name not in self._inputs:
            self._inputs[name] = T.INPUTS[name]()
        return self._inputs[name]

    def packed(self, name):
        if name not in self._packed:
            self._packed[name] = self.engine.PackedSeqs(self.engine.to_device_bytes(self.data(name)))
        return self._packed[name]

    def item(self, name, fn, **meta):
        r = dict(meta)
        try:
            r.update(fn() or {})
        except Exception as e:          # the parent decides whether this error is the expected one
            r["error"] = "%s: %s" % (type(e).__name__, e)
        self.items[name] = r

    def table_result(self, t):
        """claim counter, slot scan, duplicate keys of the unsorted export, sha of the sorted triples, flags"""
        s = t.stats_host()
        claimed = int(s[self.lib.PG_STAT_USED])
        scanned, _ = t.count()
        ks, vs, cs = t.export(sort=False)
        s = t.stats_host()
        return dict(claimed=claimed, scanned=scanned, dup=int(ks.size - np.unique(ks).size), sha=triples_sha(ks, vs, cs),
                    checksum=list(t.checksum()), lost=int(s[self.lib.PG_STAT_LOST]), overflow=int(s[self.lib.PG_STAT_OVERFLOW]),
                    capacity=int(t.capacity))

    # ---- groups ------------------------------------------------------------------------------------------------------
    def pack(self):
        def run():
            data = self.data("pack")
            p = self.engine.PackedSeqs(self.engine.to_device_bytes(data))
            pk2 = p.pk2.cpu().numpy().view(np.uint32)
            amb = p.amb.cpu().numpy().view(np.uint32)
            i = np.arange(int(p.seq_off[0]), int(p.seq_off[-1]), dtype=np.int64)       # the records' bases, junk excluded
            d = (pk2[i >> 4] >> (2 * (i & 15)).astype(np.uint32)) & 3
            a = (amb[i >> 5] >> (i & 31).astype(np.uint32)) & 1
            syms = np.where(a == 1, 4 + d, d).astype(np.uint8)
            return dict(n_rec=p.n_rec, n_bases=p.n_bases, seq_off=sha((p.seq_off - p.seq_off[0]).astype("<i8")),
                        hdr_off=sha(np.asarray(p.hdr_off, dtype="<i8")), syms=sha(syms), tiles=(len(data) + 16383) // 16384)
        self._inputs["pack"] = T.pack_input()
        self.item("pack", run, input="pack", k=T.PACK_K, kind="pack")

    def _build(self, name, inp, k, mode, **kw):
        lib = self.lib
        c = 0 if mode == lib.PG_MODE_LITERAL else 2

        def run():
            t, n_rec, b = self.builder.build_table(self.packed(inp), k, rc=mode != lib.PG_MODE_LITERAL, mode=mode, max_attempts=0, **kw)
            r = self.table_result(t)
            r.update(compact=bool(b.compact), region_bits=int(b.region_bits), levels=b.levels, rounds=int(b.n_rounds),
                     sampled=b.sampler is not None)
            del t, b
            return r
        self.item(name, run, input=inp, k=k, c=c, mode=int(mode), kind="table", **{x: kw.get(x) for x in ("compact", "region_bits")})

    def compact(self):
        C = self.lib.PG_MODE_CANONICAL
        for k in (27, 21, 16, 15):
            for inp, caps in (("pangenome", [1 << 21, 1 << 26, 1 << 28, 1 << 29]), ("hostile", [1 << 14, 1 << 21]), ("hot", [4096, 1 << 14])):
                for cap in caps:
                    for rounds in (1, 3):
                        self._build("compact %s k%d cap2^%d r%d" % (inp, k, cap.bit_length() - 1, rounds), inp, k, C, capacity=cap, rounds=rounds,
                                    region_bits=12, compact=True, sample=False)
            self.torch.cuda.empty_cache()
        for k in (27, 21, 15):
            self._build("compact pangenome k%d sampled" % k, "pangenome", k, C, region_bits=12, compact=True, sample=True)

    def b16(self):
        L = self.lib
        geo = [(12, "pan16", [1 << 20, 1 << 21, 1 << 29]), (8, "hostile", [1 << 16]), (8, "pan16", [1 << 17, 1 << 24, 1 << 25]),
               (0, "pan16", [1 << 17, 1 << 20, 1 << 24])]
        for mode, mname, k in ((L.PG_MODE_CANONICAL, "canonical", 16), (L.PG_MODE_LITERAL_RC, "literal_rc", 21), (L.PG_MODE_LITERAL, "literal", 27)):
            for rb, inp, caps in geo:
                for cap in caps:
                    for rounds in (1, 3):
                        self._build("16B %s %s k%d rb%d cap2^%d r%d" % (mname, inp, k, rb, cap.bit_length() - 1, rounds), inp, k, mode, capacity=cap,
                                    rounds=rounds, region_bits=rb, compact=False, sample=False)
            self._build("16B %s pan16 k%d sampled" % (mname, k), "pan16", k, mode, region_bits=12, compact=False, sample=True)
            self.torch.cuda.empty_cache()

    def split(self):
        lib, eng, bld = self.lib, self.engine, self.builder
        P, S, byref = eng._ptr, eng._stream, ctypes.byref

        def coarse_set(packed, k, bits):
            g0, g1 = int(packed.seq_off[0]), int(packed.seq_off[packed.n_rec])
            coarse = bld.LocalBuckets(bits, (g1 - g0) // (1 << bits) * 2 + 4096, 0, "cuda")
            desc = lib.PgTable(None, 2, None, lib.PG_MODE_CANONICAL, k, 1, 0, 0)
            eng.check(self.L.pg_kmer_partition_to(byref(desc), P(packed.pk2), P(packed.amb), P(packed.d_seq_off), packed.n_rec, g0, g1,
                                                  None, 0, 0, byref(coarse.c), None, 0, None, S()), "pg_kmer_partition_to")
            return coarse, g0, g1

        def k2b(inp, k, bits):
            """two coarse buckets stand for the segments two source ranks sent: K2b splits them into 2^bits buckets"""
            packed = self.packed(inp)
            coarse, g0, g1 = coarse_set(packed, k, 1)
            fine = bld.LocalBuckets(bits, (g1 - g0) // (1 << bits) * 2 + 2048, 1 << 16, "cuda")
            t = eng.DbgTable(1 << 21, k, lib.PG_MODE_CANONICAL)
            eng.check(self.L.pg_count_short(byref(t.c), P(packed.d_seq_off), packed.n_rec, g0, g1, S()), "pg_count_short")
            eng.check(self.L.pg_records_split(P(coarse.records), P(coarse.seg_off), P(coarse.counts), 2, coarse.part_cap, byref(fine.c),
                                              P(t.stats), S()), "pg_records_split")
            eng.check(self.L.pg_buckets_plan(byref(fine.c), P(fine.seg_cnt), P(t.stats), S()), "pg_buckets_plan")
            eng.check(self.L.pg_insert_records(byref(t.c), P(fine.records), P(fine.seg_off), P(fine.seg_cnt), fine.n_parts + 1, 1, 0, S()),
                      "pg_insert_records")
            return self.table_result(t)

        def refine(inp, k):
            """2^4 coarse buckets (K2a) -> 2^8 fine ones (K2c) -> one K3s region of 4096 slots each"""
            packed = self.packed(inp)
            coarse, g0, g1 = coarse_set(packed, k, 4)
            n_fine, part_cap, spill_cap = 1 << 8, (g1 - g0) // 256 * 2 + 2048, 1 << 16
            recs = self.torch.empty(2 * (n_fine * part_cap + spill_cap), dtype=self.torch.int64, device="cuda")
            cnts = self.torch.zeros(n_fine + 1, dtype=self.torch.int64, device="cuda")
            t = eng.DbgTable(1 << 20, k, lib.PG_MODE_CANONICAL)
            t.c.region_bits = 12
            eng.check(self.L.pg_count_short(byref(t.c), P(packed.d_seq_off), packed.n_rec, g0, g1, S()), "pg_count_short")
            eng.check(self.L.pg_records_refine(byref(coarse.c), 8 - 4, P(recs), P(cnts), part_cap, spill_cap, P(t.stats), S()), "pg_records_refine")
            eng.check(self.L.pg_region_build(byref(t.c), P(recs), P(cnts), part_cap, spill_cap, 1, S()), "pg_region_build")
            return self.table_result(t)

        for inp, k in (("pangenome", 27), ("hostile", 21)):
            for bits in (6, 9):
                self.item("K2b %s k%d 2 -> 2^%d" % (inp, k, bits), lambda: k2b(inp, k, bits), input=inp, k=k, c=2, kind="table")
            self.item("refine %s k%d 2^4 -> 2^8" % (inp, k), lambda: refine(inp, k), input=inp, k=k, c=2, kind="table")

    def misc(self):
        lib, eng, bld = self.lib, self.engine, self.builder
        torch = self.torch

        def fused(inp, k, mode):
            t, _ = eng.build_dbg(self.packed(inp), k, rc=mode != lib.PG_MODE_LITERAL, mode=mode)
            r = self.table_result(t)
            r.update(load=eng._DEFAULT_LOAD, positions=self.packed(inp).n_positions(k) * (2 if mode == lib.PG_MODE_LITERAL_RC else 1))
            return r
        for inp, k, mode in (("hot", 11, lib.PG_MODE_CANONICAL), ("hot", 11, lib.PG_MODE_LITERAL_RC), ("hot", 11, lib.PG_MODE_LITERAL),
                             ("hostile", 21, lib.PG_MODE_LITERAL_RC), ("pangenome", 27, lib.PG_MODE_CANONICAL)):
            self.item("fused %s k%d mode %d" % (inp, k, mode), lambda: fused(inp, k, mode), input=inp, k=k, c=0 if mode == lib.PG_MODE_LITERAL else 2,
                      mode=int(mode), kind="fused")

        def lazy():
            """the build bench.py times: record bounds read on the device (pg_count_short_dev), two builds of one builder"""
            packed = eng.PackedSeqs(eng.to_device_bytes(self.data("pangenome")), lazy=True)
            b = bld.RoundBuilder(27, lib.PG_MODE_CANONICAL, len(self.data("pangenome")))
            for _ in range(2):
                b.begin()
                t = b.build_async(packed)
            torch.cuda.synchronize()
            b.verify()
            return self.table_result(t)
        self.item("device-side bounds pangenome k27", lazy, input="pangenome", k=27, c=2, kind="table")

        def clear():
            """a table full of live slots of epoch 1 (a copy of a finished build), then pg_table_clear: every slot reads
            free, and a build into it is exact"""
            cap = 1 << 20
            t0, _ = eng.build_dbg(self.packed("pangenome"), 27, capacity=cap)
            t = eng.DbgTable(cap, 27, lib.PG_MODE_CANONICAL)
            t.slots.copy_(t0.slots)
            stale = t.count()[0]
            del t0
            eng.check(self.L.pg_table_clear(ctypes.byref(t.c), eng._stream()), "pg_table_clear")
            after = t.count()
            t.stats.zero_()
            t.insert(self.packed("hostile"))
            r = self.table_result(t)
            r.update(stale=stale, after_clear=list(after))
            return r
        self.item("clear stale 2^20 then hostile k27", clear, input="hostile", k=27, c=2, kind="clear")


def main(groups):
    bat = Battery()
    torch = bat.torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for g in groups:
            getattr(bat, g)()
        torch.cuda.synchronize()
    kernels = {}
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    for ev in trace.get("traceEvents", []):
        if ev.get("cat") != "kernel":
            continue
        n = T.norm_kernel(ev.get("name", ""))
        if n is not None:
            grid = (ev.get("args") or {}).get("grid")
            kernels.setdefault(n, set())
            if grid:
                kernels[n].add(int(grid[0]))
    for e in prof.key_averages():        # the same names, should the trace leave any out
        n = T.norm_kernel(e.key)
        if n is not None:
            kernels.setdefault(n, set())
    out = dict(items=bat.items, kernels={n: sorted(g) for n, g in kernels.items()},
               sms=torch.cuda.get_device_properties(0).multi_processor_count,
               env={k: v for k, v in os.environ.items() if k.startswith("PG_")})
    sys.stdout.write("\n" + json.dumps(out) + "\n")
    sys.stdout.flush()


if __name__ == "__main__":
    main(sys.argv[1:] or T.ALL_GROUPS)
