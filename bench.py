#!/usr/bin/env python
"""bench.py - dBG build throughput (G k-mers/s) of the B200 path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload cfg2|cfg3|cfg4|cfg5|small|cfg4s] [--k 27] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A *step* is one full dBG build of the workload: FASTA scan/pack (K1) + table reset +
k-mer extraction into hash-partitioned compact 8-byte update records (K2a-c; across GPUs fused with the exchange over
NVLink) + partition level(s) (K2b-c / K2c-c) + the table regions built in shared memory (K3s-c) + the wide-record
upserts.  Metric = k-mer insertions / s, an insertion being one k-mer occurrence on one strand:
2 * sum max(n_r - k + 1, 1) over records (BASELINE.md section 3).  Workload: BASELINE configs[1] at one GPU, configs[3]
(strong scaling, ONE file split by byte range) at 2 / 4 / 8 GPUs.

 value   : device-resident input (the FASTA bytes already in HBM), CUDA events around exactly K steps, max over ranks.
 e2e     : the same build through the public host API with HOST buffers: pinned FASTA bytes -> H2D, build, D2H of the
           table statistics.
 roofline: the dominant kernel (k3s_region_build_c; k3_insert_records on tables beyond 2^18 regions), timed live with
           CUDA events on the launching stream; algorithmic bytes = 16 B per insertion (SURVEY.md 8d); the other kernels
           of the path in other_kernels with their own conventions.
 cpu_baseline: the reference's numba code (oracle/_ref, kind "reference") or, if that is unavailable, the C port
           (oracle/, kind "port"), one core, on a bounded sample of the same workload.
 checksum: the built table's order-independent checksum, compared with the oracle's (configs 2 / 3) or the recorded one
           (configs 4 / 5) BEFORE anything is timed: a line is only printed for a correct table.

--dump-outputs DIR writes the table the last timed step built as DIR/<name>.npy (see dump_outputs), so that two builds
of the project can be compared output for output on the same seeded workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "dbg_build_kmers_per_s"
UNIT = "G k-mers/s"


WORKLOADS = {
    # name: (description, generator kind, genomes, genome length)
    "cfg2": ("synthetic 10 x 5 Mbp genomes, 1% SNP (BASELINE configs[1])", "pangenome", 10, 5_000_000),
    "cfg3": ("synthetic 200 x 5 Mbp pangenome (BASELINE configs[2])", "pangenome", 200, 5_000_000),
    "small": ("synthetic 4 x 1 Mbp genomes, 1% SNP", "pangenome", 4, 1_000_000),
    "cfg4": ("synthetic 8 x 500 Mbp repeat-rich plant-like genomes, 5 chromosomes each, 1% SNP (BASELINE configs[3])", "plant", 8, 500_000_000),
    "cfg5": ("synthetic 40 x 500 Mbp repeat-rich plant-like pangenome, 5 chromosomes each (BASELINE configs[4])", "plant", 40, 500_000_000),
    "cfg4s": ("plant-like 8 x 5 Mbp (configs[3] at 1/100 scale)", "plant", 8, 5_000_000),
}


def workload(name, world=1, rank=0, scale=1.0):
    """The bytes of rank ``rank``'s record-aligned byte range of the ONE workload file (SURVEY 8e), its description, and
    (begin, end, file size).  Plant-like sets are generated per rank: only the genomes inside the rank's range."""
    from pangenome_b200 import shard, synth
    if name not in WORKLOADS:
        raise SystemExit("unknown workload %r (have: %s)" % (name, ", ".join(sorted(WORKLOADS))))
    text, kind, genomes, length = WORKLOADS[name]
    length = max(1000, int(length * scale))
    if scale != 1.0:
        text += " x scale %g" % scale
    if kind == "pangenome":
        data = synth.pangenome(genomes, length)
        cuts = shard.cut_points(data, world)
        a, b = cuts[rank], cuts[rank + 1]
        return data[a:b], text, (a, b, len(data))
    n_chrom = 5
    fams = max(20, int(2000 * min(1.0, length / 500_000_000 * 10)))
    layout, size = synth.plant_layout(genomes, length, n_chrom)
    starts = [o for _, _, o, _ in layout]
    cuts = shard.cut_points_from_starts(starts, size, world)
    a, b = cuts[rank], cuts[rank + 1]
    idx = [i for i, s_ in enumerate(starts) if a <= s_ < b]
    data = synth.plant_like(genomes, length, n_chrom, n_families=fams, records=(idx[0], idx[-1] + 1)) if idx else b""
    assert len(data) == b - a, "plant_layout disagrees with the generated records"
    return data, text, (a, b, size)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML (every ~2 ms) DURING the timed region."""

    def __init__(self, index=0):
        self.sm, self.reasons, self.max_mhz, self.stop_flag, self.th = [], set(), None, False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:
            self.nv = None
            self.err = str(e)

    def _loop(self):
        nv = self.nv
        names = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("hw_thermal_slowdown", 0x40),
                 ("sw_thermal_slowdown", 0x20), ("hw_power_brake_slowdown", 0x80))
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for n, bit in names:
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv:
            self.th = threading.Thread(target=self._loop, daemon=True)
            self.th.start()

    def stop(self):
        if not self.nv:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self.stop_flag = True
        self.th.join(timeout=2)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(sm)}


def cpu_reference_rate(data, k, sample_bases, prefer="reference"):
    """Time the CPU dBG stage on the first records of `data` totalling about
    `sample_bases` bases.  Returns (M inserts/s, kind, cores, sample text)."""
    import numpy as np
    # cut the sample at a record boundary
    pos, acc, cut = 0, 0, len(data)
    while True:
        nxt = data.find(b"\n>", pos + 1)
        if nxt < 0:
            break
        acc = nxt
        pos = nxt
        if acc >= sample_bases:
            cut = nxt + 1
            break
    sample = data[:cut]
    if len(sample) > sample_bases * 1.3:      # a single huge record: truncate its body instead
        sample = data[:int(sample_bases)]
        sample = sample[:sample.rfind(b"\n") + 1]
    kind = "port"
    if prefer == "reference":
        try:
            from oracle import refrun
            if refrun.available():
                refrun.run(b">w\n" + b"ACGTTGCATG" * 20 + b"\n", k, stages="dbg")      # JIT warm-up, untimed
                tm = {}
                res = refrun.run(sample, k, stages="dbg", timings=tm)
                import oracle
                n_ins = oracle.run(sample, k, stages=1)["n_inserts"]
                return n_ins / tm["dbg"] / 1e9, "reference", 1, "%d bytes / %d insertions of the workload, numba steady state (JIT excluded)" % (len(sample), n_ins)
        except Exception as e:  # numba missing on the box, etc.
            sys.stderr.write("bench: reference unavailable (%s), using the C port\n" % e)
    import oracle
    res = oracle.run(sample, k, stages=1)
    return res["n_inserts"] / res["times"]["dbg"] / 1e9, kind, 1, "%d bytes / %d insertions of the workload, C port of the reference" % (len(sample), res["n_inserts"])


def run_reference_arm(args):
    """--impl reference: the reference's own CPU code (numba, oracle/_ref; the C port if numba is missing) on a
    bounded sample of the same workload per step, sized so that the whole run stays within a few minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # the sample is a prefix of the workload file: for the plant-like sets only the first record is generated
    n_first = 40 if WORKLOADS[args.workload][1] == "plant" else 1
    data, wl, _ = workload(args.workload, world=n_first, rank=0, scale=args.scale)
    total_steps = max(1, args.warmup + args.steps)
    budget_s = 150.0
    # calibrate on a small sample (also warms the JIT), then size the per-step sample to the time budget
    r0, kind, cores, text = cpu_reference_rate(data, args.k, 100_000)
    per_step_s = budget_s / total_steps
    sample_bases = int(min(1_000_000, max(50_000, r0 * 1e9 * per_step_s / 2)))     # 2 insertions per base
    rates = []
    t0 = time.time()
    for i in range(total_steps):
        r, kind, cores, text = cpu_reference_rate(data, args.k, sample_bases)
        if i >= args.warmup:
            rates.append(r)
    val = sum(rates) / len(rates)
    ms = 1e3 * (time.time() - t0) / total_steps
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak" if args.gpus == 1 else "strong",
            "vs_baseline": None,
            "dtype": "int64", "data": "synthetic", "config": {"workload": wl, "k": args.k, "rc": True},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": text,
                             "host_cpus": os.cpu_count()},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def golden_checksum(workload_name, k, scale):
    """The expected table checksum of a full workload, when tests/golden holds one: oracle facts for configs 2/3, the
    single-GPU build's own result for the configs the oracle cannot hold in memory (labelled as such in the file)."""
    if scale != 1.0:
        return None, None
    gold = os.path.join(ROOT, "tests", "golden")
    try:
        if workload_name == "cfg2" and k == 27:
            return json.load(open(os.path.join(gold, "cfg2_oracle_facts.json")))["dbg_checksum"], "oracle"
        if workload_name == "cfg3":
            f = json.load(open(os.path.join(gold, "cfg3_oracle_facts.json")))["k"].get(str(k))
            return (f["dbg_checksum"], "oracle") if f else (None, None)
        f = json.load(open(os.path.join(gold, "gpu_facts.json"))).get("%s_k%d" % (workload_name, k))
        return (f["dbg_checksum"], f.get("source", "gpu")) if f else (None, None)
    except (OSError, KeyError, ValueError):
        return None, None


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, table, world=1, rank=0, seed=0):
    """Write ``table`` (what RoundBuilder.build_async returned) as float arrays under ``out_dir``: its exported entries in
    key order - the 64-bit base-5 key split into exact 32-bit halves (float64 holds 53 bits), value and count - with
    their positions in that order, and the table's (entries, sum, xor) checksum, 64-bit words split the same way.  A
    table with more entries than DUMP_BYTES allows is written as a fixed, seeded sample of positions.  With several
    ranks every rank writes its own part (``_rank<r>`` names) within its share of DUMP_BYTES."""
    import numpy as np
    ks, vs, cs = table.export()
    n, s, x = table.checksum()
    per_entry = 8 + 8 + 4 + 4 + 8                       # key_hi, key_lo, position (float64), value, count (float32)
    cap = (DUMP_BYTES // world - 4096) // per_entry
    pos = np.arange(ks.size) if ks.size <= cap else np.sort(np.random.default_rng(seed).choice(ks.size, cap, replace=False))
    arrays = {
        "dbg_key_hi": (ks[pos] >> np.uint64(32)).astype(np.float64),
        "dbg_key_lo": (ks[pos] & np.uint64(0xFFFFFFFF)).astype(np.float64),
        "dbg_value": vs[pos].astype(np.float32),
        "dbg_count": cs[pos].astype(np.float32),
        "dbg_position": pos.astype(np.float64),
        "dbg_checksum": np.array([n, s >> 32, s & 0xFFFFFFFF, x >> 32, x & 0xFFFFFFFF], dtype=np.float64),
    }
    os.makedirs(out_dir, exist_ok=True)
    suffix = "_rank%d" % rank if world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default=None, help="cfg2 (default at 1 GPU), cfg3, cfg4 (default at 2/4/8 GPUs), cfg5, small, cfg4s")
    ap.add_argument("--k", type=int, default=27)
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the genome length of the workload (testing)")
    ap.add_argument("--rounds", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stages", action="store_true", help="skip the K1/K4..K8 roofline entries and the atomic ceiling")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the table the last timed step built as DIR/<name>.npy (float32 / float64, <= 64 MB; --impl ours). "
                         "Untimed, but it exports the whole table: 11 B of device memory per entry and a host sort")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.workload is None:
        # BASELINE.json: the metric is quoted on configs[1] (1 GPU); configs[3] is the one "hash-sharded at 2/4/8 GPUs"
        args.workload = "cfg2" if max(world, args.gpus) == 1 else "cfg4"
    big = WORKLOADS.get(args.workload, ("", "", 0, 0))[2] * WORKLOADS.get(args.workload, ("", "", 0, 0))[3] * args.scale > 5e8
    if args.steps is None:
        args.steps = 10 if big else 50
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU build's table: it needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference_arm(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from pangenome_b200 import _lib, builder as pgbuilder, engine, measure

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def allsum(v):
        if world == 1:
            return int(v)
        t = torch.tensor([int(v)], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item())

    def allmax(v):
        if world == 1:
            return float(v)
        t = torch.tensor([float(v)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    t_gen = time.time()
    data, wl, (b0, b1, file_size) = workload(args.workload, world, rank, args.scale)
    t_gen = time.time() - t_gen
    k = args.k
    host = torch.frombuffer(bytearray(data) if data else bytearray(16), dtype=torch.uint8)[:len(data)].pin_memory()
    d_fasta = host.to("cuda", non_blocking=True)
    torch.cuda.synchronize()

    # one untimed pack to know the unit count; table + record buffers stay resident across steps
    packed = engine.PackedSeqs(d_fasta)
    n_ins_local = packed.n_insertions(k)
    n_ins = allsum(n_ins_local)
    n_bases, n_pos_local = allsum(packed.n_bases), packed.n_positions(k)
    bld = pgbuilder.RoundBuilder(k, _lib.PG_MODE_CANONICAL, max(len(data), 1), world=world, rank=rank, rounds=args.rounds)
    stream = torch.cuda.current_stream()
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def step_device(kev=None):
        # no host synchronisation inside a step: K1's record index stays on the device and K2a / K3 take
        # their bounds from it, so the host runs ahead of the GPU
        bld.begin()                                         # empty the table: epoch bump, no HBM traffic
        p = engine.PackedSeqs(d_fasta, lazy=True)           # K1 (3 launches)
        return bld.build_async(p, ev=kev)                   # per round: K2a | (count exchange, K2b,) plan, K3

    # ---- correctness, outside the timed region: the table this configuration builds has the expected checksum
    t = step_device()
    torch.cuda.synchronize()
    bld.verify()
    cs = measure.merged_checksum(t, world)
    used = allsum(t.n_keys())
    want, want_src = golden_checksum(args.workload, k, args.scale)
    checks = {"vs_golden": None if want is None else (list(cs) == list(want)), "golden_source": want_src}
    if world == 1 and len(data) <= 2e8:
        ref_table, _ = engine.build_dbg(packed, k)          # the fused single-launch build must agree
        checks["vs_fused_build"] = (ref_table.checksum() == cs)
        del ref_table
    if any(v is False for v in checks.values()):
        raise SystemExit("bench: the built table has the wrong checksum: %r %r" % (cs, checks))
    if used == 0 and n_ins > 0:
        raise SystemExit("bench: empty table")

    for _ in range(args.warmup):
        step_device()
    torch.cuda.synchronize()
    bld.verify()
    clocks = ClockSampler(local) if rank == 0 else None
    if clocks:
        clocks.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = ev(), ev()
    e0.record(stream)
    for _ in range(args.steps):
        t = step_device()
    e1.record(stream)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clk = clocks.stop() if clocks else None
    bld.verify()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, t, world, rank)     # before the steps below rebuild into the same table
    ms_step = allmax(e0.elapsed_time(e1)) / args.steps
    value = n_ins / (ms_step * 1e-3) / 1e9
    # per-stage times (the roofline entries): the same steps again with CUDA events around every kernel group, outside the
    # headline's timed region - the event records and the host work they cost stay out of `value`
    kev = {}
    n_stage_steps = min(args.steps, 10)
    for _ in range(n_stage_steps):
        t = step_device(kev)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    bld.verify()
    stage_ms = {name: allmax(sum(a.elapsed_time(b) for a, b in pairs) / n_stage_steps) for name, pairs in sorted(kev.items())}
    k3_launch_ms = allmax(sum(a.elapsed_time(b) for a, b in kev["k3"]) / len(kev["k3"]))
    if measure.merged_checksum(t, world) != cs:
        raise SystemExit("bench: table built inside the timed region has the wrong checksum")

    # ---- end to end through the public API, host buffers: every step uploads its own copy of the FASTA bytes from
    # pinned host memory (H2D inside the timed region), builds, and reads the table statistics back (D2H).
    # The upload of step i+1 is issued on a copy stream before step i's result is awaited (double-buffered
    # device input), the way a loader feeds a stream of files; each step still waits for ITS upload.
    copy_stream = torch.cuda.Stream()
    dev_in = [torch.empty_like(d_fasta) for _ in range(2)]
    k1_done = [None, None]

    def upload(i):
        with torch.cuda.stream(copy_stream):
            if k1_done[i % 2] is not None:
                copy_stream.wait_event(k1_done[i % 2])       # K1 of the step that last read this buffer (device-side wait)
            dev_in[i % 2].copy_(host, non_blocking=True)
            done = torch.cuda.Event()
            done.record(copy_stream)
        return done

    def run_e2e(n):
        # Two steps in flight: while step i runs, the host reads step i-1's result (table statistics, D2H into
        # pinned memory) and the copy stream uploads step i+1's input.
        nxt = upload(0)
        st_, pending = None, None
        for i in range(n):
            cur = nxt
            if i + 1 < n:
                nxt = upload(i + 1)
            bld.begin()
            stream.wait_event(cur)
            p = engine.PackedSeqs(dev_in[i % 2], lazy=True)
            k1_done[i % 2] = torch.cuda.Event()
            k1_done[i % 2].record(stream)
            tt = bld.build_async(p)
            fut = tt.stats_async(i)          # D2H of the statistics (distinct keys, overflow / lost flags, short records, ...)
            if pending is not None:
                st_ = pending.wait()
                if int(st_[_lib.PG_STAT_OVERFLOW]) or int(st_[_lib.PG_STAT_LOST]):
                    raise SystemExit("bench: table overflow / lost records inside the e2e loop")
            pending = fut
        return pending.wait()
    run_e2e(2)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    g0, g1 = ev(), ev()
    g0.record(stream)
    st = run_e2e(args.steps)
    g1.record(stream)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    bld.verify()
    if allsum(int(st[_lib.PG_STAT_USED])) != used:
        raise SystemExit("bench: e2e build reports a different number of distinct keys")
    e2e_ms = allmax(g0.elapsed_time(g1)) / args.steps
    e2e_val = n_ins / (e2e_ms * 1e-3) / 1e9

    peak, peak_src = peaks()
    cap = t.capacity
    # K3, the dominant kernel: 16 B per insertion (SURVEY 8d), 2 insertions per record; per launch = per round and rank
    alg_launch = 16.0 * n_ins / world / bld.n_rounds
    achieved = alg_launch / (k3_launch_ms * 1e-3) / 1e9
    sector_launch = 64.0 * (n_ins / 2) / world / bld.n_rounds
    traffic = None
    tp = os.path.join(ROOT, "profiles", "insert_traffic.json")
    if os.path.isfile(tp):
        try:
            with open(tp) as f:
                traffic = json.load(f).get((args.workload + ("_compact" if getattr(bld, "compact", False) else
                                                             ("_region" if getattr(bld, "region_bits", 0) else ""))) if world == 1
                                           else "%s_n%d" % (args.workload, world))
        except Exception:
            traffic = None
    region = bool(getattr(bld, "region_bits", 0))
    rec_b = 8.0 if getattr(bld, "compact", False) else 16.0          # bytes per update record on the streaming stages
    roof = {"kernel": ("k3s_region_build_c" if rec_b == 8.0 else "k3s_region_build") if region else "k3_insert_records", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "peak_source": peak_src, "ms_per_launch": k3_launch_ms, "launches_per_step": bld.n_rounds,
            "algorithmic_bytes_per_launch": alg_launch,
            "convention": "insert: 16 B per insertion (SURVEY 8d), 2 insertions per record, per rank and round" +
                          (" (K3s + spill upserts; what it really moves: %d B/record read + 16 B/slot written = %.0f MB)"
                           % (rec_b, (rec_b / 2 * n_ins / world / bld.n_rounds + 16.0 * cap) / 1e6) if region else ""),
            "sector_convention": {"bytes_per_launch": sector_launch, "achieved": sector_launch / (k3_launch_ms * 1e-3) / 1e9,
                                  "frac": sector_launch / (k3_launch_ms * 1e-3) / 1e9 / peak,
                                  "what": "64 B per record: one 32-byte sector read + written back (SURVEY 8d minimum DRAM traffic)"},
            "other_kernels": {}}
    part_bytes = (0.25 * n_bases + rec_b * (n_ins / 2)) / world / bld.n_rounds
    k2a_ms = allmax(sum(a.elapsed_time(b) for a, b in kev["k2a"]) / len(kev["k2a"]))
    roof["other_kernels"]["k2a_partition"] = {
        "ms_per_launch": k2a_ms, "algorithmic_bytes_per_launch": part_bytes, "achieved": part_bytes / (k2a_ms * 1e-3) / 1e9,
        "frac": part_bytes / (k2a_ms * 1e-3) / 1e9 / peak,
        "convention": "0.25 B/base read + %d B/record written%s" % (rec_b, " (materialised for the exchange)" if world > 1 else "") +
                      (", stored into the owners' receive buffers over NVLink" if world > 1 else "")}
    if "k2c" in kev:
        k2c_ms = allmax(sum(a.elapsed_time(b) for a, b in kev["k2c"]) / len(kev["k2c"]))
        b2 = 2 * rec_b * (n_ins / 2) / world / bld.n_rounds * max(1, len(bld.levels) - 1)
        roof["other_kernels"]["k2c_refine"] = {"ms_per_launch": k2c_ms, "algorithmic_bytes_per_launch": b2, "achieved": b2 / (k2c_ms * 1e-3) / 1e9,
                                               "frac": b2 / (k2c_ms * 1e-3) / 1e9 / peak,
                                               "convention": "%d B/record read + %d B/record written per partition level, %d level(s) (hash-prefix buckets -> one bucket per table region)"
                                                             % (rec_b, rec_b, max(1, len(bld.levels) - 1))}
    if world > 1:
        k2b_ms = allmax(sum(a.elapsed_time(b) for a, b in kev["k2b"]) / len(kev["k2b"]))
        b2 = 2 * rec_b * (n_ins / 2) / world / bld.n_rounds
        roof["other_kernels"]["k2b_split"] = {"ms_per_launch": k2b_ms, "algorithmic_bytes_per_launch": b2, "achieved": b2 / (k2b_ms * 1e-3) / 1e9,
                                              "frac": b2 / (k2b_ms * 1e-3) / 1e9 / peak, "convention": "%d B/record read + %d B/record written" % (rec_b, rec_b)}
    if world == 1 and not args.no_stages and len(data) <= 2e8:
        # the other kernels the north star names, and the random-slot ceiling K3 runs against (outside the timed region)
        try:
            roof["other_kernels"].update(measure.stage_rooflines(packed, t, k, peak))
            n_rec_ops = 1 << 25
            region = max(1, (8 << 20) // 16)
            ceil = {}
            for name, mode in (("load_only", 0), ("load_red_add", 1), ("load_cas128", 2), ("config2_mix", 3), ("config2_mix_with_record_stream", 11)):
                gops, ms_ = measure.slot_ceiling(cap, min(region, cap), n_rec_ops, mode)
                ceil[name] = {"G_ops_per_s": gops, "ms": ms_}
            k3_rate = (n_ins / 2) / bld.n_rounds / (k3_launch_ms * 1e-3) / 1e9
            roof["atomic_ceiling"] = {"what": "pg_microbench_slots: pseudo-random 16-byte slots of the same table, 8 MB regions swept in order, no key arithmetic; "
                                              "2^25 operations, 5 CTAs/SM", "variants": ceil, "k3_G_records_per_s": k3_rate,
                                      "k3_frac_of_mix_ceiling": k3_rate / ceil["config2_mix_with_record_stream"]["G_ops_per_s"]}
        except Exception as e:      # measurement support must never take the headline down
            roof["other_kernels"]["error"] = repr(e)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak" if world == 1 else "strong", "vs_baseline": None,
        "dtype": "int64", "data": "synthetic",
        "config": {"workload": wl, "k": k, "rc": True, "insertions_per_step": n_ins, "bases": n_bases,
                   "input": "one FASTA file of %d bytes; rank r packs the record-aligned byte range [cut_r, cut_r+1)" % file_size if world > 1
                            else "one FASTA file of %d bytes" % file_size,
                   "table_slots_per_gpu": cap, "table_bytes_per_gpu": cap * 16, "distinct_canonical_keys": used,
                   "load_factor": used / (cap * world), "builder": bld.describe(),
                   "l2": "every step writes and re-reads %.2f GB of update records per GPU and randomly updates its %.1f GB table (both >> 126 MB L2), which evicts the input"
                         % (n_ins / 2 * rec_b / world / 1e9, cap * 16 / 1e9)},
        "e2e": {"value": e2e_val, "unit": UNIT, "ms_per_step": e2e_ms, "h2d_bytes_per_step": allsum(int(host.numel())),
                "d2h_bytes_per_step": int(8 * _lib.PG_STAT_WORDS) * world,
                "pipelining": "input i+1 uploads and result i-1 is read while step i runs"},
        "gpu_launches": (3 + bld.launches_per_build) * args.steps * world,
        "clocks": clk,
        "stages_ms": stage_ms,
        "roofline": roof,
        "checksum": list(cs), "checksum_checks": checks,
        "setup_s": {"generate_input": t_gen},
    }
    if world > 1:
        line["exchange"] = ("fused into K2a: records bucketed by owner rank only and stored into the owners' receive buffers over NVLink "
                            "(CUDA IPC peer memory); the only collective on the data path is the all-to-all of %d counts per round" % world)
        sent = bld.sent_total.cpu().tolist()                  # records this rank really stored into every owner's buffer (timed steps)
        away = sum(v for r_, v in enumerate(sent) if r_ != rank)
        line["exchange_bytes_per_gpu_per_step"] = int(allmax(rec_b * away / n_stage_steps))
        # the driver's scaling run mixes workloads (BASELINE quotes the metric on configs[1] at one GPU and configs[3] "hash-sharded at
        # 2/4/8 GPUs"): the strong-scaling base of THIS workload on one GPU is kept in profiles/
        if args.workload == "cfg4":
            try:
                with open(os.path.join(ROOT, "profiles", "r2r_bench_cfg4_n1.json")) as f:
                    b1 = json.load(f)
                line["strong_scaling_base"] = {"n_gpus": 1, "value": b1["value"], "ms_per_step": b1["ms_per_step"], "workload": "cfg4",
                                               "source": "profiles/r2r_bench_cfg4_n1.json (same workload on one GPU, 16-byte records, L2-atomic K3)"}
            except Exception:
                pass
    if world == 1 and not args.no_cpu_baseline:
        r, kind, cores, text = cpu_reference_rate(data, k, 5_000_000)
        line["cpu_baseline"] = {"value": r, "unit": UNIT, "cores": cores, "kind": kind, "sample": text,
                                "host_cpus": os.cpu_count()}
    if rank == 0:
        print(json.dumps(line), flush=True)
    bld.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
