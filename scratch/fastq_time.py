"""FASTQ input on the GPU: pg_fastq_scan_pack time (CUDA events, warmed, repeated, alternated with K1 -
pg_fasta_scan_pack - on the FASTA equivalent of the same reads) and GB/s of input on a 150 bp read set of >= 1 GB (larger
than the 126 MB L2); the pack's share of a one-GPU build of that read set; end-to-end seq2rdbg (file on disk -> dBG table
and its statistics) on the FASTQ and on its FASTA equivalent, alternated, checksums compared.  The card's name and power
limit are read in the same run.

    python scratch/fastq_time.py [out.json] [--reads 3300000]
"""
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from pangenome_b200 import builder, engine, stages, synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def pack_ms(d, fmt, reps):
    """ms per pack of the whole device buffer ``d`` (record index sized to fit, so one launch sequence per pack)"""
    p = engine.PackedSeqs(d, fmt=fmt)                 # warm-up, and the record-index capacity the input needs
    cap = p.cap_records
    for _ in range(2):
        engine.PackedSeqs(d, cap_records=cap, lazy=True, fmt=fmt)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        p._launch(cap)
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / reps, p


def e2e(path, k=27):
    torch.cuda.synchronize()
    t = time.perf_counter()
    h = stages.seq2rdbg(path, k, 5, 2 ** 63, brkpt="", chunk=2 ** 36, rc=True)
    cs = h.table.checksum()
    torch.cuda.synchronize()
    return time.perf_counter() - t, [int(x) for x in cs]


def build_ms(packed, k=27, reps=3):
    """ms of the one-GPU streaming build the CLI runs (builder.build_table) on an already packed input, warmed"""
    builder.build_table(packed, k, rc=True)
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(reps):
        builder.build_table(packed, k, rc=True)
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3 / reps


def main():
    args = sys.argv[1:]
    n_reads = 3_300_000
    if "--reads" in args:
        i = args.index("--reads")
        n_reads = int(args[i + 1])
        del args[i:i + 2]
    out_path = args[0] if args else "fastq_time.json"
    res = {"gpu": card()}
    t = time.perf_counter()
    fq = synth.reads(synth.pangenome(10, 5_000_000), n_reads, length=150)
    fa = synth.fastq_to_fasta(fq)
    r = {"reads": n_reads, "read_length": 150, "fastq_bytes": len(fq), "fasta_bytes": len(fa), "generate_s": time.perf_counter() - t}
    d_fq, d_fa = engine.to_device_bytes(fq), engine.to_device_bytes(fa)
    times = {"fastq_pack_ms": [], "k1_fasta_ms": []}
    for _ in range(3):                                 # alternated
        ms, pq = pack_ms(d_fq, "fastq", 10)
        times["fastq_pack_ms"].append(ms)
        ms, pa = pack_ms(d_fa, "fasta", 10)
        times["k1_fasta_ms"].append(ms)
    r.update(times)
    q_ms, a_ms = min(times["fastq_pack_ms"]), min(times["k1_fasta_ms"])
    r["fastq_pack_GBps_in"] = len(fq) / q_ms / 1e6
    r["k1_fasta_GBps_in"] = len(fa) / a_ms / 1e6
    r["pack_outputs_equal"] = bool(pq.n_rec == pa.n_rec == n_reads and pq.n_bases == pa.n_bases
                                   and (pq.seq_off == pa.seq_off).all()
                                   and torch.equal(pq.pk2[:pq.n_bases // 16], pa.pk2[:pa.n_bases // 16])
                                   and torch.equal(pq.amb[:pq.n_bases // 32], pa.amb[:pa.n_bases // 32]))
    b_ms = build_ms(pq)
    r["build_ms_after_pack"] = b_ms
    r["fastq_pack_share_of_pack_plus_build"] = q_ms / (q_ms + b_ms)
    r["k1_share_of_pack_plus_build_fasta"] = a_ms / (a_ms + b_ms)
    del d_fq, d_fa, pq, pa
    torch.cuda.empty_cache()
    tmp = tempfile.mkdtemp(prefix="pg_fastq_time_")
    pq_path, pa_path = os.path.join(tmp, "r.fq"), os.path.join(tmp, "r.fa")
    open(pq_path, "wb").write(fq)
    open(pa_path, "wb").write(fa)
    e2e(pq_path), e2e(pa_path)                         # warm-up
    et, sums = {"fastq": [], "fasta": []}, {}
    for _ in range(3):
        for key, p in (("fastq", pq_path), ("fasta", pa_path)):
            s, cs = e2e(p)
            et[key].append(s)
            sums[key] = cs
    r["e2e_seq2rdbg_s"] = et
    r["e2e_checksums_equal"] = sums["fastq"] == sums["fasta"]
    r["e2e_checksum"] = sums["fastq"]
    os.remove(pq_path)
    os.remove(pa_path)
    res["reads150"] = r
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
