"""BGZF input on the GPU: pg_bgzf_inflate kernel time (CUDA events, warmed, repeated) and GB/s of inflated output on
config 2 (10 x 5 Mbp, 50 MB) and on a plant-like set of >= 1 GB (bench.workload("cfg4", scale)); end-to-end seq2rdbg
(file on disk -> dBG table and its statistics) on the plain file and on its BGZF form, alternated, checksums compared;
the host's zlib inflate of the same members on one core, for scale.  The card's name and power limit are read in the
same run.

    python scratch/bgzf_time.py [out.json] [--scale 0.3]
"""
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from pangenome_b200 import _lib, engine, seqfile, stages, synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def kernel_time(gz, reps=10):
    """ms per pg_bgzf_inflate launch over the whole file (compressed bytes already on the device)"""
    buf = np.frombuffer(gz, dtype=np.uint8)
    member_off, out_off = seqfile.bgzf_index(buf)
    n = len(member_off) - 1
    L = _lib.load()
    d_gz = engine.to_device_bytes(buf)
    d_offs = torch.from_numpy(np.concatenate([member_off, out_off]).astype(np.int64)).cuda()
    out = torch.empty(int(out_off[-1]), dtype=torch.uint8, device="cuda")
    status = torch.empty(2, dtype=torch.int64, device="cuda")
    P = engine._ptr

    def launch():
        _lib.check(L.pg_bgzf_inflate(P(d_gz), len(gz), P(d_offs), P(d_offs[n + 1:]), n, P(out), int(out.numel()), P(status),
                                     engine._stream()), "pg_bgzf_inflate")
    for _ in range(2):
        launch()
    torch.cuda.synchronize()
    assert status[0].item() == 0
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        launch()
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / reps
    return out, ms, n


def host_inflate_s(gz):
    buf = np.frombuffer(gz, dtype=np.uint8)
    member_off, _ = seqfile.bgzf_index(buf)
    t = time.perf_counter()
    for i in range(len(member_off) - 1):
        zlib.decompress(gz[int(member_off[i]) + 18:int(member_off[i + 1]) - 8], wbits=-15)
    return time.perf_counter() - t


def e2e(path, k=27):
    torch.cuda.synchronize()
    t = time.perf_counter()
    h = stages.seq2rdbg(path, k, 5, 2 ** 63, brkpt="", chunk=2 ** 36, rc=True)
    cs = h.table.checksum()
    torch.cuda.synchronize()
    return time.perf_counter() - t, [int(x) for x in cs]


def main():
    args = sys.argv[1:]
    scale = 0.3
    if "--scale" in args:
        i = args.index("--scale")
        scale = float(args[i + 1])
        del args[i:i + 2]
    out_path = args[0] if args else "bgzf_time.json"
    res = {"gpu": card()}
    sets = [("cfg2", bench.workload("cfg2")[0]), ("cfg4_x%g" % scale, bench.workload("cfg4", scale=scale)[0])]
    tmp = tempfile.mkdtemp(prefix="pg_bgzf_time_")
    for name, data in sets:
        t = time.perf_counter()
        gz = synth.bgzf_bytes(data)
        r = {"bytes": len(data), "bgzf_bytes": len(gz), "ratio": len(gz) / len(data), "compress_s_threads": time.perf_counter() - t}
        d, ms, n = kernel_time(gz)
        r.update(members=n, kernel_ms=ms, kernel_GBps_out=len(data) / ms / 1e6)
        r["gpu_output_equal"] = bool(torch.equal(d, torch.from_numpy(np.frombuffer(data, dtype=np.uint8).copy()).cuda()))
        del d
        r["host_zlib_one_core_s"] = host_inflate_s(gz)
        r["host_zlib_one_core_GBps_out"] = len(data) / r["host_zlib_one_core_s"] / 1e9
        if name == "cfg2":
            plain, comp = os.path.join(tmp, "c.fa"), os.path.join(tmp, "c.fa.gz")
            open(plain, "wb").write(data)
            open(comp, "wb").write(gz)
            e2e(plain), e2e(comp)                          # warm-up
            times = {"plain": [], "bgzf": []}
            sums = {}
            for _ in range(3):
                for key, p in (("plain", plain), ("bgzf", comp)):
                    s, cs = e2e(p)
                    times[key].append(s)
                    sums[key] = cs
            r["e2e_seq2rdbg_s"] = times
            r["e2e_checksums_equal"] = sums["plain"] == sums["bgzf"]
            os.remove(plain)
            os.remove(comp)
        res[name] = r
        print(name, json.dumps(r), flush=True)
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
