"""Markov clustering (K7m) vs connected components (K7) on config 2 (10 x 5 Mbp, k = 27): graph size, iterations,
nnz / products / time per iteration, total CUDA-event time of both clusterings, cluster and row counts.

    python scratch/mcl_time.py [out.json]
"""
import json
import subprocess
import sys
import os

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from pangenome_b200 import engine, graph  # noqa: E402
from pangenome_b200.synth import pangenome  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return out, a.elapsed_time(b)


def main():
    k = 27
    data = pangenome(10, 5_000_000)
    packed = engine.PackedSeqs(engine.to_device_bytes(data))
    t, _ = engine.build_dbg(packed, k)
    rd = t.select_rdbg()
    base = graph.seq2graph_device(packed, rd, k)                  # also warms K5-K8 up
    g = base.graph
    nodes = len(base.nodes[0])
    edges = len(base.edges[0])
    rep = {"card": card(), "config": "config 2: synth.pangenome(10, 5_000_000), k = 27", "nodes": nodes, "edges": edges}
    # K7: union-find + ordering (components() as the pipeline calls it); warm run first
    g.components(rd)
    cc, ms_cc = timed(lambda: g.components(rd))
    rep["components"] = {"ms": ms_cc, "clusters": g.n_components, "rows": len(base.rows(packed, data))}
    # K7m: warm-up run, then the timed one
    g.mcl(rd)
    mc, ms_mcl = timed(lambda: g.mcl(rd))
    r = g.mcl_result
    res = graph.seq2graph_device(packed, rd, k, cluster="mcl")
    rep["mcl"] = {"ms": ms_mcl, "iterations": r.iterations, "clusters": g.n_components, "rows": len(res.rows(packed, data)),
                  "per_iteration": r.stats, "mcl_clusters_full_run": res.graph.n_components}
    line = json.dumps(rep)
    print(line)
    if len(sys.argv) > 1:
        os.makedirs(os.path.dirname(sys.argv[1]) or ".", exist_ok=True)
        with open(sys.argv[1], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
