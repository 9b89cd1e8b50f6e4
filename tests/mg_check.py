"""Run under torchrun (one rank per GPU): the hash-partitioned build of ONE input file - every rank packs its
record-aligned byte range (pangenome_b200/shard.py) - equals the oracle on the whole file: dBG triples, merged
checksum, rdBG key set, .xyz lines in file order, region rows; then the same through the drop-in CLI.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29533 tests/mg_check.py

With --one-device every rank runs on cuda:0 and the ranks talk over gloo (NCCL refuses two ranks on one device).  The
builder cannot tell: the peer stores go through CUDA IPC between processes of one device, and a gloo collective on CUDA
tensors reads its input after the current stream's work and returns only when every rank's input has arrived, so the
count exchange still orders the peer stores.  This mode also runs the CLI with --cluster mcl against a one-GPU run.
tests/test_gpu_multi_one_device.py starts it without torchrun, with the process group already set up.
"""
import io
import os
import sys
import tempfile

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def files(world):
    from pangenome_b200 import synth
    # A: diverged copies of one ancestor + a short record (sentinel) + a hot key (poly-A: every occurrence reaches one
    #    owner, the count clamps at 255 only after the cross-GPU merge)
    anc = np.random.default_rng(3).integers(0, 4, 60000, dtype=np.uint8)
    recs = [(b"g%d" % g, synth._ACGT[synth._snp_copy(np.random.default_rng(50 + g), anc, 0.02)]) for g in range(3 * max(world, 2))]
    recs += [(b"short", b"ACGT"), (b"polyA", b"A" * 700)]
    yield "diverged+short+polyA", synth.fasta_bytes(recs, width=70), 21
    # B: BASELINE configs 4/5 in miniature: repeat families, poly-A / microsatellite tracts, 5 chromosomes per genome
    yield "plant-like 8 x 300 kb", synth.plant_like(n_genomes=8, length=300_000, n_chrom=5, n_families=50), 27


def main(argv=None):
    argv = sys.argv[1:] if argv is None else argv
    one_device = "--one-device" in argv
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    if one_device:
        os.environ["LOCAL_RANK"] = "0"              # the CLI selects its device from LOCAL_RANK
        torch.cuda.set_device(0)
        if not dist.is_initialized():
            dist.init_process_group("gloo")
    else:
        local = int(os.environ["LOCAL_RANK"])
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from pangenome_b200 import _lib, builder, cli, engine, graph, measure, multigpu, shard
    import oracle
    for name, data, k in files(world):
        cuts = shard.cut_points(data, world)
        mine = data[cuts[rank]:cuts[rank + 1]]
        packed = engine.PackedSeqs(engine.to_device_bytes(mine))
        ref = oracle.run(data, k, stages=1) if rank == 0 else None
        for rounds in (1, 3):
            b = builder.RoundBuilder(k, _lib.PG_MODE_CANONICAL, max(len(mine), 1), world=world, rank=rank, rounds=rounds)
            for it in range(3):                     # repeated builds: buffer parity and the epoch bump carry over
                b.begin()
                if it == 1:                         # device-side bounds, nothing read back between K1 and K3
                    t = b.build_async(engine.PackedSeqs(engine.to_device_bytes(mine), lazy=True))
                else:
                    t = b.build_async(packed, packed.n_rec)
                torch.cuda.synchronize()
                b.verify()
                cs = measure.merged_checksum(t, world)
                if rank == 0:
                    assert cs == oracle.table_checksum(*ref["dbg"]), "merged checksum differs (rounds %d, build %d)" % (rounds, it)
            merged = multigpu.gather_export(t, world, rank)
            if rank == 0:
                ks, vs, cs_ = merged
                assert np.array_equal(ks, ref["dbg"][0]), "keys differ"
                assert np.array_equal(vs, ref["dbg"][1]), "masks differ"
                assert np.array_equal(cs_, ref["dbg"][2]), "counts differ"
                print("mg_check ok: dBG %s, world %d, rounds %d (%d planned), %d entries, max count %d, records: %s" %
                      (name, world, rounds, b.n_rounds, ks.size, int(cs_.max()), b.describe().get("records")), flush=True)
            if rounds == 1:
                # stages 2-5 distributed: rdBG all-gather, hits gathered to rank 0, K6-K8 there
                for c_flag in (2, 3):
                    res, rows = multigpu.seq2graph_distributed(packed, t, k, world, rank, mine, rc=bool(c_flag & 1))
                    if rank == 0:
                        full = oracle.run(data, k, c=c_flag)
                        rk, _ = res.rdbg.rdbg_export()
                        assert np.array_equal(rk, full["rdbg"]), "rdBG differs"
                        assert res.xyz_lines() == full["xyz"], "xyz differs"
                        assert rows == full["rows"], "rows differ"
                        print("mg_check ok: graph %s -c %d: %d rdBG nodes, %d edges, %d rows" %
                              (name, c_flag, rk.size, len(full["xyz"]), len(rows)), flush=True)
            b.close()
        # the drop-in CLI under torchrun: one file on disk, every rank reads its byte range, rank 0 prints the table
        tmp = [None]
        if rank == 0:
            tmp[0] = tempfile.mkdtemp(prefix="pg_mg_")
            with open(os.path.join(tmp[0], "in.fa"), "wb") as f:
                f.write(data)
        dist.broadcast_object_list(tmp, src=0)
        path = os.path.join(tmp[0], "in.fa")
        out = io.StringIO()
        cli.entry_point(["prog", "-m", "-i", path, "-k", str(k), "-n", "2**63"], out=out)
        if rank == 0:
            full = oracle.run(data, k, c=2)
            got = [tuple(l.split("\t")) for l in out.getvalue().splitlines() if not l.startswith("#")]
            want = [(a, str(s), str(e), d, str(l)) for a, s, e, d, l in full["rows"]]
            assert got == want, "CLI rows differ"
            assert open(path + "_rdbg_weight.xyz").read().splitlines() == full["xyz"], "CLI .xyz differs"
            z = np.load(path + "_db.npz")
            assert int(z["parameters"][2]) == ref["dbg"][0].size, "CLI _db.npz entry count differs"
            print("mg_check ok: CLI %s under torchrun: %d rows, %d edges" % (name, len(got), len(full["xyz"])), flush=True)
        if one_device:
            # --cluster mcl: K7m runs on rank 0 over the gathered edges; cluster file and rows equal a one-GPU run
            mpath = os.path.join(tmp[0], "mcl.fa")
            if rank == 0:
                with open(mpath, "wb") as f:
                    f.write(data)
            dist.barrier()
            out = io.StringIO()
            cli.entry_point(["prog", "-i", mpath, "-k", str(k), "--cluster", "mcl", "--no-dump-db"], out=out)
            if rank == 0:
                whole = engine.PackedSeqs(engine.to_device_bytes(data))
                t1, _ = engine.build_dbg(whole, k)
                one = graph.seq2graph_device(whole, t1.select_rdbg(), k, cluster="mcl")
                got = [l for l in out.getvalue().splitlines() if l and not l.startswith("#")]
                assert got == ["%s\t%d\t%d\t%s\t%d" % r for r in one.rows(whole, data)], "CLI --cluster mcl rows differ"
                assert open(mpath + "_rdbg_weight.xyz.mcl").read().split("\n")[:-1] == one.mcl_lines(), "CLI .mcl differs"
                print("mg_check ok: CLI --cluster mcl %s: %d rows, %d clusters" % (name, len(got), len(one.mcl_lines())), flush=True)
        dist.barrier()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
