"""Drop-in command line of kmer_numba.py (entry_point, kmer_numba.py:1971-2144).

    python kmer_b200.py -m -i input.fasta -k 27 > result.tab

Same flags (``-i -k -n -c -r -d -R -D``; ``-k27`` and ``-k 27`` forms; unknown
flags such as ``-m`` are skipped exactly like upstream, F1), same ``# `` banner
lines, same table rows, same side-file names.  ``-d`` / ``-D`` read tables in the
reference's ``.npz`` layout; like upstream the dBG is saved to ``<input>_db.npz`` after stage 1
(``--no-dump-db`` skips the file, the banners stay).  Extra long options (ignored by the reference's
parser, so scripts stay portable): ``--min-edge-weight W``, ``--no-mcl-file``, ``--no-dump-db``, and
``--cluster {components,mcl}`` with ``--inflation R``: the region labels come from the connected components of the
edge list (the default) or from Markov clustering on the GPU with inflation R (default 1.5, what the reference passes
to ``mcl -I``; R > 1) in place of the reference's external ``mcl`` run.  An existing ``<xyz>.mcl`` still wins.

Input: plain FASTA or FASTQ, or either compressed by ``bgzip`` (BGZF: its members are inflated on the GPU) or by ``gzip``
(inflated on the host).  Side files keep the name given with ``-i`` (``input.fa.gz_rdbg_weight.xyz``, ``input.fa.gz_db.npz``);
``-r`` checkpoint offsets are positions in the decompressed stream.  A FASTQ file (first byte '@'; four-line records)
gives exactly what the FASTA of its header and sequence lines gives; quality lines are checked for length only.  A
malformed FASTQ exits naming the byte offset of its first bad record.  ``-r`` takes FASTA only.

Multi-GPU: ``torchrun --nproc-per-node N kmer_b200.py -i input.fasta -k 27`` - every rank packs its
record-aligned byte range of the one input file, the dBG is hash-partitioned across the GPUs
(pangenome_b200/builder.py), rank 0 prints the table and writes the side files.
"""
import sys
from time import time


def manual_print(out=sys.stdout):
    w = lambda s: print(s, file=out)
    w('Usage:')
    w('  pyhton this.py -i qry.fsa -k 10 -n 1000000')
    w('Parameters:')
    w('  -i: query sequences in fasta format')
    w('  -k: kmer length')
    w('  -d: the de bruijn graph')
    w('  -r: break point of de bruijn graph')
    w('  -D: the reduced de bruijn graph')
    w('  -R: break point of reduced de bruijn graph')
    w('  -n: length of query sequences for pan-genomic analysis')
    w('  -c: complementary reverse sequence. 00,01,10,11')


def parse_args(argv):
    args = {'-i': '', '-k': '50', '-n': '2**63', '-r': '', '-d': '', '-R': '', '-D': '', '-c': '2'}
    extra = {'--min-edge-weight': '1', '--cluster': 'components', '--inflation': '1.5'}
    flags = set()
    N = len(argv)
    for i in range(1, N):
        k = argv[i]
        if k in args:
            args[k] = argv[i + 1] if i + 1 < N else ''
        elif k in extra:
            extra[k] = argv[i + 1] if i + 1 < N else extra[k]
        elif k[:2] in args and len(k) > 2 and not k.startswith('--'):
            args[k[:2]] = k[2:]
        elif k.startswith('--'):
            flags.add(k)
    return args, extra, flags


def cluster_options(extra):
    """(method, inflation) from ``--cluster`` / ``--inflation``; a bad value exits with a message."""
    method = extra['--cluster']
    if method not in ('components', 'mcl'):
        raise SystemExit("pangenome_b200: --cluster must be 'components' or 'mcl', got %r" % method)
    try:
        r = float(extra['--inflation'])
    except ValueError:
        raise SystemExit("pangenome_b200: --inflation needs a number, got %r" % extra['--inflation'])
    if not 1.0 < r < 64.0:
        raise SystemExit("pangenome_b200: --inflation must be greater than 1 (and below 64), got %r" % extra['--inflation'])
    return method, r


def _eval_n(text):
    # the reference eval()s -n ('2**63', '5e8'); accept the same arithmetic without eval
    import ast
    import operator as op
    ops = {ast.Add: op.add, ast.Sub: op.sub, ast.Mult: op.mul, ast.Pow: op.pow, ast.Div: op.truediv, ast.FloorDiv: op.floordiv}

    def ev(n):
        if isinstance(n, ast.Constant) and isinstance(n.value, (int, float)):
            return n.value
        if isinstance(n, ast.BinOp) and type(n.op) in ops:
            return ops[type(n.op)](ev(n.left), ev(n.right))
        if isinstance(n, ast.UnaryOp) and isinstance(n.op, ast.USub):
            return -ev(n.operand)
        raise ValueError("unsupported -n expression: %r" % text)
    return int(ev(ast.parse(text, mode="eval").body))


CHUNK = 2 ** 33      # bases (both strands counted) between dBG checkpoints, kmer_numba.py entry_point


def _init_distributed():
    """Under torchrun (WORLD_SIZE > 1): one process per GPU, NCCL.  Returns (world, rank)."""
    import os
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world <= 1:
        return 1, 0
    import torch
    import torch.distributed as dist
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return dist.get_world_size(), dist.get_rank()


def entry_point(argv, out=sys.stdout):
    args, extra, flags = parse_args(argv)
    qry, kmer, Ns, rc = args['-i'], int(args['-k']), _eval_n(args['-n']), int(args['-c'])
    if not qry:
        manual_print(out)
        raise SystemExit()
    method, inflation = cluster_options(extra)
    if args['-R']:
        raise SystemExit("pangenome_b200: -R (resuming the edge-weight stage from a _rdb_brkpt.npz) is not supported by the "
                         "GPU path; -r (dBG checkpoint) is")
    world, rank = _init_distributed()
    from . import stages
    if args['-r'] and stages.seq_chk(qry) == "fastq":
        raise SystemExit("pangenome_b200: -r (dBG checkpoint resume) reads FASTA only; %s is FASTQ" % qry)
    p = (lambda *a: print(*a, file=out)) if rank == 0 else (lambda *a: None)      # rank 0 owns stdout and the side files
    dbs, rdb = args['-d'], args['-D']
    if world > 1 and (dbs or rdb or args['-r']):
        raise SystemExit("pangenome_b200: -d / -D / -r start from a saved table and run on one GPU; launch without torchrun")
    rc1 = ((rc & 1) == 1)
    if dbs or rdb:
        # kmer_numba.py:2072-2100: start from a dBG (-d) or rdBG (-D) table saved in the reference's .npz layout
        if not rdb:
            p('load dBG from disk')
            p('# build the reduced dBG')
        kmer_dict = stages.load_dbg(qry, dbs or rdb, kmer)
        rdbg_dict = stages.dbg2rdbg(kmer_dict)      # an rdBG file only holds members: selecting again keeps all of them
        del kmer_dict
        p('# find fr')
        stages.seq2graph(qry, kmer=kmer, bits=5, Ns=Ns, rdbg_dict=rdbg_dict, rc=rc1, out=out,
                         min_weight=int(extra['--min-edge-weight']), write_mcl='--no-mcl-file' not in flags,
                         cluster_method=method, inflation=inflation)
        return 0
    p('# build the dBG')
    st = time()
    rc0 = ((rc >> 1) == 1)
    kmer_dict = stages.seq2rdbg(qry, kmer, 5, Ns, brkpt=args['-r'], chunk=CHUNK, rc=rc0)    # :2111
    p('# finished in', time() - st, 'seconds')
    # the reference dumps the table to <qry>_db.npz and reloads it here (:2116-2126).  The file is written like upstream
    # (kmer_numba.py -d reads it); the reload is skipped - the GPU table stays resident - but its banner is kept so the
    # stdout of the two programs differs in the timing figures only
    p('# save dBG to disk')
    st = time()
    if '--no-dump-db' not in flags:
        stages.dump(kmer_dict, qry + '_db')
    p('# finished in', time() - st, 'seconds')
    p('# load dBG from disk')
    p('# finished in', 0.0, 'seconds')
    p('# build the reduced dBG')
    st = time()
    rdbg_dict = stages.dbg2rdbg(kmer_dict)
    del kmer_dict
    p('# finished in', time() - st, 'seconds')
    p('# find fr')
    st = time()
    rc1 = ((rc & 1) == 1)
    stages.seq2graph(qry, kmer=kmer, bits=5, Ns=Ns, rdbg_dict=rdbg_dict, rc=rc1, out=out,
                     min_weight=int(extra['--min-edge-weight']), write_mcl='--no-mcl-file' not in flags,
                     cluster_method=method, inflation=inflation)
    p('# finished in', time() - st, 'seconds')
    return 0


def main():
    entry_point(sys.argv)
