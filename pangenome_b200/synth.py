"""Seeded synthetic genome sets for the configurations BASELINE.json names
(SURVEY.md section 8d).  Pure numpy; used by bench.py and the tests.

All sets: uppercase ACGT only, ``>g{g} synthetic`` headers, 80-column LF lines,
trailing newline.
"""
import struct
import zlib

import numpy as np

_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def fasta_bytes(records, width=80):
    """records: iterable of (header_bytes_without_gt, uint8 ASCII array or bytes)."""
    parts = []
    for hdr, seq in records:
        seq = np.frombuffer(seq, dtype=np.uint8) if isinstance(seq, (bytes, bytearray)) else seq
        n = seq.size
        nfull, rem = divmod(n, width)
        body = np.empty(n + nfull + (1 if rem else 0), dtype=np.uint8)
        if nfull:
            blk = body[:nfull * (width + 1)].reshape(nfull, width + 1)
            blk[:, :width] = seq[:nfull * width].reshape(nfull, width)
            blk[:, width] = 10
        if rem:
            body[nfull * (width + 1):-1] = seq[nfull * width:]
            body[-1] = 10
        parts.append(b">" + hdr + b"\n")
        parts.append(body.tobytes())
    return b"".join(parts)


def _snp_copy(rng, anc, rate):
    s = anc.copy()
    m = rng.random(anc.size) < rate
    s[m] = (s[m] + rng.integers(1, 4, int(m.sum()), dtype=np.uint8)) % 4
    return s


def survey_4x1m():
    """SURVEY.md App. C: 4 x 1 Mbp, 1 % SNP, seed 1234 (4 050 056 bytes)."""
    rng = np.random.default_rng(1234)
    anc = rng.integers(0, 4, 1_000_000, dtype=np.uint8)
    recs = []
    for g in range(4):
        recs.append((b"g%d synthetic" % g, _ACGT[_snp_copy(rng, anc, 0.01)]))
    return fasta_bytes(recs)


def pangenome(n_genomes=10, length=5_000_000, snp=0.01, seed=1):
    """Configs 2/3: ancestor = iid uniform ACGT (seed); genome g = ancestor with
    each site substituted w.p. ``snp`` to a different base (seed 100+g)."""
    anc = np.random.default_rng(seed).integers(0, 4, length, dtype=np.uint8)
    recs = []
    for g in range(n_genomes):
        recs.append((b"g%d synthetic" % g, _ACGT[_snp_copy(np.random.default_rng(100 + g), anc, snp)]))
    return fasta_bytes(recs)


def plant_ancestor(length=500_000_000, seed=2, repeat_frac=0.6, n_families=2000):
    """Ancestor of the "repeat-rich plant-like" sets (configs 4/5): iid ACGT of which ~``repeat_frac`` is overwritten by
    copies of a repeat-family library (family length 200-10 000, copy divergence 5-20 %), plus 0.5 % poly-A /
    microsatellite tracts of 20-60 bases.  uint8 digits 0..3."""
    rng = np.random.default_rng(seed)
    anc = rng.integers(0, 4, length, dtype=np.uint8)
    fam_len = rng.integers(200, min(10_001, max(201, length // 8)), n_families)
    fams = [rng.integers(0, 4, int(l), dtype=np.uint8) for l in fam_len]
    filled = 0
    target = int(length * repeat_frac)
    while filled < target:
        f = fams[int(rng.integers(0, n_families))]
        div = rng.uniform(0.05, 0.20)
        cp = _snp_copy(rng, f, div)
        pos = int(rng.integers(0, max(1, length - cp.size)))
        cp = cp[:length - pos]
        anc[pos:pos + cp.size] = cp
        filled += cp.size
    n_tracts = int(length * 0.005 / 40)
    for _ in range(n_tracts):
        pos = int(rng.integers(0, max(1, length - 64)))
        tl = int(rng.integers(20, 61))
        if rng.random() < 0.5:
            anc[pos:pos + tl] = 0
        else:
            unit = rng.integers(0, 4, int(rng.integers(2, 5)), dtype=np.uint8)
            anc[pos:pos + tl] = np.resize(unit, tl)
    return anc


def _snp_copy_blocked(rng, anc, rate, block=1 << 26):
    """_snp_copy for arrays of hundreds of Mbp: same model, drawn block by block to bound the temporaries."""
    s = anc.copy()
    for a in range(0, anc.size, block):
        v = s[a:a + block]
        m = rng.random(v.size) < rate
        v[m] = (v[m] + rng.integers(1, 4, int(m.sum()), dtype=np.uint8)) % 4
    return s


def plant_genome_records(anc, g, n_chrom=5, genome_seed0=300, snp=0.01):
    """The ``n_chrom`` records of genome ``g``: the ancestor at ``snp`` substitutions per site (seed genome_seed0+g),
    cut into equal chromosomes."""
    s = _ACGT[_snp_copy_blocked(np.random.default_rng(genome_seed0 + g), anc, snp)]
    bounds = np.linspace(0, anc.size, n_chrom + 1).astype(np.int64)
    return [(b"g%d chr%d synthetic" % (g, c + 1), s[bounds[c]:bounds[c + 1]]) for c in range(n_chrom)]


def plant_layout(n_genomes, length, n_chrom=5, width=80):
    """Byte layout of the plant-like FASTA file without generating it: [(genome, chrom, byte offset, byte length)] and
    the file size.  Lets every rank of a multi-GPU run find ITS byte range of the one file (SURVEY 8e) and generate only
    the genomes that fall into it."""
    bounds = np.linspace(0, length, n_chrom + 1).astype(np.int64)
    out, off = [], 0
    for g in range(n_genomes):
        for c in range(n_chrom):
            n = int(bounds[c + 1] - bounds[c])
            size = len(b">g%d chr%d synthetic\n" % (g, c + 1)) + n + (n + width - 1) // width
            out.append((g, c, off, size))
            off += size
    return out, off


def plant_like(n_genomes=8, length=500_000_000, n_chrom=5, seed=2, genome_seed0=300,
               repeat_frac=0.6, n_families=2000, snp=0.01, records=None):
    """Configs 4/5 ("repeat-rich plant-like"): see plant_ancestor; genomes at 1 % SNP; ``n_chrom`` records per genome.
    ``records``: optional (first, end) range of record indices (genome-major) - only those are generated and returned,
    byte-identical to the same records of the whole file."""
    anc = plant_ancestor(length, seed, repeat_frac, n_families)
    first, end = (0, n_genomes * n_chrom) if records is None else records
    recs = []
    for g in range(first // n_chrom, (end + n_chrom - 1) // n_chrom if end > first else first // n_chrom):
        rr = plant_genome_records(anc, g, n_chrom, genome_seed0, snp)
        for c in range(n_chrom):
            if first <= g * n_chrom + c < end:
                recs.append(rr[c])
    return fasta_bytes(recs)


def n_kmer_insertions(seq_lengths, k, rc=True):
    """The metric's unit (BASELINE.md section 3): 2 * sum max(n - k + 1, 1)."""
    tot = sum(max(int(n) - k + 1, 1) for n in seq_lengths)
    return tot * (2 if rc else 1)


# the empty member every BGZF file ends with (SAM/BAM specification 4.1.2)
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf_member(chunk, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    """One BGZF member (gzip header with the BC extra subfield, raw DEFLATE, CRC-32, ISIZE) holding ``chunk``."""
    c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
    d = c.compress(chunk) + c.flush()
    bsize = 12 + 6 + len(d) + 8
    if bsize > 65536:
        raise ValueError("a BGZF member holds at most 65536 bytes: %d input bytes compressed to a %d-byte member" % (len(chunk), bsize))
    return (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", bsize - 1) + d
            + struct.pack("<II", zlib.crc32(chunk), len(chunk)))


def bgzf_bytes(data, block=65280, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    """``data`` as a BGZF file (what ``bgzip`` writes): members of ``block`` input bytes, then the 28-byte EOF member.
    Large inputs are compressed by a thread pool (zlib releases the GIL)."""
    data = bytes(data)
    chunks = [data[i:i + block] for i in range(0, len(data), block)]
    if len(chunks) > 64:
        import os
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(min(32, os.cpu_count() or 1)) as ex:
            members = list(ex.map(lambda c: bgzf_member(c, level, strategy), chunks))
    else:
        members = [bgzf_member(c, level, strategy) for c in chunks]
    return b"".join(members) + BGZF_EOF
