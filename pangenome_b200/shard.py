"""Splitting ONE input file across the ranks of a multi-GPU run (SURVEY.md 8e): rank r takes the byte range
[cut_r, cut_{r+1}) where cut_r is the first record start ('>' at the beginning of a line) at or after the nominal
offset r * size / world.  Ranges are record-aligned, so every rank packs whole records and the k-mers of a record never
straddle ranks; no communication is needed to agree on the cuts (every rank can compute all of them from the file).
A record larger than size / world is not split (the ranks whose nominal offsets fall inside it get empty ranges).

Host logic only - no CUDA here."""
import mmap
import os


def cut_points_from_starts(starts, size, world):
    """starts: ascending byte offsets of the record starts.  Returns world + 1 cut offsets."""
    import bisect
    cuts = [0]
    for r in range(1, world):
        nominal = r * size // world
        j = bisect.bisect_left(starts, nominal)
        cuts.append(starts[j] if j < len(starts) else size)
    cuts.append(size)
    # the bytes before the first header belong to rank 0 (they are dropped by the reader anyway)
    for i in range(1, len(cuts)):
        cuts[i] = max(cuts[i], cuts[i - 1])
    return cuts


def _first_record_start(buf, size, nominal):
    """First offset >= nominal that holds a '>' at a line start."""
    if nominal <= 0:
        return 0
    j = buf.find(b"\n>", nominal - 1)
    return size if j < 0 else j + 1


def cut_points(buf, world):
    """Cut offsets for a bytes-like / mmap object."""
    size = len(buf)
    cuts = [0] + [_first_record_start(buf, size, r * size // world) for r in range(1, world)] + [size]
    for i in range(1, len(cuts)):
        cuts[i] = max(cuts[i], cuts[i - 1])
    return cuts


def member_rank_range(out_off, world, rank, inflate):
    """The cut rule above applied to the INFLATED stream of a file of independently compressed members (BGZF), reading
    only the members around this rank's range.  ``out_off``: the n + 1 offsets of the members' output in the inflated
    stream (exclusive scan of their sizes); ``inflate(i0, i1)``: the inflated bytes of members [i0, i1).  The search
    starts at the member holding byte nominal_r - 1 and extends in doubling batches of members until the cut after
    nominal_{r+1} is found or the file ends.  Returns what read_rank_range returns, with the inflated size for the
    file size."""
    import bisect
    n, size = len(out_off) - 1, int(out_off[-1])
    if size == 0:
        return b"", (0, 0), 0
    lo, hi = rank * size // world, (rank + 1) * size // world
    first = bisect.bisect_right(out_off, max(lo - 1, 0)) - 1         # the member holding that byte (empty ones skipped)
    base, end, batch = int(out_off[first]), first, 1
    buf = bytearray()

    def grow():
        nonlocal end, batch
        nxt = min(n, end + batch)
        buf.extend(inflate(end, nxt))
        end, batch = nxt, 2 * batch

    def cut(nominal):
        if nominal <= 0:
            return 0
        if nominal >= size:
            return size
        pos = nominal - 1 - base
        while True:
            j = buf.find(b"\n>", pos)
            if j >= 0:
                return base + j + 1
            if end == n:
                return size
            pos = max(pos, len(buf) - 1)
            grow()

    a, b = cut(lo), cut(hi)
    while base + len(buf) < b:         # the last rank's range runs to the end of the file
        grow()
    return bytes(buf[a - base:b - base]), (a, b), size


def plain_rank_range(path, world, rank):
    """read_rank_range of an uncompressed file: only the rank's own pages are read (plus the few a cut search touches)."""
    size = os.path.getsize(path)
    if size == 0:
        return b"", (0, 0), 0
    with open(path, "rb") as f:
        mm = mmap.mmap(f.fileno(), 0, access=mmap.ACCESS_READ)
        try:
            cuts = cut_points(mm, world)
            a, b = cuts[rank], cuts[rank + 1]
            data = mm[a:b]
        finally:
            mm.close()
    return data, (a, b), size


def read_rank_range(path, world, rank):
    """(bytes of this rank's record-aligned range of the decompressed input, (begin, end), decompressed size).  The
    input may be plain FASTA or gzip / BGZF compressed (pangenome_b200/seqfile.py)."""
    from . import seqfile
    return seqfile.read_rank_range(path, world, rank)
