"""Reading the input sequence file.  The one place that knows about input formats: it looks at the first bytes and
hands the rest of the package the DECOMPRESSED FASTA or FASTQ stream (``detect`` tells which), on the device for K1 (``engine.PackedSeqs``) and on the
host for what reads header text and byte offsets (``graph.record_ids``, the chunked build and its checkpoints).

- plain FASTA: the file is mapped (np.memmap) and copied to the device as it is;
- BGZF (``bgzip``; gzip members of at most 64 KiB, each an independent DEFLATE stream whose sizes are in its header
  and trailer): the member headers are indexed on the host (pg_host_bgzf_index), the COMPRESSED bytes are copied to the
  device and all members are inflated in one launch (pg_bgzf_inflate) into the buffer K1 reads; the host copy is one
  device-to-host copy of that buffer into pinned memory;
- any other gzip file (one member from ``gzip``, or several): inflated on the host by zlib.  A single DEFLATE stream
  cannot be split among threads - where a block starts is known only once the previous one is decoded - so this
  format gets no GPU path.

Offsets everywhere (the multi-GPU cut points, ``-r`` checkpoint offsets, header offsets) are positions in the
decompressed stream.
"""
import os

import numpy as np

from . import _lib, shard

GZIP_MAGIC = b"\x1f\x8b"


def detect(first):
    """Format of a decompressed stream from its first bytes (``head``): "fastq" when the first byte is '@', "fasta" when
    it is '>' or a line starts with '>' (the reference's seq_chk, kmer_numba.py:873-886), then "fastq" when a line starts
    with '@'; None otherwise.  A FASTQ file whose quality line starts with '>' is still FASTQ."""
    first = bytes(first)
    if first[:1] == b"@":
        return "fastq"
    if first[:1] == b">" or b"\n>" in first:
        return "fasta"
    if b"\n@" in first:
        return "fastq"
    return None


def input_format(path):
    """detect() of the first 40 bytes of the decompressed input."""
    return detect(head(path, 40))


def _map(path):
    """The whole file as a read-only uint8 view of its page-cache pages (nothing is copied on the host)."""
    if os.path.getsize(path) == 0:
        return np.zeros(0, dtype=np.uint8)
    return np.memmap(path, dtype=np.uint8, mode="r")


def bgzf_index(buf):
    """(member_off, out_off), n + 1 int64 offsets each (compressed, inflated), of the BGZF file image ``buf`` (uint8
    array); None when ``buf`` does not start with a BGZF member.  A damaged member raises PgError."""
    import ctypes
    L = _lib.load()
    nbytes = int(buf.size)
    ptr = buf.ctypes.data_as(ctypes.c_void_p) if nbytes else None
    cap = max(16, nbytes // 65536 + 2)             # members of a bgzip file: one per 64 KiB, but any size is valid
    while True:
        moff = np.empty(cap + 1, dtype=np.int64)
        ooff = np.empty(cap + 1, dtype=np.int64)
        counts = np.zeros(2, dtype=np.int64)
        rc = L.pg_host_bgzf_index(ptr, nbytes, moff.ctypes.data_as(ctypes.c_void_p), ooff.ctypes.data_as(ctypes.c_void_p),
                                  cap, counts.ctypes.data_as(ctypes.c_void_p))
        if rc == _lib.PG_ERR_NOT_BGZF:
            return None
        _lib.check(rc, "pg_host_bgzf_index")
        n = int(counts[0])
        if n <= cap:
            return moff[:n + 1], ooff[:n + 1]
        cap = n


def inflate_members(buf, member_off, out_off, i0, i1):
    """Members [i0, i1) of the BGZF image ``buf`` inflated on the GPU: a uint8 CUDA tensor of out_off[i1] - out_off[i0]
    bytes.  Only those members' compressed bytes are copied to the device.  A member that fails to decode raises
    PgError naming its file offset; nothing of the output is returned then."""
    import torch
    from . import engine
    engine._require_cuda()
    L = _lib.load()
    g0, g1 = int(member_off[i0]), int(member_off[i1])
    n = i1 - i0
    out = torch.empty(int(out_off[i1] - out_off[i0]), dtype=torch.uint8, device="cuda")
    if n == 0:
        return out
    d_gz = engine.to_device_bytes(buf[g0:g1])
    offs = np.concatenate([member_off[i0:i1 + 1] - g0, out_off[i0:i1 + 1] - out_off[i0]]).astype(np.int64)
    d_offs = torch.from_numpy(offs).to("cuda")
    status = torch.empty(2, dtype=torch.int64, device="cuda")
    P = engine._ptr
    _lib.check(L.pg_bgzf_inflate(P(d_gz), g1 - g0, P(d_offs), P(d_offs[n + 1:]), n, P(out), int(out.numel()), P(status),
                                 engine._stream()), "pg_bgzf_inflate")
    failed, first = status.cpu().tolist()          # synchronises
    if failed:
        m, kind = i0 + (first >> 8), first & 255
        raise _lib.PgError("BGZF member %d at byte %d of the file failed to inflate: %s (%d member(s) failed)"
                           % (m, int(member_off[m]), _lib.PG_INF_ERRORS.get(kind, "error %d" % kind), failed))
    return out


def _to_host(d):
    """One device-to-host copy into pinned memory, as a uint8 numpy array."""
    import torch
    h = torch.empty(d.numel(), dtype=torch.uint8, pin_memory=True)
    h.copy_(d)
    return h.numpy()


def _kind(buf):
    if bytes(buf[:2]) != GZIP_MAGIC:
        return "plain", None
    idx = bgzf_index(buf)
    return ("bgzf", idx) if idx is not None else ("gzip", None)


def load(path):
    """(host bytes, device bytes) of the whole decompressed input: a uint8 numpy array (np.memmap for plain FASTA) and
    the 16-byte aligned uint8 CUDA tensor K1 packs."""
    from . import engine
    buf = _map(path)
    kind, idx = _kind(buf)
    if kind == "plain":
        return buf, engine.to_device_bytes(buf)
    if kind == "gzip":
        data = np.frombuffer(_gunzip(buf), dtype=np.uint8)
        return data, engine.to_device_bytes(data)
    member_off, out_off = idx
    d = inflate_members(buf, member_off, out_off, 0, len(member_off) - 1)
    return _to_host(d), d


def _gunzip(buf):
    """A (multi-member) gzip file inflated on the host."""
    import gzip
    return gzip.decompress(buf.tobytes())


def read_rank_range(path, world, rank):
    """This rank's record-aligned range of the decompressed input (shard.py's cut rule for its format): (bytes, (begin, end),
    decompressed size).  BGZF: only the members around the range are inflated (shard.member_rank_range), on the GPU."""
    buf = _map(path)
    kind, idx = _kind(buf)
    fmt = input_format(path)
    if kind == "plain":
        return shard.plain_rank_range(path, world, rank, fmt)
    if kind == "gzip":
        raw = _gunzip(buf)
        cuts = shard.cut_points(raw, world, fmt)
        return raw[cuts[rank]:cuts[rank + 1]], (cuts[rank], cuts[rank + 1]), len(raw)
    member_off, out_off = idx
    return shard.member_rank_range(out_off, world, rank,
                                   lambda i0, i1: inflate_members(buf, member_off, out_off, i0, i1).cpu().numpy().tobytes(), fmt)


def head(path, n=40):
    """The first ``n`` bytes of the decompressed input (what seq_chk peeks at)."""
    with open(path, "rb") as f:
        first = f.read(max(n, 2))
    if first[:2] != GZIP_MAGIC:
        return first[:n]
    buf = _map(path)
    idx = bgzf_index(buf)
    if idx is None:
        import gzip
        with gzip.open(path, "rb") as g:
            return g.read(n)
    member_off, out_off = idx
    m = min(int(np.searchsorted(out_off, n, side="left")), len(out_off) - 1)      # members covering the first n bytes
    return inflate_members(buf, member_off, out_off, 0, m).cpu().numpy().tobytes()[:n]
