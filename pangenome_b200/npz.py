"""`_db.npz` interop with the reference (SURVEY 8 f1): ``dump`` writes a GPU-built dBG in the
layout of kmer_numba.py's ``dump`` (:243-261) so that ``kmer_numba.py -d`` can load it; ``load``
reads such a file (written by either side) into a GPU table (``load_on_disk`` :289-335).

A device table is written without a host round trip of its entries: the oakht slot arrays are placed on the GPU
(``pg_oakht_place``) and every member is deflated there in independent chunks (``pg_deflate_chunks``), slab by slab,
overlapped with the D2H copy and the file write; ``write_container`` wraps the members in the zip that ``np.load``
reads.  Host entries (``dump_entries``) keep the host placement and ``np.savez_compressed``."""
import ctypes
import io
import struct

import numpy as np

from . import _lib
from ._lib import check


def oakht_image(keys, vals, cnts, offset=0):
    """(parameters, keys[cap], values[cap], counts[cap]) - the arrays the reference saves."""
    L = _lib.load()
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    vals = np.ascontiguousarray(vals, dtype=np.uint16)
    cnts = np.ascontiguousarray(cnts, dtype=np.uint8)
    n = int(keys.size)
    cap = int(L.pg_host_oakht_capacity(n))
    okeys = np.empty(cap, np.uint64)
    ovals = np.empty(cap, np.uint16)
    ocnts = np.empty(cap, np.uint8)
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    check(L.pg_host_build_oakht(P(keys), P(vals), P(cnts), n, cap, P(okeys), P(ovals), P(ocnts)), "pg_host_build_oakht")
    # parameters = [capacity, load_factor * 1e9, size, ksize, vsize, offset]   (:252-258)
    params = np.asarray([cap, int(0.75 * 1e9), n, 1, 1, int(offset)], dtype="uint64")
    return params, okeys, ovals, ocnts


def dump(table, fn, compressed=True, offset=0):
    """Write ``fn`` (``.npz`` appended like the reference does) from a DbgTable: compressed, on the GPU
    (``dump_device``); ``compressed=False``: stored members from the host.  ``offset``: the byte offset a chunk
    checkpoint resumes from (parameters[5], :258)."""
    if not compressed:
        k, v, c = table.export(sort=False)
        return dump_entries(k, v, c, fn, compressed, offset)
    return dump_device(*table.export_device(), fn, offset=offset)


def dump_entries(k, v, c, fn, compressed=True, offset=0):
    """The same from (key, val, count) entries in the reference's convention (e.g. the merged export of a
    hash-partitioned table)."""
    fn = fn[:-4] if fn.endswith(".npz") else fn
    params, okeys, ovals, ocnts = oakht_image(k, v, c, offset)
    (np.savez_compressed if compressed else np.savez)(fn, parameters=params, keys=okeys, values=ovals, counts=ocnts)
    return fn + ".npz"


def load(fn, k, device="cuda", mode=_lib.PG_MODE_LITERAL, min_capacity=0, with_offset=False):
    """Read a reference-layout dBG (or rdBG) file into a literal-key GPU table (``mode``:
    PG_MODE_LITERAL, or PG_MODE_LITERAL_RC when more records will be inserted on both strands).
    ``with_offset``: also return parameters[5], the resume offset of a chunk checkpoint."""
    import torch
    from . import engine
    if mode == _lib.PG_MODE_CANONICAL:
        raise ValueError("a table image holds literal keys: load it as PG_MODE_LITERAL or PG_MODE_LITERAL_RC")
    z = np.load(fn)
    counts = z["counts"]
    live = counts > 0
    keys = z["keys"][live].astype(np.uint64)
    vals = z["values"][live].astype(np.uint64)
    cnts = counts[live].astype(np.uint64)
    sent = keys == np.uint64(0xFFFFFFFFFFFFFFFF)          # the short-record sentinel lives outside the GPU table
    short = int(cnts[sent][0]) if sent.any() else 0
    keys, vals, cnts = keys[~sent], vals[~sent], cnts[~sent]
    t = engine.DbgTable(max(1024, 2 * int(keys.size) + 2, int(min_capacity)), k, mode, device=device)
    if keys.size:
        d_k = torch.from_numpy(keys.view(np.int64)).to(device)
        d_v = torch.from_numpy((vals | (cnts << np.uint64(32))).view(np.int64)).to(device)
        check(t.L.pg_table_insert_raw(ctypes.byref(t.c), engine._ptr(d_k), engine._ptr(d_v), int(keys.size), engine._stream()),
              "pg_table_insert_raw")
    t.stats[_lib.PG_STAT_SHORT] = short
    t.stats[_lib.PG_STAT_USED] = int(keys.size)
    if t.overflowed():
        raise _lib.PgError("table overflow while loading %s" % fn)
    if with_offset:
        return int(z["parameters"][5]), t
    return t


# ---- the device path ---------------------------------------------------------------------------------------------
CHUNK = 32768            # bytes per independently deflated chunk: one stored block at worst, one CTA each
SLAB = 256 << 20         # input bytes per slab: bounds the staging, the compacted output and the pinned copy


def npy_header(dtype, n):
    """The .npy format 1.0 header ``np.save`` writes for a C-ordered 1-D array of ``n`` ``dtype`` values."""
    buf = io.BytesIO()
    np.lib.format.write_array_header_1_0(buf, {"descr": np.lib.format.dtype_to_descr(np.dtype(dtype)),
                                               "fortran_order": False, "shape": (int(n),)})
    return buf.getvalue()


def place_device(keys, vals, cnts):
    """oakht slot arrays of device entries (int64 / int16 / uint8 tensors, distinct keys) on their device: returns
    (cap, okeys, ovals, ocnts) tensors of the same dtypes."""
    import torch
    from . import engine
    L = _lib.load()
    n = int(keys.numel())
    cap = int(L.pg_host_oakht_capacity(n))
    dev = keys.device
    okeys = torch.empty(cap, dtype=torch.int64, device=dev)
    ovals = torch.empty(cap, dtype=torch.int16, device=dev)
    ocnts = torch.empty(cap, dtype=torch.uint8, device=dev)
    ws_bytes = int(L.pg_oakht_place_workspace_bytes(n))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    P = engine._ptr
    check(L.pg_oakht_place(P(keys), P(vals), P(cnts), n, cap, P(okeys), P(ovals), P(ocnts), P(ws), ws_bytes, engine._stream()),
          "pg_oakht_place")
    return cap, okeys, ovals, ocnts


def device_bytes_needed(n, chunk=CHUNK, slab=SLAB):
    """Device bytes ``dump_device`` allocates for ``n`` entries besides the entries themselves: the image, the
    placement work lists and the slab pair of the encoder."""
    L = _lib.load()
    cap = int(L.pg_host_oakht_capacity(int(n)))
    per = max(1, slab // chunk)
    return 11 * cap + int(L.pg_oakht_place_workspace_bytes(int(n))) + 2 * (2 * per * int(L.pg_deflate_slot_bytes(chunk)) + 12 * per)


def deflate_device(hdr, data, write, chunk=CHUNK, slab=SLAB):
    """Stream the raw DEFLATE of ``hdr`` (host bytes) followed by the device tensor ``data`` (its bytes) through
    ``write``, slab by slab: while the host writes slab s, the GPU compresses slab s + 1.  Returns (crc32, size)."""
    import torch
    from . import engine
    L = _lib.load()
    P, S = engine._ptr, engine._stream
    d = data.contiguous().view(torch.uint8).reshape(-1)
    dev = d.device
    total = len(hdr) + int(d.numel())
    n_chunks = max(1, -(-total // chunk))
    per = max(1, min(slab // chunk, n_chunks))
    slot = int(L.pg_deflate_slot_bytes(chunk))
    bufs = [dict(staging=torch.empty(per * slot, dtype=torch.uint8, device=dev),
                 sizes=torch.empty(per + 1, dtype=torch.int64, device=dev),
                 crcs=torch.empty(per, dtype=torch.int32, device=dev),
                 out=torch.empty(per * slot, dtype=torch.uint8, device=dev),
                 host=torch.empty(per * slot, dtype=torch.uint8).pin_memory(),
                 state=torch.empty(2, dtype=torch.int64).pin_memory(),
                 done=torch.cuda.Event(), copied=torch.cuda.Event()) for _ in range(min(2, -(-n_chunks // per)))]
    state = torch.zeros(2, dtype=torch.int64, device=dev)       # running CRC-32 of the member, bytes of the last slab
    slabs = [(c, min(per, n_chunks - c)) for c in range(0, n_chunks, per)]
    dptr = ctypes.c_void_p(d.data_ptr()) if d.numel() else None

    def enqueue(i):
        b = bufs[i % len(bufs)]
        first, m = slabs[i]
        check(L.pg_deflate_chunks(hdr, len(hdr), dptr, int(d.numel()), chunk, first, m, P(b["staging"]), slot, P(b["sizes"]),
                                  P(b["crcs"]), S()), "pg_deflate_chunks")
        check(L.pg_deflate_compact(P(b["staging"]), slot, P(b["sizes"]), P(b["crcs"]), first, m, chunk, total, P(b["out"]),
                                   P(state), S()), "pg_deflate_compact")
        b["state"].copy_(state, non_blocking=True)
        b["done"].record()

    enqueue(0)
    for i in range(len(slabs)):
        b = bufs[i % len(bufs)]
        b["done"].synchronize()
        nbytes = int(b["state"][1])
        b["host"][:nbytes].copy_(b["out"][:nbytes], non_blocking=True)
        b["copied"].record()
        if i + 1 < len(slabs):
            enqueue(i + 1)            # the other buffer: its bytes were written to the file in the previous iteration
        b["copied"].synchronize()
        write(b["host"][:nbytes].numpy())
    return int(bufs[(len(slabs) - 1) % len(bufs)]["state"][0]) & 0xFFFFFFFF, total


def dump_device(keys, vals, cnts, fn, offset=0):
    """``dump`` from device entries (int64 / int16 / uint8 tensors in the reference's convention, distinct keys)."""
    import torch
    fn = fn[:-4] if fn.endswith(".npz") else fn
    n = int(keys.numel())
    cap, okeys, ovals, ocnts = place_device(keys, vals, cnts)
    # parameters = [capacity, load_factor * 1e9, size, ksize, vsize, offset]   (:252-258)
    params = np.asarray([cap, int(0.75 * 1e9), n, 1, 1, int(offset)], dtype="uint64")
    d_params = torch.from_numpy(params.view(np.int64)).to(keys.device)
    members = [("parameters", "<u8", d_params), ("keys", "<u8", okeys), ("values", "<u2", ovals), ("counts", "|u1", ocnts)]
    write_container(fn + ".npz", [(name + ".npy", (lambda w, t=t, dt=dt: deflate_device(npy_header(dt, t.numel()), t, w)))
                                  for name, dt, t in members])
    return fn + ".npz"


# ---- the zip container np.load reads (what np.savez_compressed writes: ZIP_DEFLATED members, zip64 extra fields in
# every local header) ------------------------------------------------------------------------------------------------
_ZIP64_LIMIT = (1 << 31) - 1      # zipfile's threshold for zip64 fields in the central directory and end records
_DOS_DATE = (0 << 9) | (1 << 5) | 1   # 1980-01-01 00:00:00: a fixed time stamp keeps two dumps of one table identical


def _local_header(name, crc, csize, usize):
    extra = struct.pack("<HHQQ", 1, 16, usize, csize)
    return struct.pack("<4s2B4HL2L2H", b"PK\x03\x04", 45, 0, 0, 8, 0, _DOS_DATE, crc, 0xFFFFFFFF, 0xFFFFFFFF,
                       len(name), len(extra)) + name + extra


def write_container(path, members):
    """Write the zip archive ``path`` from ``members``: (name, compress) pairs in order, where ``compress(write)``
    streams the member's raw-DEFLATE bytes through ``write`` and returns (crc32, uncompressed size).  The local header
    is written first and patched once the sizes are known."""
    entries = []
    with open(path, "wb") as f:
        for name, compress in members:
            name_b = name.encode()
            off = f.tell()
            f.write(_local_header(name_b, 0, 0, 0))
            start = f.tell()
            crc, usize = compress(f.write)
            end = f.tell()
            f.seek(off)
            f.write(_local_header(name_b, crc, end - start, usize))
            f.seek(end)
            entries.append((name_b, crc, end - start, usize, off))
        cd_off = f.tell()
        for name_b, crc, csize, usize, off in entries:
            z64, fields = [], [usize, csize, off]
            for i, v in enumerate(fields):
                if v > _ZIP64_LIMIT:
                    z64.append(v)
                    fields[i] = 0xFFFFFFFF
            extra = struct.pack("<HH%dQ" % len(z64), 1, 8 * len(z64), *z64) if z64 else b""
            f.write(struct.pack("<4s4B4HL2L5H2L", b"PK\x01\x02", 45, 3, 45, 0, 0, 8, 0, _DOS_DATE, crc, fields[1], fields[0],
                                len(name_b), len(extra), 0, 0, 0, 0o644 << 16, fields[2]) + name_b + extra)
        cd_end = f.tell()
        cd_size, count = cd_end - cd_off, len(entries)
        if count > 0xFFFF or cd_off > _ZIP64_LIMIT or cd_size > _ZIP64_LIMIT:
            f.write(struct.pack("<4sQ2H2L4Q", b"PK\x06\x06", 44, 45, 45, 0, 0, count, count, cd_size, cd_off))
            f.write(struct.pack("<4sLQL", b"PK\x06\x07", 0, cd_end, 1))
            count, cd_size, cd_off = min(count, 0xFFFF), min(cd_size, 0xFFFFFFFF), min(cd_off, 0xFFFFFFFF)
        f.write(struct.pack("<4s4H2LH", b"PK\x05\x06", 0, 0, count, count, cd_size, cd_off, 0))
