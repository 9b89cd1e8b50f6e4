"""ctypes binding of libpgdbg.so (include/pgdbg.h).  Fails loudly: there is no
CPU fallback anywhere in this package."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libpgdbg.so")

PG_MODE_LITERAL, PG_MODE_LITERAL_RC, PG_MODE_CANONICAL = 0, 1, 2
PG_STAT_OVERFLOW, PG_STAT_SHORT, PG_STAT_USED, PG_STAT_ENTRIES, PG_STAT_LOST, PG_STAT_WORDS = 0, 1, 2, 3, 4, 8
# Markov clustering constants (include/pgdbg.h PG_MCL_*): theta, S, tau, T and the stats block layout
PG_MCL_PRUNE_THETA, PG_MCL_SELECT_S, PG_MCL_CHAOS_TAU, PG_MCL_MAX_ITER = 1e-4, 1024, 1e-4, 100
# BGZF input (include/pgdbg.h): "not BGZF" return code and the member error kinds d_status reports
PG_ERR_NOT_BGZF = -5
PG_INF_ERRORS = {1: "bad header", 2: "truncated deflate data", 3: "invalid block type", 4: "stored block length check",
                 5: "invalid code lengths", 6: "invalid code", 7: "distance too far back", 8: "more output than ISIZE",
                 9: "length mismatch", 10: "CRC-32 mismatch"}
# FASTQ input (include/pgdbg.h PG_FQ_*): the malformed-record kinds pg_fastq_scan_pack's d_status reports
PG_FQ_ERRORS = {1: "header line does not start with '@'", 2: "separator line does not start with '+'",
                3: "quality length differs from sequence length", 4: "truncated record (line count not a multiple of 4)"}
PG_MCL_WARP_PRODUCTS, PG_MCL_SMEM_SLOTS = 64, 2048
PG_MCL_STAT_CHAOS, PG_MCL_STAT_NNZ, PG_MCL_STAT_PRODUCTS, PG_MCL_STAT_MAXPROD, PG_MCL_STAT_LARGE, PG_MCL_STAT_WORDS = 0, 1, 2, 3, 4, 8

c_i64, c_int, c_vp = ctypes.c_int64, ctypes.c_int, ctypes.c_void_p


class PgTable(ctypes.Structure):
    _fields_ = [("d_slots", c_vp), ("capacity", c_i64), ("d_stats", c_vp), ("mode", ctypes.c_int32),
                ("k", ctypes.c_int32), ("epoch", ctypes.c_int32), ("region_bits", ctypes.c_int32),
                ("alloc_capacity", c_i64), ("hash_kind", ctypes.c_int32), ("reserved", ctypes.c_int32)]


PT = ctypes.POINTER(PgTable)


class PgGraph(ctypes.Structure):
    _fields_ = [("d_node_keys", c_vp), ("d_node_parent", c_vp), ("d_node_label", c_vp), ("d_edge_keys", c_vp),
                ("d_edge_w", c_vp), ("d_edge_first", c_vp), ("d_visit_keys", c_vp), ("d_stats", c_vp),
                ("node_cap", c_i64), ("edge_cap", c_i64), ("visit_cap", c_i64)]


GT = ctypes.POINTER(PgGraph)


class PgBucketSet(ctypes.Structure):
    _fields_ = [("d_records", c_vp), ("d_peer_bases", c_vp), ("d_part_counts", c_vp), ("part_cap", c_i64), ("spill_cap", c_i64),
                ("owner_bits", ctypes.c_int32), ("sub_bits", ctypes.c_int32), ("my_rank", ctypes.c_int32), ("reserved", ctypes.c_int32)]


BT = ctypes.POINTER(PgBucketSet)


class PgCBuckets(ctypes.Structure):
    """Compact (8-byte) update records: include/pgdbg.h pg_cbuckets."""
    _fields_ = [("d_records", c_vp), ("d_counts", c_vp), ("part_cap", c_i64), ("bits", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("d_wide", c_vp), ("d_wide_count", c_vp), ("wide_cap", c_i64), ("d_peer_bases", c_vp), ("d_wide_peer_bases", c_vp),
                ("my_rank", ctypes.c_int32), ("reserved2", ctypes.c_int32)]


CT = ctypes.POINTER(PgCBuckets)

# name -> (restype, argtypes); every symbol include/pgdbg.h declares
SIGNATURES = {
    "pg_last_error": (ctypes.c_char_p, []),
    "pg_version": (c_int, []),
    "pg_device_sms": (c_int, []),
    "pg_pack_words": (c_i64, [c_i64]),
    "pg_fasta_workspace_bytes": (c_i64, [c_i64]),
    "pg_fasta_scan_pack": (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp]),
    "pg_fastq_workspace_bytes": (c_i64, [c_i64, c_i64]),
    "pg_fastq_scan_pack": (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "pg_table_bytes": (c_i64, [c_i64]),
    "pg_table_clear": (c_int, [PT, c_vp]),
    "pg_table_reset": (c_int, [PT, c_vp]),
    "pg_kmer_insert": (c_int, [PT, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp]),
    "pg_count_short": (c_int, [PT, c_vp, c_i64, c_i64, c_i64, c_vp]),
    "pg_kmer_partition": (c_int, [PT, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_int, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "pg_peer_alloc": (c_int, [c_i64, ctypes.POINTER(c_vp), ctypes.c_char_p]),
    "pg_peer_open": (c_int, [ctypes.c_char_p, ctypes.POINTER(c_vp)]),
    "pg_peer_close": (c_int, [c_vp]),
    "pg_peer_free": (c_int, [c_vp]),
    "pg_kmer_partition_dev": (c_int, [PT, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_int, c_int, c_vp, c_i64, c_vp, c_vp]),
    "pg_count_short_dev": (c_int, [PT, c_vp, c_vp, c_i64, c_vp]),
    "pg_insert_records": (c_int, [PT, c_vp, c_vp, c_vp, c_int, c_int, c_i64, c_vp]),
    "pg_kmer_partition_to": (c_int, [PT, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_i64, BT, c_vp, c_i64, c_vp, c_vp]),
    "pg_records_split": (c_int, [c_vp, c_vp, c_vp, c_int, c_i64, BT, c_vp, c_vp]),
    "pg_records_refine": (c_int, [BT, c_int, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp]),
    "pg_records_resplit": (c_int, [c_vp, c_vp, c_int, c_i64, c_i64, c_int, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp]),
    "pg_region_build": (c_int, [PT, c_vp, c_vp, c_i64, c_i64, c_int, c_vp]),
    "pg_buckets_plan": (c_int, [BT, c_vp, c_vp, c_vp]),
    "pg_kmer_partition_c": (c_int, [PT, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_i64, CT, c_vp, c_i64, c_vp, c_vp]),
    "pg_records_resplit_c": (c_int, [CT, c_int, CT, c_int, c_vp, c_vp]),
    "pg_region_build_c": (c_int, [PT, CT, c_int, c_int, c_vp]),
    "pg_records_split_c": (c_int, [CT, CT, c_int, c_vp, c_vp]),
    "pg_wide_insert": (c_int, [PT, c_vp, c_vp, c_i64, c_int, c_vp]),
    "pg_microbench_slots": (c_int, [c_vp, c_i64, c_i64, c_i64, c_int, c_int, c_int, c_vp, c_vp, c_vp]),
    "pg_table_count": (c_int, [PT, c_vp]),
    "pg_table_export": (c_int, [PT, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "pg_table_checksum": (c_int, [PT, c_vp, c_vp]),
    "pg_rdbg_count": (c_int, [PT, c_vp, c_vp]),
    "pg_rdbg_select": (c_int, [PT, PT, c_vp]),
    "pg_rdbg_export": (c_int, [PT, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "pg_table_export_raw": (c_int, [PT, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "pg_table_insert_raw": (c_int, [PT, c_vp, c_vp, c_i64, c_vp]),
    "pg_hits_decode": (c_int, [PT, c_vp, c_i64, c_vp, c_vp]),
    "pg_hits_rekey": (c_int, [PT, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "pg_host_write_xyz": (c_int, [ctypes.c_char_p, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64]),
    "pg_host_write_mcl": (c_int, [ctypes.c_char_p, c_vp, c_vp, c_vp, c_i64]),
    "pg_host_bgzf_index": (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp]),
    "pg_bgzf_inflate": (c_int, [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp]),
    "pg_host_oakht_capacity": (c_i64, [c_i64]),
    "pg_host_build_oakht": (c_int, [c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "pg_path_workspace_bytes": (c_i64, [c_i64]),
    "pg_path_hits": (c_int, [PT, c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp,
                             c_i64, c_vp]),
    "pg_graph_clear": (c_int, [GT, c_vp]),
    "pg_graph_add_hits": (c_int, [GT, c_vp, c_vp, c_i64, c_vp, c_int, c_int, c_vp]),
    "pg_graph_components": (c_int, [GT, ctypes.c_uint32, c_vp]),
    "pg_graph_export_edges": (c_int, [GT, PT, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "pg_graph_export_nodes": (c_int, [GT, PT, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "pg_mcl_scan_workspace_bytes": (c_i64, [c_i64]),
    "pg_mcl_slab_slots": (c_i64, [c_i64, c_i64]),
    "pg_mcl_normalise": (c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "pg_mcl_plan": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "pg_mcl_expand": (c_int, [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_i64, ctypes.c_float, c_vp, c_vp, c_vp, c_vp,
                              c_vp, c_i64, c_int, c_vp]),
    "pg_mcl_compact": (c_int, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "pg_mcl_components": (c_int, [c_vp, c_vp, c_i64, c_vp, c_vp]),
    "pg_label_workspace_bytes": (c_i64, [c_i64]),
    "pg_label_regions": (c_int, [GT, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp,
                                 c_i64, c_vp]),
}

_lib = None


class PgError(RuntimeError):
    pass


def load():
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise PgError("libpgdbg.so is missing (%s): build it with `python -m pangenome_b200.build`; "
                          "pangenome_b200 has no CPU fallback" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)      # AttributeError if the library lacks a declared symbol
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def check(rc, what):
    if rc != 0:
        raise PgError("%s failed (%d): %s" % (what, rc, load().pg_last_error().decode(errors="replace")))
