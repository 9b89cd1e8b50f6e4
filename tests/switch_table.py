"""Every PG_* environment switch of the package, what it selects, and the profiles that run it against the oracle.

The switches choose between compiled variants of the hot-path kernels (DESIGN §4).  The C++ ones are read once per
process into a ``static``, so tests/test_gpu_switches.py starts tests/switch_child.py once per profile with the
profile's environment; the Python ones are read per call and are tested in-process.  tests/test_switch_inventory.py
checks that this table names every switch the sources read, and nothing else.

Kernel names are normalised by ``norm_kernel``: ``k2a_partition_c<256,false,27,3,false>``.  Patterns are fnmatch
patterns over normalised names.

Imports numpy only: the inventory test runs without a GPU, and the child imports torch after it has read this."""
import fnmatch
import re

import numpy as np

# ---------------------------------------------------------------------------------------------------------------------
# kernel names

_KERNEL = re.compile(r"(k[0-9a-z_]*)(<.*?>)?\(")


def norm_kernel(name):
    """``void <unnamed>::k2a_partition_c<(int)256, (bool)0, ...>(<unnamed>::CPartArgs)`` (cu++filt) and
    ``void (anonymous namespace)::k2a_partition_c<256, false, ...>(...)`` (CUPTI) -> ``k2a_partition_c<256,false,...>``;
    None for a name that is not one of this project's kernels (k* in an anonymous namespace)."""
    name = name.strip().replace("(anonymous namespace)::", "").replace("<unnamed>::", "")
    m = _KERNEL.match(re.sub(r"^void ", "", name))
    if not m:
        return None
    base, targs = m.groups()
    if not targs:
        return base
    args = [{"(bool)0": "false", "(bool)1": "true"}.get(a.strip(), a.strip()) for a in targs[1:-1].split(",")]
    return "%s<%s>" % (base, ",".join(re.sub(r"^\(\w[\w ]*\)", "", a) for a in args))


def matches(names, pattern):
    return [n for n in names if fnmatch.fnmatchcase(n, pattern)]


def expand(pattern):
    """``a<{x|y},1>`` -> [``a<x,1>``, ``a<y,1>``]: every alternative must be launched"""
    m = re.search(r"\{([^{}]*)\}", pattern)
    if not m:
        return [pattern]
    out = []
    for alt in m.group(1).split("|"):
        out += expand(pattern[:m.start()] + alt + pattern[m.end():])
    return out


# ---------------------------------------------------------------------------------------------------------------------
# the switches.  launches / replaces: kernel patterns ({a|b}: each alternative); the profiles below carry them.

SWITCHES = {
    # K1 (fasta_pack.cu)
    "PG_K1_SINGLE_PASS": dict(values=["1"], launches=["k1_fused_pack"], replaces=["k1x_tile_aggs", "k1x_scan", "k1x_pack"]),
    "PG_K1_LEGACY": dict(values=["1"], launches=["k1_tile_summaries", "k1_tile_scan", "k1_tile_pack"],
                         replaces=["k1x_tile_aggs", "k1x_scan", "k1x_pack"]),
    "PG_K1_GRID": dict(values=["1"], launches=["k1x_tile_aggs", "k1x_pack"], replaces=[],
                       note="the same kernels on a grid of 148 CTAs: every CTA loops over several 16 KB tiles"),
    # K2a-c / K2c-c / K3s-c (compact_build.cu)
    "PG_K2AC_GENERIC": dict(values=["1"], launches=["k2a_partition_c<256,{false|true},0,3,false>"],
                            replaces=["k2a_partition_c<256,*,27,*,false>", "k2a_partition_c<256,*,21,*,false>"]),
    "PG_K2AC_CTAS": dict(values=["4"], launches=["k2a_partition_c<256,false,{27|21},4,false>"],
                         replaces=["k2a_partition_c<256,false,27,3,false>", "k2a_partition_c<256,false,21,3,false>"]),
    "PG_SPLITC_THREADS": dict(values=["256", "512", "1024"], launches=["k2c_multisplit_c<T,true>"], replaces=["k2c_multisplit_c<other T,true>"]),
    "PG_K3SC_CFG": dict(values=["2"], launches=["k3s_region_build_c<{true|false},{true|false},1024,2,*>"],
                        replaces=["k3s_region_build_c<*,*,512,4,*>"]),
    "PG_K3SC_FP": dict(values=["1"], launches=["k3s_region_build_c<{true|false},{true|false},*,*,true>"],
                       replaces=["k3s_region_build_c<*,*,*,*,false>"]),
    # K2a / K2b / K2c / K3s / K3 on 16-byte records (partition.cu, region_build.cu, multisplit.cu)
    "PG_K2A_THREADS": dict(values=["128", "512"], launches=["k2a_partition<{0|1|2},128,{false|true}>", "k2a_partition<{0|2},512,{false|true}>"],
                           replaces=["k2a_partition<*,256,*>"], note="512 refuses PG_MODE_LITERAL_RC with a pg_fail"),
    "PG_SPLIT_THREADS": dict(values=["256", "512", "1024"], launches=["k2x_multisplit<T>"], replaces=["k2x_multisplit<other T>"]),
    "PG_SPLIT_V1": dict(values=["1"], launches=["k2b_split<*>", "k2c_refine<256>"], replaces=["k2x_multisplit<*>"]),
    "PG_K2B_THREADS": dict(values=["256", "512"], launches=["k2b_split<T>"], replaces=["k2b_split<other T>"], note="only with PG_SPLIT_V1=1"),
    "PG_K3S_THREADS": dict(values=["256"], launches=["k3s_region_build<{8|12},{true|false},256,4>"], replaces=["k3s_region_build<*,*,512,2>"]),
    "PG_K3_GRID": dict(values=["8", "4", "5", "6"], launches=["k3_insert_records<8,*>", "k3_insert_ahead<{4|5|6}>"],
                       replaces=["k3_insert_records<6,true>"]),
    "PG_K3_ROTATE": dict(values=["0"], launches=["k3_insert_records<{6|8},false>"], replaces=["k3_insert_records<*,true>"]),
    "PG_K3_AHEAD": dict(values=["1"], launches=["k3_insert_ahead<{4|5|6}>"], replaces=["k3_insert_records<*>"]),
    # dbg_table.cu, engine.py
    "PG_CLEAR_CTAS_PER_SM": dict(values=["1"], launches=["k_table_clear"], replaces=[],
                                 note="the same kernel on 148 CTAs: a table of more than 148 x 256 slots takes several passes"),
    "PG_TABLE_LOAD": dict(values=["0.9"], launches=["k2_kmer_insert<*>"], replaces=[], note="read at import of engine.py"),
    # inert / not run
    "PG_SPLIT_POLICY": dict(values=["1"], inert="multisplit.cu stores it in PgMultiSplit::policy and no kernel reads that field"),
    "PG_L2_FETCH": dict(not_run="sets cudaLimitMaxL2FetchGranularity on the context and launches no other kernel"),
    # Python switches, read per call (builder.py): tested in-process against their explicit arguments
    "PG_LEVELS": dict(in_process="plan_levels(): partition levels other than the plan, and level lists the kernels refuse"),
    "PG_REGION_BITS": dict(in_process="RoundBuilder(region_bits=...)"),
    "PG_COMPACT": dict(in_process="RoundBuilder(compact=...)"),
    "PG_ROUNDS": dict(in_process="RoundBuilder(rounds=...)"),
    "PG_SUB_MB": dict(in_process="RoundBuilder(sub_bytes=...)"),
}

# ---------------------------------------------------------------------------------------------------------------------
# profiles: (name, env, battery groups, must launch, must not launch).  Orthogonal switches share a child.

_K3SC = "k3s_region_build_c<{true|false},{true|false},%s>"
BASELINE = [
    "k1x_tile_aggs", "k1x_scan", "k1x_pack",
    "k2a_partition_c<256,{false|true},{27|21|0},3,false>", "k2c_multisplit_c<{256|512|1024},true>", _K3SC % "512,4,false", "k3s_wide_insert",
    "k2a_partition<{0|1|2},256,{false|true}>", "k2x_multisplit<{256|512}>", "k3s_region_build<{8|12},{true|false},512,2>", "k3s_spill_insert",
    "k3_insert_records<6,true>", "k2b_split<512>", "k_table_clear", "k2_kmer_insert<{0|1|2}>", "k2_count_short", "k2_count_short_dev",
]
ALL_GROUPS = ["pack", "compact", "b16", "split", "misc"]

PROFILES = [
    ("default", {}, ALL_GROUPS, BASELINE, ["k1_fused_pack", "k1_tile_*", "k2b_split<256>", "k2c_refine<*>",
                                           "k3s_region_build_c<*,*,1024,2,*>", "k3s_region_build_c<*,*,*,*,true>"]),
    ("k1-legacy", {"PG_K1_LEGACY": "1"}, ["pack"], ["k1_tile_summaries", "k1_tile_scan", "k1_tile_pack"], ["k1x_*", "k1_fused_pack"]),
    ("k1-grid", {"PG_K1_GRID": "1"}, ["pack"], ["k1x_tile_aggs", "k1x_scan", "k1x_pack"], ["k1_tile_*", "k1_fused_pack"]),
    ("k1-single", {"PG_K1_SINGLE_PASS": "1"}, ["pack"], ["k1_fused_pack"], ["k1x_*", "k1_tile_*"]),
    ("k2ac-generic+splitc-512", {"PG_K2AC_GENERIC": "1", "PG_SPLITC_THREADS": "512"}, ["compact"],
     ["k2a_partition_c<256,{false|true},0,3,false>", "k2c_multisplit_c<512,true>"],
     ["k2a_partition_c<*,*,27,*,*>", "k2a_partition_c<*,*,21,*,*>", "k2c_multisplit_c<256,true>", "k2c_multisplit_c<1024,true>"]),
    ("k2ac-4+splitc-256", {"PG_K2AC_CTAS": "4", "PG_SPLITC_THREADS": "256"}, ["compact"],
     ["k2a_partition_c<256,false,{27|21},4,false>", "k2a_partition_c<256,false,0,3,false>", "k2c_multisplit_c<256,true>"],
     ["k2a_partition_c<256,false,27,3,false>", "k2a_partition_c<256,false,21,3,false>", "k2c_multisplit_c<512,true>",
      "k2c_multisplit_c<1024,true>"]),
    ("k3sc-1024+splitc-1024", {"PG_K3SC_CFG": "2", "PG_SPLITC_THREADS": "1024"}, ["compact"],
     [_K3SC % "1024,2,false", "k2c_multisplit_c<1024,true>"],
     ["k3s_region_build_c<*,*,512,4,*>", "k3s_region_build_c<*,*,*,*,true>", "k2c_multisplit_c<256,true>", "k2c_multisplit_c<512,true>"]),
    ("k3sc-fp", {"PG_K3SC_FP": "1"}, ["compact"], [_K3SC % "512,4,true"], ["k3s_region_build_c<*,*,*,*,false>", "k3s_region_build_c<*,*,1024,2,*>"]),
    ("k3sc-1024-fp", {"PG_K3SC_CFG": "2", "PG_K3SC_FP": "1"}, ["compact"], [_K3SC % "1024,2,true"],
     ["k3s_region_build_c<*,*,512,4,*>", "k3s_region_build_c<*,*,*,*,false>"]),
    ("split-256+k2a-128+k3s-256+k3-grid8-norotate", {"PG_SPLIT_THREADS": "256", "PG_K2A_THREADS": "128", "PG_K3S_THREADS": "256",
                                                      "PG_K3_GRID": "8", "PG_K3_ROTATE": "0"}, ["b16", "split"],
     ["k2x_multisplit<256>", "k2a_partition<{0|1|2},128,{false|true}>", "k3s_region_build<{8|12},{true|false},256,4>", "k3_insert_records<8,false>"],
     ["k2x_multisplit<512>", "k2x_multisplit<1024>", "k2a_partition<*,256,*>", "k2a_partition<*,512,*>", "k3s_region_build<*,*,512,2>",
      "k3_insert_records<6,*>", "k3_insert_records<8,true>", "k3_insert_ahead<*>"]),
    ("split-512+k3-norotate", {"PG_SPLIT_THREADS": "512", "PG_K3_ROTATE": "0"}, ["b16", "split"],
     ["k2x_multisplit<512>", "k3_insert_records<6,false>"], ["k2x_multisplit<256>", "k2x_multisplit<1024>", "k3_insert_records<*,true>"]),
    ("split-1024+k3-grid8", {"PG_SPLIT_THREADS": "1024", "PG_K3_GRID": "8"}, ["b16", "split"],
     ["k2x_multisplit<1024>", "k3_insert_records<8,true>"], ["k2x_multisplit<256>", "k2x_multisplit<512>", "k3_insert_records<6,*>"]),
    ("k2a-512+k3-ahead4", {"PG_K2A_THREADS": "512", "PG_K3_AHEAD": "1", "PG_K3_GRID": "4"}, ["b16"],
     ["k2a_partition<{0|2},512,{false|true}>", "k3_insert_ahead<4>"], ["k2a_partition<*,256,*>", "k2a_partition<*,128,*>", "k3_insert_records<*>"]),
    ("k3-ahead5", {"PG_K3_AHEAD": "1", "PG_K3_GRID": "5"}, ["b16"], ["k3_insert_ahead<5>"], ["k3_insert_records<*>", "k3_insert_ahead<4>"]),
    ("k3-ahead6", {"PG_K3_AHEAD": "1", "PG_K3_GRID": "6"}, ["b16"], ["k3_insert_ahead<6>"], ["k3_insert_records<*>", "k3_insert_ahead<5>"]),
    ("split-v1-k2b-256", {"PG_SPLIT_V1": "1", "PG_K2B_THREADS": "256"}, ["split"], ["k2b_split<256>", "k2c_refine<256>"],
     ["k2b_split<512>", "k2x_multisplit<*>"]),
    ("split-v1-k2b-512", {"PG_SPLIT_V1": "1", "PG_K2B_THREADS": "512"}, ["split"], ["k2b_split<512>", "k2c_refine<256>"],
     ["k2b_split<256>", "k2x_multisplit<*>"]),
    ("clear", {"PG_CLEAR_CTAS_PER_SM": "1"}, ["misc"], ["k_table_clear"], []),
    ("table-load", {"PG_TABLE_LOAD": "0.9"}, ["misc"], ["k2_kmer_insert<{0|1|2}>"], []),
    ("split-policy", {"PG_SPLIT_POLICY": "1"}, ALL_GROUPS, BASELINE, []),
]

# instantiations no profile launches, and why
ALLOWLIST = {
    "k2a_partition_c<512,false,{27|21|0},2,true>": "PEER (world > 1, stores into the owners' receive buffers): test_gpu_multi_one_device.py",
    "k2c_multisplit_c<{256|512|1024},false>": "K2b-c, the receive side of the compact multi-GPU build: test_gpu_multi_one_device.py",
}


# ---------------------------------------------------------------------------------------------------------------------
# battery inputs (seeded; the child builds them, the parent runs the oracle on the same bytes)

_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def pack_input():
    """About 13.6 MB: more than 148 x 5 tiles of 16 KB, so a grid of 148 (PG_K1_GRID=1) or 740 CTAs (the single-pass
    kernel) loops over several tiles.  Junk before the first header, line widths 1, 17, 61 and 100000, CRLF line ends in
    one record, lowercase / N / IUPAC codes, and no newline at the end of the file."""
    rng = np.random.default_rng(41)
    alpha = np.frombuffer(b"ACGTNacgtRY", dtype=np.uint8)
    p = [.23, .23, .23, .22, .03, .01, .01, .01, .01, .01, .01]
    out = [b"junk before the first header\nACGT\n"]
    for r, (width, n, eol) in enumerate([(61, 4_000_000, b"\n"), (17, 2_000_000, b"\r\n"), (1, 1_200_000, b"\n"), (100000, 4_100_000, b"\n"),
                                         (61, 333, b"\n")]):
        s = rng.choice(alpha, size=n, p=p).tobytes()
        out.append(b">r%d some text\n" % r + eol.join(s[i:i + width] for i in range(0, n, width)) + eol)
    data = b"".join(out)
    return data[:-1]


def hostile_input(seed=77, total=3000):
    """The multi-record generator of test_host_emul.py::test_emul_compact_records_random_inputs: N runs, IUPAC codes,
    lowercase, poly-A, ACGT x 16 (palindromic at every even k), records of 0 bases and of k - 1 and k bases for k 15, 21
    and 27.  No record has k + 1 bases for a k the battery uses: the reference leaves that length undefined."""
    rng = np.random.default_rng(seed)
    recs, r = [], 0
    while sum(len(x) for x in recs) < total:
        n = int(rng.choice([0, 14, 15, 20, 21, 26, 27, int(rng.integers(300, 1200)), int(rng.integers(300, 1200))]))
        s = bytearray(_ACGT[rng.integers(0, 4, n)].tobytes())
        if n > 300:
            a = int(rng.integers(0, n - 100)); s[a:a + 40] = b"N" * 40
            a = int(rng.integers(0, n - 100)); s[a:a + 50] = bytes(s[a:a + 50]).lower()
            a = int(rng.integers(0, n - 100)); s[a] = ord("R")
            a = int(rng.integers(0, n - 120)); s[a:a + 90] = b"A" * 90
            a = int(rng.integers(0, n - 120)); s[a:a + 64] = b"ACGT" * 16
        recs.append(b">r%d\n" % r + bytes(s) + b"\n")
        r += 1
    return b"".join(recs)


def hot_input():
    """test_gpu_parity.py::test_count_saturation_and_hot_keys: > 255 occurrences of one key, counts clamp at 255"""
    return b">a\n" + b"A" * 5000 + b"\n>b\n" + b"AC" * 3000 + b"\n>c\n" + b"A" * 300 + b"G" + b"A" * 300 + b"\n"


def pangenome_input(n, length):
    from pangenome_b200.synth import pangenome
    return pangenome(n, length)


INPUTS = {
    "pangenome": lambda: pangenome_input(4, 250_000),
    "pan16": lambda: pangenome_input(3, 20_000),
    "hostile": hostile_input,
    "hot": hot_input,
}
PACK_K = 5
