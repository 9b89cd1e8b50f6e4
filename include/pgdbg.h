/*
 * pgdbg.h - C ABI of libpgdbg.so: the B200 (sm_100a) implementation of the
 * de Bruijn-graph hot path of Rinoahu/pangenome's kmer_numba.py.
 *
 * The reference has no FFI: its hot path is a chain of numba-jitted Python
 * functions (SURVEY.md 8b).  Each entry point below names the reference
 * function(s) it replaces (file:line in /root/reference/kmer_numba.py); the
 * Python host in pangenome_b200/ binds them with ctypes and re-creates the
 * reference's stage API (seq2rdbg / dbg2rdbg / seq2graph) on top.
 *
 * Conventions
 *   - every function returns PG_OK (0) or a negative PG_ERR_* code; the text of
 *     the last error is available from pg_last_error(); nothing throws;
 *   - all `d_` pointers are CALLER-OWNED DEVICE buffers (e.g. a torch tensor's
 *     data_ptr()); the library allocates nothing on the device;
 *   - sizes are int64_t; `stream` is a cudaStream_t passed as void*; work is
 *     enqueued on it and the call returns without synchronising unless stated;
 *   - one host thread per GPU (one process per GPU under torchrun).
 *
 * Key / value conventions (the compared artefacts, SURVEY.md App. A)
 *   key   = base-5 code of the k-mer, little-endian digits A0 G1 C2 T3 other 4
 *           (kmer_numba.py:763-768, 975-985), k <= 27, as uint64;
 *   val12 = (lastc[prev] << 6) | lastc[next], bit order A,T,G,C,N,$ (:736-747);
 *   count = uint8 saturating at 255 (:551).
 * Internally a table in PG_MODE_CANONICAL stores one slot per {X, rc(X)} pair
 * holding both orientations' masks; exports expand it back to the reference's
 * "both orientations are separate keys" form.
 */
#ifndef PGDBG_H
#define PGDBG_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PG_OK 0
#define PG_ERR_INVALID (-1)    /* bad argument */
#define PG_ERR_CUDA (-2)       /* a CUDA runtime call failed */
#define PG_ERR_WORKSPACE (-3)  /* workspace too small */
#define PG_ERR_CAPACITY (-4)   /* an output buffer / table is too small */
#define PG_ERR_NOT_BGZF (-5)   /* pg_host_bgzf_index: the file does not start with a BGZF member */
#define PG_ERR_INFLATE (-6)    /* pg_bgzf_inflate: a member failed to decode (see its d_status) */

#define PG_MODE_LITERAL 0      /* one strand, literal keys            (-c 0 / -c 1)       */
#define PG_MODE_LITERAL_RC 1   /* both strands, two literal inserts per position (-c 2/3) */
#define PG_MODE_CANONICAL 2    /* both strands, one paired slot per position     (-c 2/3) */

/* indices into the int64 stats block of a table */
#define PG_STAT_OVERFLOW 0     /* != 0: probing gave up, table too small          */
#define PG_STAT_SHORT 1        /* insertions of the short-record sentinel key (Q5) */
#define PG_STAT_USED 2         /* occupied slots: kept by the inserts, recomputed by pg_table_count */
#define PG_STAT_ENTRIES 3      /* entries in reference convention (pg_table_count) */
#define PG_STAT_LOST 4         /* != 0: update records were dropped before they reached the table (a bucket and its
                                  spill overflowed, pg_buckets_plan): rebuild with smaller rounds */
#define PG_STAT_WORDS 8

typedef void *pg_stream_t;

/* An open-addressing table: `capacity` (power of two) 16-byte slots
 * {uint64 key, uint32 masks, uint32 count:22 | generation tag:10}.  A slot is live
 * only while its tag equals `epoch`, which makes emptying the table O(1)
 * (pg_table_reset).  Replaces class oakht (kmer_numba.py:340-679) and init_dict
 * (:1097-1122).  Life cycle: allocate, set epoch = 1, pg_table_clear once;
 * before every further build pg_table_reset. */
typedef struct pg_table {
    uint64_t *d_slots;   /* device, 2 * capacity uint64 */
    int64_t capacity;    /* power of two */
    int64_t *d_stats;    /* device, PG_STAT_WORDS int64 */
    int32_t mode;        /* PG_MODE_* */
    int32_t k;           /* k-mer length, 1..27 */
    int32_t epoch;       /* 1..1023: generation of the live slots (host side; pg_table_reset advances it) */
    int32_t region_bits; /* 0: linear probing wraps around the whole table.  r > 0: it wraps inside the aligned block of 2^r
                            slots the home slot lies in, so that block holds every key that hashes into it - the layout
                            pg_region_build produces (one block = one shared-memory table) and every later upsert keeps */
    int64_t alloc_capacity; /* slots allocated behind d_slots when `capacity` selects only a prefix of the buffer
                               (0 = same as capacity).  When the 10-bit tag wraps, pg_table_reset rewrites ALL of
                               them: a slot beyond `capacity` must not keep a tag of the previous cycle. */
    int32_t hash_kind;   /* which code the slot-placement hash is taken of: 0 = the base-5 key (default), 1 = the 2-bit code of
                            an ACGT-only key (keys with an ambiguity digit: the complemented base-5 key) - the layout
                            pg_region_build_c produces from compact 8-byte records; every later upsert / look-up keeps it */
    int32_t reserved;
} pg_table;

const char *pg_last_error(void);
int pg_version(void);
/* number of SMs of the current device (grid sizing); negative on error */
int pg_device_sms(void);

/* ---- K1: FASTA scan + pack --------------------------------------------------
 * Replaces seq2bytes/readline_jit_/seqio_jit_ (kmer_numba.py:117-188) and the
 * alpha / lastc / tab_rev_bytes character tables (:191-195, 736-768).
 * Input : d_fasta[nbytes], the raw file.
 * Output: d_pk2  - 2 bits per base, 16 bases per uint32 (base i of the
 *                  concatenated sequence stream at bits 2*(i%16) of word i/16);
 *                  ACGT hold the base-5 digit (A0 G1 C2 T3); ambiguous bases
 *                  hold 0 for N/n and 1 for anything else;
 *         d_amb  - 1 bit per base, 32 per uint32: set for non-ACGT bytes;
 *         both must hold pg_pack_words(cap_bases) uint32 (padding included) and
 *         cap_bases >= nbytes always suffices;
 *         d_hdr_off[r] - byte offset of record r's '>' in the file;
 *         d_seq_off[r] - offset of record r's first base in the stream,
 *                        d_seq_off[n_rec] = end of the last record;
 *         d_counts[0] = n_rec (may exceed cap_records: then only the first
 *                       cap_records entries were written - grow and call again),
 *         d_counts[1] = total bases in the stream, d_counts[2] = '\n' count.
 * Bases that precede the first header occupy [0, d_seq_off[0]) and belong to no
 * record (the reference drops them, :150-152).  Quirks kept: the last byte of
 * every line is dropped even without a final newline (Q8); '\r' is a base (Q9).
 */
int64_t pg_pack_words(int64_t cap_bases);
int64_t pg_fasta_workspace_bytes(int64_t nbytes);
int pg_fasta_scan_pack(const uint8_t *d_fasta, int64_t nbytes,
                       uint32_t *d_pk2, uint32_t *d_amb, int64_t cap_bases,
                       int64_t *d_hdr_off, int64_t *d_seq_off, int64_t cap_records,
                       int64_t *d_counts, void *d_ws, int64_t ws_bytes, pg_stream_t stream);

/* ---- FASTQ pack: pg_fasta_scan_pack's outputs from a FASTQ file -----------------------------------
 * A FASTQ record is exactly four lines: header ('@'), sequence, separator ('+'), quality (as long as the
 * sequence line; never read otherwise).  The file F is packed as the FASTA file fasta(F) - each record's
 * header line with '>' for '@', then its sequence line - would be by pg_fasta_scan_pack: same d_pk2 / d_amb,
 * d_seq_off, d_counts[0..1]; d_hdr_off[r] = offset of record r's '@' line in F; d_counts[2] = '\n' count of F.
 * Every byte of a sequence line but its '\n' is a base ('\r' too, Q9).  Lines of '\n' alone may follow the
 * last record.  cap_records as for pg_fasta_scan_pack: d_counts[0] > cap_records means the index did not
 * fit (grow and call again; d_status is then not set).  The workspace size depends on cap_records.
 * d_status (2 int64, device): {-1, 0} for a valid file; otherwise {byte offset of the first malformed
 * record's header line, PG_FQ_BAD_*} and d_counts[0] = d_counts[1] = 0, so nothing is built from it.
 * The input is untrusted: any bytes give a status, never an out-of-bounds access.
 */
#define PG_FQ_BAD_HEADER 1         /* the header line does not start with '@' */
#define PG_FQ_BAD_SEPARATOR 2      /* the separator line does not start with '+' */
#define PG_FQ_BAD_QUALITY_LENGTH 3 /* quality and sequence lines differ in length */
#define PG_FQ_TRUNCATED 4          /* the last record has fewer than four lines (e.g. wrapped FASTQ) */
int64_t pg_fastq_workspace_bytes(int64_t nbytes, int64_t cap_records);
int pg_fastq_scan_pack(const uint8_t *d_fastq, int64_t nbytes,
                       uint32_t *d_pk2, uint32_t *d_amb, int64_t cap_bases,
                       int64_t *d_hdr_off, int64_t *d_seq_off, int64_t cap_records,
                       int64_t *d_counts, int64_t *d_status, void *d_ws, int64_t ws_bytes, pg_stream_t stream);

/* ---- BGZF input: gzip members of at most 64 KiB, each a self-contained raw-DEFLATE stream -------
 * (the `bgzip` / `samtools faidx` format: gzip header with FLG = FEXTRA and a "BC" extra subfield of
 * SLEN 2 holding BSIZE = member size - 1; CRC-32 and ISIZE trailer).  A concatenation of BGZF files is
 * BGZF too (its empty EOF marker members then appear mid-file).
 * pg_host_bgzf_index (HOST pointers): walks the member headers of the file image gz[nbytes];
 *   member_off[i] = byte offset of member i in the file, out_off[i] = offset of its output in the
 *   inflated stream (exclusive scan of ISIZE); both need cap + 1 entries, entry n_members holds the
 *   file size / the inflated size.  counts[0] = n_members (may exceed cap: then only the first cap
 *   entries were written - grow and call again), counts[1] = inflated size.  Returns PG_ERR_NOT_BGZF
 *   when the first member is not BGZF (plain text, a `gzip` file, an empty file), PG_ERR_INVALID when
 *   a later member is not BGZF, is truncated, or claims more than 65536 output bytes.
 * pg_bgzf_inflate: inflates members [0, n_members) of d_gz[gz_bytes] into d_out[out_bytes] in ONE
 *   launch, member i from d_gz[d_member_off[i], d_member_off[i + 1]) into
 *   d_out[d_out_off[i], d_out_off[i + 1]) (device arrays of n_members + 1 entries: the index above,
 *   or any contiguous slice of it rebased to its first entry).  Every member is checked: header,
 *   Huffman codes, back-reference distances, output length = ISIZE = its window, CRC-32.  A bad
 *   member never makes the kernel read or write outside its own input and output ranges.
 *   d_status (device, 2 int64, overwritten): [0] = members that failed, [1] = (first failed member
 *   << 8) | its PG_INF_ERR_* kind, INT64_MAX when none failed.  Returns without synchronising: the
 *   caller reads d_status before it uses d_out.
 */
#define PG_INF_ERR_HEADER 1     /* not a BGZF member header, or its window does not fit */
#define PG_INF_ERR_TRUNCATED 2  /* the compressed data ends inside a block */
#define PG_INF_ERR_BLOCK 3      /* block type 3 */
#define PG_INF_ERR_STORED 4     /* stored block: LEN and NLEN disagree */
#define PG_INF_ERR_CODE 5       /* bad code lengths: over-subscribed or incomplete code, bad repeat, too many symbols */
#define PG_INF_ERR_SYMBOL 6     /* a bit pattern no code word matches, or literal/length 286-287, distance 30-31 */
#define PG_INF_ERR_DISTANCE 7   /* a back-reference before the start of the member's output */
#define PG_INF_ERR_OVERFLOW 8   /* more output than ISIZE */
#define PG_INF_ERR_LENGTH 9     /* less output than ISIZE, ISIZE != window, or bytes left after the final block */
#define PG_INF_ERR_CRC 10       /* CRC-32 of the output differs from the trailer's */
int pg_host_bgzf_index(const uint8_t *gz, int64_t nbytes, int64_t *member_off, int64_t *out_off, int64_t cap,
                       int64_t *counts);
int pg_bgzf_inflate(const uint8_t *d_gz, int64_t gz_bytes, const int64_t *d_member_off, const int64_t *d_out_off,
                    int64_t n_members, uint8_t *d_out, int64_t out_bytes, int64_t *d_status, pg_stream_t stream);

/* ---- K2+K3: k-mer extraction fused with table insertion ---------------------
 * pg_table_clear  : all slots empty (for every epoch), stats zero: 16 B/slot of HBM writes
 *                   (oakht.__init__ :341-352)
 * pg_table_reset  : the same effect between builds without touching the slots: ++t->epoch, stats
 *                   zero (falls back to pg_table_clear when the 10-bit tag wraps)
 * pg_kmer_insert  : for every k-mer occurrence of records [0, n_rec) whose
 *                   start lies in stream range [g_begin, g_end): key/val as
 *                   build_dbg + add_kmer (:1036-1093), both strands unless
 *                   mode == PG_MODE_LITERAL (seq2dbg_jit_ :1202-1230), including
 *                   Q1 (predecessor of each strand's last k-mer), Q3, Q4, Q5.
 *                   Records shorter than k only bump PG_STAT_SHORT (counted
 *                   when their offset lies in the range).
 */
int64_t pg_table_bytes(int64_t capacity);
int pg_table_clear(const pg_table *t, pg_stream_t stream);
int pg_table_reset(pg_table *t, pg_stream_t stream);
/* adds (strands x records of [0,n_rec) shorter than k whose offset lies in [g_begin, g_end)) to PG_STAT_SHORT;
 * the range that reaches the end of the stream (g_end >= d_seq_off[n_rec]) also owns records AT g_end (trailing
 * empty records), so consecutive ranges [a,b) [b,c) never count a record twice.
 * pg_kmer_insert calls it itself, the two-phase path (pg_kmer_partition) does not */
int pg_count_short(const pg_table *t, const int64_t *d_seq_off, int64_t n_rec, int64_t g_begin, int64_t g_end,
                   pg_stream_t stream);
int pg_kmer_insert(const pg_table *t, const uint32_t *d_pk2, const uint32_t *d_amb,
                   const int64_t *d_seq_off, int64_t n_rec, int64_t g_begin, int64_t g_end,
                   pg_stream_t stream);

/* ---- K2a + K3: the two-phase build (single-GPU fast path and the multi-GPU split) ---------
 * pg_kmer_partition: same occurrences as pg_kmer_insert, but each position emits one
 *   16-byte update record {uint64 key, uint32 masks, uint32 inc} (mode/k taken from `t`;
 *   its slots are not touched) into bucket
 *       (owner << sub_bits) | sub,   owner = low owner_bits of mix64(key)  (which GPU owns the key)
 *                                    sub   = top sub_bits of mix64(key)    (= which 1/2^sub_bits region
 *                                            of ANY power-of-two table the key's home slot lies in)
 *   d_records holds 2^(owner_bits+sub_bits) buckets of part_cap records each; d_part_counts[b]
 *   = records produced for bucket b (records beyond part_cap are dropped: compare and fall back).
 *   Optional distinct-key estimator (d_sample_keys != NULL): keys whose mix has bits 8..15 == 0 - a 1/256
 *   sample of the key space - are collected in a power-of-two CAS set the caller filled with 0xFF;
 *   *d_sample_count (caller-zeroed) ends as its size, so 256 x that estimates the slots the table needs
 *   (a value >= 2^40 means the set overflowed: use the upper bound).  This is how the table is sized
 *   BEFORE it is cleared and filled - the reference instead grows x1.62 and rehashes (:423-474).
 * pg_insert_records: upsert the records of n_regions x n_src segments
 *   [seg_off[b*n_src+j], +seg_cnt[b*n_src+j]) of d_records (record units), region after region
 *   (n_src = source ranks x pipeline chunks that contributed to a region; 1 on a single GPU), so
 *   that the table region being updated stays in L2.  seg_cap (> 0) clamps every segment count: a count
 *   above the bucket capacity only says that K2a dropped records, K3 must not read past the bucket.
 *   Replaces the same reference lines as pg_kmer_insert; the all-to-all between the two calls is
 *   the host's (torch.distributed / NCCL).
 */
int pg_kmer_partition(const pg_table *t, const uint32_t *d_pk2, const uint32_t *d_amb, const int64_t *d_seq_off,
                      int64_t n_rec, int64_t g_begin, int64_t g_end, int owner_bits, int sub_bits,
                      uint64_t *d_records, int64_t part_cap, int64_t *d_part_counts,
                      uint64_t *d_sample_keys, int64_t sample_cap, int64_t *d_sample_count, pg_stream_t stream);
/* CUDA IPC plumbing for the receive buffers of the fused extraction + exchange (peer bucket sets, below):
 * pg_peer_alloc / open / close / free (64-byte handle; one process per GPU). */
int pg_peer_alloc(int64_t bytes, void **d_ptr, uint8_t *handle64);
int pg_peer_open(const uint8_t *handle64, void **d_ptr);
int pg_peer_close(void *d_ptr);
int pg_peer_free(void *d_ptr);
/* Device-argument variants for a fully asynchronous build of ALL records of a packed stream: n_rec and the
 * stream range are read on the device from pg_fasta_scan_pack's outputs (d_counts, d_seq_off; cap_records as
 * passed to it; max_bases = an upper bound such as the file size, for grid sizing), so K1 -> K2a -> K3 can be
 * enqueued back to back.  If the record index was truncated (n_rec > cap_records) bucket 0's count is set to
 * 2^62 and nothing else is written: the host notices at its next read-back and falls back. */
int pg_kmer_partition_dev(const pg_table *t, const uint32_t *d_pk2, const uint32_t *d_amb, const int64_t *d_seq_off,
                          const int64_t *d_counts, int64_t cap_records, int64_t max_bases, int owner_bits, int sub_bits,
                          uint64_t *d_records, int64_t part_cap, int64_t *d_part_counts, pg_stream_t stream);
int pg_count_short_dev(const pg_table *t, const int64_t *d_seq_off, const int64_t *d_counts, int64_t cap_records,
                       pg_stream_t stream);

/* ---- bucket sets: rounds, spill, receiver-side split (the streaming single- and multi-GPU builders) ----------
 * A bucket set names where K2a (or K2b) puts its update records:
 *   local : d_records holds 2^(owner_bits+sub_bits) buckets of part_cap records followed by ONE spill bucket of
 *           spill_cap records.  A record whose bucket is full goes to the spill instead of being dropped, so hash
 *           skew (one k-mer making up a visible share of the input: poly-A, satellites - BASELINE configs 4/5) is
 *           absorbed; K3 sweeps the spill as one more region (table_upsert finds the home slot from the key, a
 *           record does not have to sit in "its" region to be inserted correctly).
 *   peer  : d_peer_bases[owner] = rank `owner`'s receive buffer (pg_peer_alloc/open); bucket (owner, sub) lands at
 *           [my_rank][sub][part_cap] there.  No spill across NVLink: overflow shows in the counts.
 * d_part_counts has 2^(owner_bits+sub_bits) + 1 counters: records PRODUCED per bucket (may exceed part_cap) and,
 * last, records offered to the spill.
 * pg_kmer_partition_to: K2a into a bucket set (counters zeroed first).  With d_counts != NULL the record count and
 *   stream range are read on the device (pg_kmer_partition_dev) and [g_begin, g_end) is RELATIVE to the first
 *   record's offset (g_end < 0 = to the end): one round of a multi-round build without any host read-back.
 * pg_records_split (K2b): re-sort n_seg segments of records (e.g. what each source rank sent, bucketed by owner only
 *   so the NVLink runs are long) into the 2^sub_bits hash-prefix regions of a local bucket set: 32 B of HBM traffic
 *   per record buys L2-resident K3 regions for tables of any size.  A segment count above seg_cap (the sender's
 *   wire bucket overflowed) is clamped and raises PG_STAT_LOST in d_table_stats (may be NULL).
 * pg_buckets_plan: d_seg_cnt[i] = min(count, capacity) for the 2^bits buckets + the spill (what pg_insert_records
 *   sweeps, with seg offsets i * part_cap), and PG_STAT_LOST in d_table_stats when records were dropped.
 * Replaces oakht.resize's grow-and-rehash (kmer_numba.py:423-474) as the answer to "the table / a bucket is full". */
typedef struct pg_bucket_set {
    uint64_t *d_records;
    uint64_t *const *d_peer_bases;
    int64_t *d_part_counts;
    int64_t part_cap, spill_cap;
    int32_t owner_bits, sub_bits, my_rank, reserved;
} pg_bucket_set;
int pg_kmer_partition_to(const pg_table *t, const uint32_t *d_pk2, const uint32_t *d_amb, const int64_t *d_seq_off,
                         int64_t n_rec, int64_t g_begin, int64_t g_end, const int64_t *d_counts, int64_t cap_records,
                         int64_t max_bases, const pg_bucket_set *out, uint64_t *d_sample_keys, int64_t sample_cap,
                         int64_t *d_sample_count, pg_stream_t stream);
int pg_records_split(const uint64_t *d_records_in, const int64_t *d_seg_off, const int64_t *d_seg_cnt, int n_seg,
                     int64_t seg_cap, const pg_bucket_set *out, int64_t *d_table_stats, pg_stream_t stream);
int pg_buckets_plan(const pg_bucket_set *b, int64_t *d_seg_cnt, int64_t *d_table_stats, pg_stream_t stream);
int pg_insert_records(const pg_table *t, const uint64_t *d_records, const int64_t *d_seg_off,
                      const int64_t *d_seg_cnt, int n_regions, int n_src, int64_t seg_cap, pg_stream_t stream);

/* ---- K2c + K3s: the table built region by region in shared memory (csrc/region_build.cu) ----------------------
 * Instead of one L2 atomic per update record (pg_insert_records, bound by the chip's random-atomic rate), the records
 * are bucketed down to ONE bucket per table region of 2^region_bits slots (t->region_bits = 12: 64 KB, or 8 for tiny
 * tables) and a CTA builds each region in shared memory - 64-bit CAS claim, atomicOr / atomicAdd merge - streaming its
 * bucket once and writing the finished region to HBM once.  All HBM traffic is sequential.
 * pg_records_refine (K2c): every bucket of the local set `coarse` (2^sub_bits buckets by the TOP hash bits, owner_bits 0,
 *   with its spill) is split 2^fine_bits ways by the NEXT hash bits (fine_bits 1..8; 32 B of HBM traffic per record):
 *   d_fine_records holds 2^(sub_bits+fine_bits) buckets of fine_part_cap records followed by a spill of fine_spill_cap
 *   records, d_fine_counts one counter more than buckets (zeroed here; same meaning as pg_bucket_set.d_part_counts).
 *   The coarse spill's records move to the fine spill.  A spill above its capacity raises PG_STAT_LOST in
 *   d_table_stats (may be NULL).
 * pg_region_build (K3s): bucket b of d_records (capacity >> region_bits buckets of part_cap records, then the spill)
 *   becomes region b of the table.  first_round != 0: regions start empty and EVERY slot of the table is rewritten;
 *   0: they start from what earlier rounds left in HBM.  The spill's records are upserted afterwards with L2 atomics.
 *   A region that fills up raises PG_STAT_OVERFLOW (rebuild with a larger table), a count above part_cap without a spill
 *   or a spill above spill_cap raises PG_STAT_LOST.  Probing wraps inside a region (pg_table.region_bits), in this
 *   call and in every later upsert into the table.
 * Replaces oakht.__setitem__ + resize (kmer_numba.py:423-474, 540-561) on the build path. */
int pg_records_refine(const pg_bucket_set *coarse, int fine_bits, uint64_t *d_fine_records, int64_t *d_fine_counts,
                      int64_t fine_part_cap, int64_t fine_spill_cap, int64_t *d_table_stats, pg_stream_t stream);
/* pg_records_resplit: pg_records_refine on raw arrays, for chains of splits (wire -> 2^5 -> 2^11 -> 2^18 buckets: three
 * passes of <= 2^7 ways (in_bits <= 13) move a record at ~4 TB/s each, one pass of 2^10 ways at ~1 TB/s because its runs are 128 bytes):
 * d_in holds 2^in_bits buckets of in_part_cap records + a spill of in_spill_cap (counters in d_in_counts, one more than
 * buckets); bucket s is split 2^bits ways by hash bits [in_bits, in_bits + bits) into buckets [s << bits, ...) of d_out. */
int pg_records_resplit(const uint64_t *d_in, const int64_t *d_in_counts, int in_bits, int64_t in_part_cap, int64_t in_spill_cap,
                       int bits, uint64_t *d_out, int64_t *d_out_counts, int64_t out_part_cap, int64_t out_spill_cap,
                       int64_t *d_table_stats, pg_stream_t stream);
int pg_region_build(const pg_table *t, const uint64_t *d_records, const int64_t *d_counts, int64_t part_cap, int64_t spill_cap,
                    int first_round, pg_stream_t stream);

/* ---- the same build on COMPACT 8-byte update records (csrc/compact_build.cu) -----------------------------------
 * An interior position (the k-mer, the base before and the base after it are ACGT inside one record) travels as
 *     [ 2-bit code of the canonical k-mer : 54 | previous base * 4 + next base : 4 | rc strand is the key : 1 | palindrome : 1 | 0 : 4 ]
 * and every other position (record edges: '#', '$', Q1; ambiguity codes) as a 16-byte WIDE record {base-5 key, masks,
 * increment} in the set's wide spill, where a compact record whose bucket is full goes as well.  Half the record
 * traffic of the 16-byte path and no base-5 arithmetic in the extraction (both strands' codes roll with shifts); the
 * base-5 key the reference's table holds (kmer_numba.py:975-988) is produced when a finished region is written out.
 * Buckets and slots are placed by mix64 of the 2-BIT code: the table must carry hash_kind = 1 (and region_bits = 12).
 * PG_MODE_CANONICAL only.  One pg_cbuckets per partition level; all levels of a round share the wide spill.
 * pg_kmer_partition_c (K2a-c): arguments as pg_kmer_partition_to; zeroes out->d_counts and *out->d_wide_count.
 * pg_records_resplit_c (K2c-c): bucket s of `in` is split 2^bits ways (1..10; the builder uses at most 8) by hash bits [in->bits, in->bits + bits)
 *   into buckets [s << bits, ...) of `out` (out->bits == in->bits + bits; zeroes out->d_counts).
 * pg_region_build_c (K3s-c): bucket b of `b` (b->bits == log2(capacity) - 12) becomes region b of the table, then the
 *   wide spill is upserted with L2 atomics.  first_round as pg_region_build.  last_round = 0: more rounds follow - the
 *   table is left in an INTERMEDIATE form (ACGT-only keys as 2-bit codes under bit 63) that only the next
 *   pg_region_build_c / pg_wide_insert calls of the same build may read; last_round != 0 writes the base-5 keys.
 *   A single-round build passes 1, 1.  PG_STAT_OVERFLOW: a region filled up;
 *   PG_STAT_LOST: the wide spill exceeded wide_cap (or K1's record index was truncated) - rebuild on the 16-byte path. */
typedef struct pg_cbuckets {
    uint64_t *d_records;     /* 2^bits buckets of part_cap (even) 8-byte records, 16-byte aligned */
    int64_t *d_counts;       /* 2^bits counters: records PRODUCED for the bucket (the surplus over part_cap went to the wide spill) */
    int64_t part_cap;
    int32_t bits, reserved;
    uint64_t *d_wide;        /* wide_cap 16-byte records */
    int64_t *d_wide_count;   /* one counter: records offered to the wide spill (peer sets: one per owner rank) */
    int64_t wide_cap;
    /* fused exchange (pg_kmer_partition_c across GPUs; all NULL / 0 otherwise): bucket = owner rank = the LOW bits of
     * mix64(2-bit code), bits = log2(ranks); bucket o is stored straight into rank o's receive buffers over NVLink at the
     * slice of source rank my_rank - compact records at d_peer_bases[o] + my_rank * part_cap, wide ones at
     * d_wide_peer_bases[o] + my_rank * wide_cap (records).  d_records / d_wide stay NULL.  What arrived is split into
     * hash-prefix buckets by pg_records_split_c (out->bits 0..10; 0 = one bucket, for a table of one region per rank)
     * and the wide segments are upserted by pg_wide_insert. */
    uint64_t *const *d_peer_bases;
    uint64_t *const *d_wide_peer_bases;
    int32_t my_rank, reserved2;
} pg_cbuckets;
int pg_kmer_partition_c(const pg_table *t, const uint32_t *d_pk2, const uint32_t *d_amb, const int64_t *d_seq_off,
                        int64_t n_rec, int64_t g_begin, int64_t g_end, const int64_t *d_counts, int64_t cap_records,
                        int64_t max_bases, const pg_cbuckets *out, uint64_t *d_sample_keys, int64_t sample_cap,
                        int64_t *d_sample_count, pg_stream_t stream);
int pg_records_resplit_c(const pg_cbuckets *in, int bits, const pg_cbuckets *out, int k, int64_t *d_table_stats, pg_stream_t stream);
int pg_region_build_c(const pg_table *t, const pg_cbuckets *b, int first_round, int last_round, pg_stream_t stream);
int pg_records_split_c(const pg_cbuckets *in, const pg_cbuckets *out, int k, int64_t *d_table_stats, pg_stream_t stream);
int pg_wide_insert(const pg_table *t, const uint64_t *d_wide, const int64_t *d_count, int64_t cap, int last_round, pg_stream_t stream);

/* ---- table read-out ---------------------------------------------------------
 * pg_table_count   : fills PG_STAT_USED / PG_STAT_ENTRIES in t->d_stats.
 * pg_table_export  : unsorted (key, val12, count<=255) in the reference's
 *                    convention (iteritems :623-631): both orientations as
 *                    separate keys, plus the sentinel key 2^64-1 (val 32) if
 *                    any short record was inserted.  *d_n = entries produced;
 *                    entries beyond cap are dropped (compare *d_n with cap).
 * pg_table_checksum: d_out[0..2] = (entries, sum, xor) of mix64 over the same
 *                    entries - order independent, equals
 *                    oracle.table_checksum() of the reference's table.
 */
int pg_table_count(const pg_table *t, pg_stream_t stream);
int pg_table_export(const pg_table *t, uint64_t *d_keys, uint16_t *d_vals, uint8_t *d_cnts,
                    int64_t cap, int64_t *d_n, pg_stream_t stream);
int pg_table_checksum(const pg_table *t, uint64_t *d_out, pg_stream_t stream);

/* ---- K4: reduced-dBG selection ---------------------------------------------
 * Replaces nbit + build_rdbg_jit_ + dbg2rdbg (kmer_numba.py:723-727, 1292-1321):
 * keep k-mers with popcount(in6) != 1 or popcount(out6) != 1.
 * pg_rdbg_count : d_out[0] = slots the rdBG table needs, d_out[1] = members.
 * pg_rdbg_select: inserts the members of `dbg` into the cleared table `rdbg`
 *                 (same mode/k; capacity >= 2 * d_out[0] recommended).  The
 *                 rdBG count word holds flags: bit0/bit1 = orientation 0/1 is a
 *                 member, bit2 = key present only as the phantom key 0 (Q6).
 * pg_rdbg_export: unsorted member (key, val12), reference convention.
 */
int pg_rdbg_count(const pg_table *dbg, int64_t *d_out, pg_stream_t stream);
int pg_rdbg_select(const pg_table *dbg, const pg_table *rdbg, pg_stream_t stream);
int pg_rdbg_export(const pg_table *rdbg, uint64_t *d_keys, uint16_t *d_vals,
                   int64_t cap, int64_t *d_n, pg_stream_t stream);

/* ---- K5: compressed-path hits ---------------------------------------------------
 * Replaces the first half of rdbg_edge_weight (kmer_numba.py:1446-1468) and of
 * seq2path_jit_ (:1523-1549): walk one strand of records [0, n_rec) and keep the
 * occurrences whose k-mer is an rdBG member (`has_key`, including the phantom
 * key 0, Q6).  strand 0 = forward, 1 = reverse complement (hits are still
 * emitted in ascending forward position).  Outputs, ordered by position:
 *   d_hit_g    stream offset of the k-mer's first base
 *   d_hit_node node key = ((rdBG slot << 1 | orientation) << 11) | v5 with
 *              v5 = (lastc[prev] << 5) | lastc[next]   (offbit 5, F7)
 *   d_hit_rec  record index,  d_hit_v6 = (lastc[prev] << 6) | lastc[next]
 * *d_n_hits = hits found; hits beyond cap_hits are dropped (grow and repeat).
 */
int64_t pg_path_workspace_bytes(int64_t n_bases);
int pg_path_hits(const pg_table *rdbg, const uint32_t *d_pk2, const uint32_t *d_amb, const int64_t *d_seq_off,
                 int64_t n_rec, int64_t g_begin, int64_t g_end, int strand,
                 int64_t *d_hit_g, uint64_t *d_hit_node, int32_t *d_hit_rec, uint16_t *d_hit_v6, int64_t cap_hits,
                 int64_t *d_n_hits, void *d_ws, int64_t ws_bytes, pg_stream_t stream);

/* ---- K6/K7: rdBG edge weights and connected components ----------------------------
 * pg_graph: three single-word open-addressing tables in caller-owned buffers
 * (capacities: powers of two <= 2^32; size each >= 2x the number of hits).
 * Replaces the typed-Dict edge map + `visit` dict (:1446-1518) and the label
 * dict built from the external `mcl` output (:1907-1944).  The reference's
 * clustering itself is third-party MCL; here components are the connected
 * components of the edge list restricted to weight >= min_weight (min_weight 1 =
 * the definition of the reference's other/test_net.py).
 * d_stats: [0] overflow flag, [1] node slots used (every hit; only nodes that occur in an
 * edge are exported / labelled - the reference builds its label dict from the edge list),
 * [2] edges.
 */
typedef struct pg_graph {
    uint64_t *d_node_keys;    /* node_cap                                  */
    uint32_t *d_node_parent;  /* node_cap: union-find parent / root         */
    int32_t *d_node_label;    /* node_cap: region label of the node's component (written by the host) */
    uint64_t *d_edge_keys;    /* edge_cap: (node slot a << 32) | node slot b */
    uint32_t *d_edge_w;       /* edge_cap: weight = record-strands containing the edge */
    uint64_t *d_edge_first;   /* edge_cap: smallest walk ordinal (= .xyz file order)    */
    uint64_t *d_visit_keys;   /* visit_cap: (edge slot << 32) | record-strand id        */
    int64_t *d_stats;         /* 8 int64 */
    int64_t node_cap, edge_cap, visit_cap;
} pg_graph;
int pg_graph_clear(const pg_graph *g, pg_stream_t stream);
int pg_graph_add_hits(const pg_graph *g, const uint64_t *d_hit_node, const int32_t *d_hit_rec, int64_t n_hits,
                      uint32_t *d_hit_nslot, int strand, int n_strands, pg_stream_t stream);
int pg_graph_components(const pg_graph *g, uint32_t min_weight, pg_stream_t stream);
int pg_graph_export_edges(const pg_graph *g, const pg_table *rdbg, uint64_t *d_c0, uint32_t *d_v0, uint64_t *d_c1,
                          uint32_t *d_v1, uint32_t *d_w, uint64_t *d_first, int64_t cap, int64_t *d_n, pg_stream_t stream);
int pg_graph_export_nodes(const pg_graph *g, const pg_table *rdbg, uint32_t *d_nslot, uint64_t *d_code, uint32_t *d_v5,
                          uint32_t *d_root, int64_t cap, int64_t *d_n, pg_stream_t stream);

/* ---- K7m: Markov clustering of the rdBG edge graph (opt-in, `--cluster mcl`) -------------
 * Replaces the external `mcl <xyz> --abc -I r` run (kmer_numba.py:1911).  The definition (DESIGN.md §3) is
 * this project's: agreement with micans mcl is unverified.  Column-stochastic matrix M in CSC form
 * (int64 column pointers, int32 rows ascending inside a column, float32 values); one iteration is
 *   M <- normalise(inflate_r(prune(M.M)))
 * with every float32 sum taken left to right (expansion: ascending k; column sums and sums of squares:
 * ascending row) and correctly rounded operations only, so the CPU oracle matches bit for bit when r is a
 * multiple of 1/2 (x^r = x^floor(r) by repeated products, times sqrt(x) for the half; any other r: powf).
 * prune: keep the min(S, #entries >= theta) largest entries of a column (value descending, row ascending);
 * a column with no entry >= theta keeps its largest one.  chaos_j = max_i M[i,j] / sum_i M[i,j]^2 - 1 after
 * normalisation; the run stops when max_j chaos_j < tau or after T iterations.
 *
 * pg_mcl_normalise: normalise every column in place; d_stats[PG_MCL_STAT_CHAOS] = max_j max(chaos_j, 0)
 *   (float bits), d_stats[PG_MCL_STAT_NNZ] = nonzeros.
 * pg_mcl_plan: d_prod[j] = products of column j (sum of nnz(col k) over k in col j); d_stage_off = exclusive
 *   scan of min(d_prod[j], S) (n + 1 entries: the staging size is d_stage_off[n]); columns with more than
 *   PG_MCL_WARP_PRODUCTS products are listed in d_large (cap n) and counted in d_stats[PG_MCL_STAT_LARGE];
 *   d_stats[PG_MCL_STAT_PRODUCTS] / [PG_MCL_STAT_MAXPROD] = total / largest product count.
 * pg_mcl_expand: expansion + prune + inflation + normalisation of every column into the staging arrays
 *   (column j at d_stage_off[j], d_kept[j] entries, rows ascending); columns up to PG_MCL_WARP_PRODUCTS
 *   products take one warp each, larger ones one CTA each (shared-memory accumulator up to
 *   PG_MCL_SMEM_SLOTS slots, else a slab of the caller's workspace d_ws per resident CTA; the slab holds
 *   pg_mcl_slab_slots(max products, n) slots).  n_ctas large-column CTAs run at once: ws_bytes >=
 *   n_ctas * 8 * slab slots.  Writes d_stats CHAOS / NNZ like pg_mcl_normalise.
 * pg_mcl_compact: next CSC from the staging arrays: d_colptr_out = exclusive scan of d_kept (n + 1 entries),
 *   rows / values copied; d_rows_out / d_vals_out hold d_stats[PG_MCL_STAT_NNZ] entries.
 * pg_mcl_components: one root per column (the smallest index of its component) of the undirected graph with
 *   an edge {i, j} per stored entry.
 * d_stats: PG_MCL_STAT_WORDS int64, zeroed by the caller before pg_mcl_plan / pg_mcl_normalise.
 * Scans use d_scan_ws of pg_mcl_scan_workspace_bytes(n) bytes.
 */
#define PG_MCL_PRUNE_THETA 1e-4f    /* theta: entries below it are pruned after expansion */
#define PG_MCL_SELECT_S 1024        /* S: entries a column keeps at most                   */
#define PG_MCL_CHAOS_TAU 1e-4f      /* tau: convergence when max chaos falls below it      */
#define PG_MCL_MAX_ITER 100         /* T: iterations at most                               */
#define PG_MCL_WARP_PRODUCTS 64     /* columns with at most this many products take the warp path */
#define PG_MCL_SMEM_SLOTS 2048      /* accumulator slots a CTA keeps in shared memory      */
#define PG_MCL_STAT_CHAOS 0
#define PG_MCL_STAT_NNZ 1
#define PG_MCL_STAT_PRODUCTS 2
#define PG_MCL_STAT_MAXPROD 3
#define PG_MCL_STAT_LARGE 4
#define PG_MCL_STAT_WORDS 8
int64_t pg_mcl_scan_workspace_bytes(int64_t n);
int64_t pg_mcl_slab_slots(int64_t max_products, int64_t n);
int pg_mcl_normalise(const int64_t *d_colptr, const int32_t *d_rows, float *d_vals, int64_t n, int64_t *d_stats,
                     pg_stream_t stream);
int pg_mcl_plan(const int64_t *d_colptr, const int32_t *d_rows, int64_t n, int64_t *d_prod, int64_t *d_stage_off,
                int32_t *d_large, int64_t *d_stats, void *d_scan_ws, int64_t scan_ws_bytes, pg_stream_t stream);
int pg_mcl_expand(const int64_t *d_colptr, const int32_t *d_rows, const float *d_vals, int64_t n, const int64_t *d_prod,
                  const int64_t *d_stage_off, const int32_t *d_large, int64_t n_large, int64_t max_products, float inflation,
                  int32_t *d_stage_rows, float *d_stage_vals, int64_t *d_kept, int64_t *d_stats, void *d_ws, int64_t ws_bytes,
                  int n_ctas, pg_stream_t stream);
int pg_mcl_compact(const int64_t *d_stage_off, const int32_t *d_stage_rows, const float *d_stage_vals, const int64_t *d_kept,
                   int64_t n, int64_t *d_colptr_out, int32_t *d_rows_out, float *d_vals_out, void *d_scan_ws,
                   int64_t scan_ws_bytes, pg_stream_t stream);
int pg_mcl_components(const int64_t *d_colptr, const int32_t *d_rows, int64_t n, int32_t *d_root, pg_stream_t stream);

/* ---- K8: per-record breakpoint labelling -------------------------------------------
 * Replaces seq2path_jit_ (:1523-1573): a hit matches when (code, v6) equals some
 * node's (code, v5) (Q7); matched hits are chained greedily ("starts[-1] < idx":
 * accept iff position > last accepted position + k, first iff position > 0), runs
 * of equal labels merge, every run yields the row (prev_end, last_pos + k, label).
 * Outputs one (record, end, label) per row in record/position order; the row's
 * start is the previous row's end within the record, else 0.  d_n_rows[0] = rows,
 * d_n_rows[1] = matched hits.  Synchronises the stream once.
 */
int64_t pg_label_workspace_bytes(int64_t n_hits);
int pg_label_regions(const pg_graph *g, const int64_t *d_hit_g, const uint64_t *d_hit_node, const int32_t *d_hit_rec,
                     const uint16_t *d_hit_v6, int64_t n_hits, const int64_t *d_seq_off, int k, int strand,
                     int32_t *d_row_rec, int64_t *d_row_end, int32_t *d_row_label, int64_t cap_rows, int64_t *d_n_rows,
                     void *d_ws, int64_t ws_bytes, pg_stream_t stream);

/* ---- multi-GPU plumbing for the stages after the dBG --------------------------------------
 * pg_table_export_raw / pg_table_insert_raw: move occupied slots {key, 64-bit value word} between
 *   tables (all-gather of the per-rank rdBG tables into one full rdBG table per rank; values are
 *   OR-ed, keys are unique across ranks).
 * pg_hits_decode: node key -> literal base-5 code (rank independent);
 * pg_hits_rekey : (code, v5) -> node key in THIS rank's rdBG table, so that hits gathered from all
 *   ranks can run through K6-K8 on one rank.
 */
int pg_table_export_raw(const pg_table *t, uint64_t *d_keys, uint64_t *d_vals, int64_t cap, int64_t *d_n, pg_stream_t stream);
int pg_table_insert_raw(const pg_table *t, const uint64_t *d_keys, const uint64_t *d_vals, int64_t n, pg_stream_t stream);
int pg_hits_decode(const pg_table *rdbg, const uint64_t *d_hit_node, int64_t n, uint64_t *d_hit_code, pg_stream_t stream);
int pg_hits_rekey(const pg_table *rdbg, const uint64_t *d_hit_code, const uint32_t *d_hit_v5, int64_t n, uint64_t *d_hit_node,
                  pg_stream_t stream);

/* ---- host-side text writers (HOST pointers) -------------------------------------------
 * The side files of seq2graph (kmer_numba.py:1893-1904 and the cluster file `mcl` leaves):
 * pg_host_write_xyz: "code0_v0\tcode1_v1\tweight\n" per edge in the order given;
 * pg_host_write_mcl: one tab-separated line of "code_v5" names per label; input sorted by
 *                    (label, code, v5).
 */
int pg_host_write_xyz(const char *path, const uint64_t *c0, const uint32_t *v0, const uint64_t *c1,
                      const uint32_t *v1, const uint32_t *w, int64_t n);
int pg_host_write_mcl(const char *path, const uint64_t *code, const uint32_t *v5, const int64_t *label, int64_t n);
/* `_db.npz` interop (dump :243-261, load_on_disk :289-335): lay (key, val, count) entries out as the
 * slot arrays of the reference's `oakht` (prime capacity, FNV-1a over the low 4 key bytes, quadratic
 * probing) so that `kmer_numba.py -d` can read a GPU-built dBG.  pg_host_oakht_capacity = the capacity
 * the reference's own table reaches after that many distinct keys. */
int64_t pg_host_oakht_capacity(int64_t n_entries);
int pg_host_build_oakht(const uint64_t *keys, const uint16_t *vals, const uint8_t *cnts, int64_t n, int64_t cap,
                        uint64_t *okeys, uint16_t *ovals, uint8_t *ocnts);
/* The same image on the GPU (npz_dump.cu).
 * pg_oakht_place: device entries d_keys/d_vals/d_cnts[n] (distinct keys, e.g. pg_table_export's) ->
 *   d_okeys/d_ovals/d_ocnts[cap] (cap = pg_host_oakht_capacity(n)).  Placement in rounds: in round s every
 *   unplaced entry bids for its s-th probe slot of oakht.pointer() if no earlier round took it, the
 *   smallest key wins; the sentinel key 2^64-1 takes its first probe slot before round 0.  The image
 *   depends only on the set of entries (it is not the host's insertion-order arrangement); every key is
 *   found by pointer(), empty slots hold key 0, value 0, count 0, live slots count >= 1.  d_ws: at least
 *   pg_oakht_place_workspace_bytes(n).  Synchronises the stream every few rounds to read the number of
 *   entries left; PG_ERR_CAPACITY when some are still unplaced after 4096 rounds.
 * pg_deflate_chunks: raw DEFLATE of chunks [first_chunk, first_chunk + n_chunks) of one member whose bytes
 *   are the HOST header hdr[hdr_len] (hdr_len <= PG_DEFLATE_HDR_MAX: the .npy header) followed by the
 *   device array d_data[data_len], cut into chunks of chunk_bytes (<= 65535).  Chunk first_chunk + i goes
 *   to d_staging + i * slot_bytes (slot_bytes >= pg_deflate_slot_bytes(chunk_bytes), a multiple of 16);
 *   d_sizes[i] = its compressed size, d_crcs[i] = the CRC-32 of its input.  Chunks are independent and
 *   byte-aligned; only the member's last chunk sets BFINAL, so the chunks in order form one raw-DEFLATE
 *   stream.  One CTA per chunk (csrc/deflate.cuh, which the CPU test harness compiles too).
 * pg_deflate_compact: after pg_deflate_chunks on the same slab: d_sizes[0, n_chunks) -> exclusive offsets,
 *   d_sizes[n_chunks] = the slab's compressed bytes (d_sizes holds n_chunks + 1 entries); the slots are
 *   copied to d_out at those offsets.  d_state[0]: in, the CRC-32 of the member's bytes before this slab
 *   (0 for the first); out, including it.  d_state[1] = the slab's compressed bytes.  total_bytes =
 *   hdr_len + data_len of the member. */
#define PG_DEFLATE_HDR_MAX 256
int pg_oakht_place(const uint64_t *d_keys, const uint16_t *d_vals, const uint8_t *d_cnts, int64_t n, int64_t cap,
                   uint64_t *d_okeys, uint16_t *d_ovals, uint8_t *d_ocnts, void *d_ws, int64_t ws_bytes, pg_stream_t stream);
int64_t pg_oakht_place_workspace_bytes(int64_t n);
int64_t pg_deflate_slot_bytes(int64_t chunk_bytes);
int pg_deflate_chunks(const uint8_t *hdr, int64_t hdr_len, const uint8_t *d_data, int64_t data_len, int64_t chunk_bytes,
                      int64_t first_chunk, int64_t n_chunks, uint8_t *d_staging, int64_t slot_bytes, int64_t *d_sizes,
                      uint32_t *d_crcs, pg_stream_t stream);
int pg_deflate_compact(const uint8_t *d_staging, int64_t slot_bytes, int64_t *d_sizes, const uint32_t *d_crcs,
                       int64_t first_chunk, int64_t n_chunks, int64_t chunk_bytes, int64_t total_bytes, uint8_t *d_out,
                       int64_t *d_state, pg_stream_t stream);

/* ---- measurement support (SURVEY.md 8d: "a micro-benchmark ceiling (random atomicCAS + atomicOr into a table of the
 * same byte size)") - not part of the hot path.  n_ops operations, each on one pseudo-random 16-byte slot; the regions
 * (region_slots slots each) are swept in order by the whole grid like pg_insert_records does.  mode: 0 load, 1 load +
 * red.add, 2 load + cas.b128, 3 the config-2 mix (1/3 cas, 2/3 red), 4 red only, 5 load + red.or + red.add; +8 also
 * streams one 16-byte record per operation from d_records; ilp = 1, 2, 4 or 8 independent operations in flight per
 * thread.  Overwrites the slots. */
int pg_microbench_slots(uint64_t *d_slots, int64_t capacity, int64_t region_slots, int64_t n_ops, int mode, int ctas_per_sm,
                        int ilp, const uint64_t *d_records, uint64_t *d_sink, pg_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PGDBG_H */
