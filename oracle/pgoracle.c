/*
 * pgoracle.c - CPU restatement of the reference's de Bruijn-graph hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  This file is the *checker* for the CUDA path in
 * pangenome_b200/csrc; nothing the product ships links, imports or calls it.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may use it.
 *
 * Parity status: PINNED for the dBG (key,val,count) set, the rdBG key set, the
 * edge list (order + weights) and the region rows - checked against the
 * reference's own numba code run in this container (oracle/refrun.py,
 * fixtures under tests/golden/).  UNPINNED for cluster membership: the
 * reference delegates that to the third-party `mcl` binary (not vendored, no
 * version pinned; call site kmer_numba.py:1911).  Components here are plain
 * undirected connected components of the edge list, the definition of the
 * reference's helper other/test_net.py:3-12; cluster order = decreasing size,
 * ties by smallest (code, v5).
 *
 * Every function cites the lines of /root/reference/kmer_numba.py it follows.
 * Quirk labels Q1..Q12 are defined in SURVEY.md App. A.  "Zero-memory
 * semantics": empty table slots hold key 0 / value 0 (patch 5 of
 * oracle/make_ref.py), which keeps Q6 (key 0 is always "present") and drops
 * the allocator noise Q10.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>
#include <time.h>

#define MINUS_ONE 0xFFFFFFFFFFFFFFFFull

/* ---- character tables -------------------------------------------------- */
static int8_t ALPHA[256];  /* kmer_numba.py:763-768  a0 g1 c2 t3 else 4   */
static int8_t LASTC[256];  /* kmer_numba.py:736-743  A1 T2 G4 C8 N16 $32  */
static uint8_t COMP[256];  /* kmer_numba.py:191-195  A<->T G<->C else N   */
static int tables_ready = 0;

static void init_tables(void) {
    if (tables_ready) return;
    for (int i = 0; i < 256; i++) { ALPHA[i] = 4; LASTC[i] = 0; COMP[i] = 'N'; }
    ALPHA['a'] = ALPHA['A'] = 0; ALPHA['t'] = ALPHA['T'] = 3;
    ALPHA['g'] = ALPHA['G'] = 1; ALPHA['c'] = ALPHA['C'] = 2;
    LASTC['a'] = LASTC['A'] = 1; LASTC['t'] = LASTC['T'] = 2;
    LASTC['g'] = LASTC['G'] = 4; LASTC['c'] = LASTC['C'] = 8;
    LASTC['n'] = LASTC['N'] = 16; LASTC['$'] = 32; LASTC['#'] = 0;
    COMP['A'] = COMP['a'] = 'T'; COMP['T'] = COMP['t'] = 'A';
    COMP['G'] = COMP['g'] = 'C'; COMP['C'] = COMP['c'] = 'G';
    COMP['N'] = COMP['n'] = 'N';
    tables_ready = 1;
}

/* ---- growable arrays --------------------------------------------------- */
#define VEC(T, name) typedef struct { T *p; int64_t n, cap; } name
VEC(uint8_t, vec_u8); VEC(int64_t, vec_i64); VEC(uint64_t, vec_u64);
VEC(int32_t, vec_i32);
#define VPUSH(v, x) do { if ((v).n == (v).cap) { (v).cap = (v).cap ? (v).cap * 2 : 64; \
    (v).p = realloc((v).p, (size_t)(v).cap * sizeof(*(v).p)); } (v).p[(v).n++] = (x); } while (0)

/* ---- oakht (kmer_numba.py:340-679), ksize = vsize = 1 ------------------- */
typedef struct {
    int64_t capacity, size;
    float load;            /* spec['load'] = float32, kmer_numba.py:1101 */
    uint64_t *keys; uint16_t *values; uint8_t *counts;
    int64_t n_probe;       /* statistics only */
} oakht;

static int isprime(int64_t n) {            /* :356-366 */
    if (n <= 1 || n % 2 == 0 || n % 3 == 0) return 0;
    for (int64_t i = 5; i * i <= n; i += 6)
        if (n % i == 0 || n % (i + 2) == 0) return 0;
    return 1;
}
static int64_t find_prime(int64_t n) {     /* :369-372 */
    for (int64_t i = n;; i++) if (isprime(i)) return i;
}
static uint64_t fnv4(uint64_t val) {        /* :400-411, ksize==1 branch: low 4 bytes only */
    uint64_t a = 0xcbf29ce484222325ull;
    for (int i = 0; i < 4; i++) { a ^= (val & 0xff); a *= 0x100000001b3ull; val >>= 8; }
    return a;
}
/* first probe slot: the reference hashes in int64 and numba's % is Python's floor modulo, so a hash with bit 63 set
   starts at (signed hash) mod M, not at the unsigned remainder */
static int64_t oakht_slot0(uint64_t key, int64_t M) {
    int64_t j = (int64_t)fnv4(key) % M;
    return j < 0 ? j + M : j;
}
static void oakht_init(oakht *h) {          /* :341-352; init_dict ignores `capacity` (:1121) */
    h->capacity = find_prime(1 << 20);
    h->load = 0.75f; h->size = 0; h->n_probe = 0;
    h->keys = calloc((size_t)h->capacity, 8);     /* zero-memory semantics */
    h->values = calloc((size_t)h->capacity, 2);
    h->counts = calloc((size_t)h->capacity, 1);
}
static void oakht_free(oakht *h) { free(h->keys); free(h->values); free(h->counts); memset(h, 0, sizeof *h); }

static int64_t oakht_pointer(oakht *h, uint64_t key) {   /* :521-538 */
    int64_t M = h->capacity;
    int64_t j = oakht_slot0(key, M), j_init = j;
    for (int64_t k = 0; k < M; k++) {
        if (h->keys[j] == key || h->counts[j] == 0) break;   /* equality tested BEFORE occupancy: Q6 */
        j = (j_init + k * k) % M;
    }
    return j;
}
static void oakht_resize(oakht *h) {        /* :423-474 */
    int64_t N = h->capacity;
    int64_t M = find_prime((int64_t)((double)N * 1.62));
    uint64_t *keys = calloc((size_t)M, 8); uint16_t *values = calloc((size_t)M, 2); uint8_t *counts = calloc((size_t)M, 1);
    for (int64_t i = 0; i < N; i++) {
        if (h->counts[i] == 0) continue;
        int64_t j = oakht_slot0(h->keys[i], M), j_init = j;
        for (int64_t k = 0; k < N; k++) {
            if (counts[j] == 0 || keys[j] == h->keys[i]) break;
            j = (j_init + k * k) % M;
        }
        keys[j] = h->keys[i]; values[j] = h->values[i]; counts[j] = h->counts[i];
    }
    free(h->keys); free(h->values); free(h->counts);
    h->keys = keys; h->values = values; h->counts = counts; h->capacity = M;
}
static void oakht_push(oakht *h, uint64_t key, uint16_t value) {   /* __setitem__ :540-561 */
    int64_t j = oakht_pointer(h, key);
    if (h->counts[j] == 0) { h->size += 1; h->keys[j] = key; }
    h->values[j] = value;
    h->counts[j] = (uint8_t)(h->counts[j] + 1 < 255 ? h->counts[j] + 1 : 255);
    double lfr = (double)h->size * 1.0 / (double)h->capacity;
    if (lfr > (double)h->load) oakht_resize(h);
}
static int oakht_has_key(oakht *h, uint64_t key) {       /* :599-603 - no occupancy test (Q6) */
    int64_t j = oakht_pointer(h, key);
    return h->keys[j] == key;
}
static uint16_t oakht_get(oakht *h, uint64_t key) {      /* :566-575 */
    int64_t j = oakht_pointer(h, key);
    return h->values[j];
}

/* ---- A1 records: readline_jit_ :122-132 + seqio_jit_ :135-168 ----------- */
typedef struct {
    int64_t n_rec;
    vec_i64 hdr_off, hdr_len;   /* header line without its last byte (includes '>') */
    vec_i64 seq_off;            /* n_rec+1 offsets into seq */
    vec_u8 seq;                 /* concatenated record sequences */
} records;

static void rec_line(records *R, const uint8_t *b, int64_t st, int64_t ed, int *have_hdr) {
    if (b[st] == 62) {                      /* '>' : close the open record, start a new one */
        if (*have_hdr) VPUSH(R->seq_off, R->seq.n);
        else R->seq.n = 0;                  /* bytes before the first header are dropped (start=end=0 reset) */
        VPUSH(R->hdr_off, st); VPUSH(R->hdr_len, ed - st - 1);
        if (!*have_hdr) { R->seq_off.n = 0; VPUSH(R->seq_off, 0); }
        *have_hdr = 1;
    } else {
        for (int64_t i = st; i < ed - 1; i++) VPUSH(R->seq, b[i]);   /* line[:-1] */
    }
}
static void parse_records(records *R, const uint8_t *b, int64_t n, int64_t offset) {
    memset(R, 0, sizeof *R);
    int have_hdr = 0;
    int64_t start = 0, end = 0;
    for (end = offset; end < n; end++) {
        if (b[end] == 10) { rec_line(R, b, start, end + 1, &have_hdr); start = end + 1; }
    }
    end = (n > offset) ? n - 1 : 0;          /* python loop variable after the loop */
    if (end > start && start > 0) rec_line(R, b, start, end + 1, &have_hdr);   /* Q8: last byte is still dropped */
    if (have_hdr) VPUSH(R->seq_off, R->seq.n);
    else { R->seq.n = 0; VPUSH(R->seq_off, 0); }
    R->n_rec = R->hdr_off.n;
}
static void records_free(records *R) { free(R->hdr_off.p); free(R->hdr_len.p); free(R->seq_off.p); free(R->seq.p); }

static void reverse_strand(const uint8_t *s, int64_t n, uint8_t *out) {   /* reverse_jit_ :197-204 */
    for (int64_t i = 0; i < n; i++) out[i] = COMP[s[n - 1 - i]];
}

/* ---- A3 occurrences: build_dbg :1052-1090 == seq2ns_jit_ :991-1033 ------- */
typedef void (*occ_fn)(void *ctx, int64_t idx, uint64_t code, int hd, int nt);

static uint64_t k2n(const uint8_t *s, int k) {           /* k2n_jit :975-985 */
    uint64_t N = 0, p = 1;
    for (int i = 0; i < k; i++) { N += (uint64_t)ALPHA[s[i]] * p; p *= 5; }
    return N;
}
static int64_t g_ub_count = 0;   /* records with n == k+1 (Q2: undefined in the reference) */

static void occurrences(const uint8_t *t, int64_t n, int k, occ_fn fn, void *ctx) {
    if (n > k) {
        uint64_t Nu = k2n(t, k);
        fn(ctx, 0, Nu, 35, t[k]);                                    /* '#' */
        uint64_t shift = 1; for (int i = 0; i < k - 1; i++) shift *= 5;
        int64_t i, idx = 1;
        for (i = k; i < n - 1; i++) {
            Nu = Nu / 5 + (uint64_t)ALPHA[t[i]] * shift;
            fn(ctx, idx, Nu, t[i - k], t[i + 1]);
            idx++;
        }
        /* after the loop the reference reuses the loop variable: i == n-2 (Q1) */
        int hd;
        if (n >= k + 2) { i = n - 2; hd = t[i - k]; }
        else { i = k - 1; hd = t[0]; g_ub_count++; }                 /* Q2: n == k+1 is UB upstream; sane value here */
        Nu = Nu / 5 + (uint64_t)ALPHA[t[i + 1]] * shift;
        fn(ctx, idx, Nu, hd, 36);                                    /* '$' */
    } else if (n == k) {
        fn(ctx, 0, k2n(t, k), 35, 36);
    } else {
        fn(ctx, 0, MINUS_ONE, 35, 36);                               /* Q5 short-record sentinel */
    }
}

/* ---- A4 dBG: add_kmer :1036-1047 --------------------------------------- */
typedef struct { oakht *h; int64_t n_ins; } dbg_ctx;
static void add_kmer(void *vctx, int64_t idx, uint64_t Nu, int hd, int nt) {
    (void)idx;
    dbg_ctx *c = vctx;
    uint16_t h = (uint16_t)(LASTC[hd] << 6), d = (uint16_t)LASTC[nt];
    if (oakht_has_key(c->h, Nu)) {
        uint16_t val = oakht_get(c->h, Nu);
        oakht_push(c->h, Nu, val | h | d);
    } else {
        oakht_push(c->h, Nu, h | d);
    }
    c->n_ins++;
}

/* ---- result object ------------------------------------------------------ */
typedef struct {
    records R;
    /* stage 1 */
    oakht dbg; int64_t dbg_n; uint64_t *dbg_keys; uint16_t *dbg_vals; uint8_t *dbg_cnts; int64_t n_ins;
    /* stage 2 */
    oakht rdbg; int64_t rdbg_n; uint64_t *rdbg_keys; uint16_t *rdbg_vals;
    /* stage 3: edges in first-insertion order */
    vec_u64 e_c0, e_v0, e_c1, e_v1; vec_i64 e_w;
    /* nodes + labels */
    int64_t n_nodes; uint64_t *node_code; uint64_t *node_v; int64_t *node_label; int64_t n_comp;
    /* rows */
    vec_i64 row_rec, row_st, row_ed, row_lab; vec_i32 row_strand;
    int64_t ub_count;
    double t_dbg, t_rdbg, t_edge, t_label;
} pgo_result;

static double now(void) { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + ts.tv_nsec * 1e-9; }

/* seq2dbg_jit_ :1202-1230 driven by seq2rdbg :1234-1268 (chunk checkpoints do not change the table) */
static void stage_dbg(pgo_result *r, int k, int rc, uint64_t Ns) {
    oakht_init(&r->dbg);
    dbg_ctx c = { &r->dbg, 0 };
    uint64_t N = 0; uint8_t *rv = NULL; int64_t rvcap = 0;
    for (int64_t i = 0; i < r->R.n_rec; i++) {
        const uint8_t *s = r->R.seq.p + r->R.seq_off.p[i];
        int64_t n = r->R.seq_off.p[i + 1] - r->R.seq_off.p[i];
        occurrences(s, n, k, add_kmer, &c);
        N += (uint64_t)n;
        if (rc) {
            if (n > rvcap) { rvcap = n; rv = realloc(rv, (size_t)n + 1); }
            reverse_strand(s, n, rv);
            occurrences(rv, n, k, add_kmer, &c);
            N += (uint64_t)n;
        }
        if (N > Ns) break;
    }
    free(rv);
    r->n_ins = c.n_ins;
}

static int cmp_u64(const void *a, const void *b) { uint64_t x = *(const uint64_t *)a, y = *(const uint64_t *)b; return x < y ? -1 : x > y; }

static int64_t export_sorted(oakht *h, uint64_t **keys, uint16_t **vals, uint8_t **cnts) {
    /* iteritems :623-631 (live = counts > 0), then canonical ascending key order */
    int64_t n = 0;
    for (int64_t i = 0; i < h->capacity; i++) n += h->counts[i] > 0;
    uint64_t *idx = malloc((size_t)(n ? n : 1) * 16);
    int64_t m = 0;
    for (int64_t i = 0; i < h->capacity; i++) if (h->counts[i] > 0) { idx[2 * m] = h->keys[i]; idx[2 * m + 1] = (uint64_t)i; m++; }
    qsort(idx, (size_t)n, 16, cmp_u64);
    *keys = malloc((size_t)(n ? n : 1) * 8); *vals = malloc((size_t)(n ? n : 1) * 2);
    if (cnts) *cnts = malloc((size_t)(n ? n : 1));
    for (int64_t i = 0; i < n; i++) {
        int64_t s = (int64_t)idx[2 * i + 1];
        (*keys)[i] = h->keys[s]; (*vals)[i] = h->values[s]; if (cnts) (*cnts)[i] = h->counts[s];
    }
    free(idx);
    return n;
}

static int nbit(unsigned x) { return __builtin_popcount(x); }   /* nbit :723-725 */

/* build_rdbg_jit_ :1292-1309 */
static void stage_rdbg(pgo_result *r) {
    oakht_init(&r->rdbg);
    oakht *d = &r->dbg;
    for (int64_t i = 0; i < d->capacity; i++) {
        if (d->counts[i] == 0) continue;
        unsigned hn = d->values[i];
        int pr = nbit(hn >> 6), sf = nbit(hn & 63);
        if (pr == 1 && sf == 1) continue;           /* `sf != 0b100000` is always true (Q12) */
        oakht_push(&r->rdbg, d->keys[i], d->values[i]);
    }
}

/* ---- A6 edges: rdbg_edge_weight :1446-1518 ------------------------------ */
typedef struct { uint64_t c0, v0, c1, v1; } ekey;
typedef struct {
    pgo_result *r;
    int64_t *slot; int64_t cap;            /* open-addressing index over the edge arrays (typed Dict stand-in) */
    vec_i64 last_seen;                     /* per edge: id of the last record-strand that counted it (= `visit`) */
    int64_t cur_id;
    uint64_t n0, v0; int have0;
    int offbit;
} edge_ctx;

static uint64_t mix64(uint64_t x) { x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33; return x; }
static uint64_t ehash(const ekey *e) { return mix64(e->c0 ^ mix64(e->c1 + 0x9e3779b97f4a7c15ull) ^ mix64((e->v0 << 16) ^ e->v1 ^ 0x1234567ull)); }

static void edge_grow(edge_ctx *c) {
    int64_t ncap = c->cap ? c->cap * 2 : 1024;
    int64_t *ns = malloc((size_t)ncap * 8);
    for (int64_t i = 0; i < ncap; i++) ns[i] = -1;
    pgo_result *r = c->r;
    for (int64_t e = 0; e < r->e_c0.n; e++) {
        ekey k = { r->e_c0.p[e], r->e_v0.p[e], r->e_c1.p[e], r->e_v1.p[e] };
        uint64_t j = ehash(&k) & (uint64_t)(ncap - 1);
        while (ns[j] >= 0) j = (j + 1) & (uint64_t)(ncap - 1);
        ns[j] = e;
    }
    free(c->slot); c->slot = ns; c->cap = ncap;
}
static void edge_add(edge_ctx *c, const ekey *k) {
    pgo_result *r = c->r;
    if ((r->e_c0.n + 1) * 2 > c->cap) edge_grow(c);
    uint64_t j = ehash(k) & (uint64_t)(c->cap - 1);
    for (;;) {
        int64_t e = c->slot[j];
        if (e < 0) {
            c->slot[j] = r->e_c0.n;
            VPUSH(r->e_c0, k->c0); VPUSH(r->e_v0, k->v0); VPUSH(r->e_c1, k->c1); VPUSH(r->e_v1, k->v1);
            VPUSH(r->e_w, 1); VPUSH(c->last_seen, c->cur_id);
            return;
        }
        if (r->e_c0.p[e] == k->c0 && r->e_v0.p[e] == k->v0 && r->e_c1.p[e] == k->c1 && r->e_v1.p[e] == k->v1) {
            if (c->last_seen.p[e] != c->cur_id) { c->last_seen.p[e] = c->cur_id; r->e_w.p[e] += 1; }   /* `visit` :1479-1484 */
            return;
        }
        j = (j + 1) & (uint64_t)(c->cap - 1);
    }
}
static void edge_occ(void *vctx, int64_t idx, uint64_t code, int hd, int nt) {
    (void)idx;
    edge_ctx *c = vctx;
    if (code == MINUS_ONE) return;                          /* :1461 */
    if (!oakht_has_key(&c->r->rdbg, code)) return;          /* :1465, includes phantom key 0 (Q6) */
    uint64_t v = ((uint64_t)LASTC[hd] << c->offbit) | (uint64_t)LASTC[nt];   /* offbit == 5 at head (Q7 / F7) */
    if (!c->have0) { c->n0 = code; c->v0 = v; c->have0 = 1; return; }
    ekey k = { c->n0, c->v0, code, v };
    edge_add(c, &k);
    c->n0 = code; c->v0 = v;
}
/* rdbg_edge_weight_jit_ :1808-1827 */
static void stage_edges(pgo_result *r, int k, int rc, uint64_t Ns, int offbit) {
    edge_ctx c; memset(&c, 0, sizeof c); c.r = r; c.offbit = offbit;
    uint64_t N = 0; uint8_t *rv = NULL; int64_t rvcap = 0;
    for (int64_t i = 0; i < r->R.n_rec; i++) {
        const uint8_t *s = r->R.seq.p + r->R.seq_off.p[i];
        int64_t n = r->R.seq_off.p[i + 1] - r->R.seq_off.p[i];
        c.cur_id++; c.have0 = 0;
        occurrences(s, n, k, edge_occ, &c);
        if (rc) {
            if (n > rvcap) { rvcap = n; rv = realloc(rv, (size_t)n + 1); }
            reverse_strand(s, n, rv);
            c.cur_id++; c.have0 = 0;
            occurrences(rv, n, k, edge_occ, &c);
        }
        N += (uint64_t)n;
        if (N > Ns) break;
    }
    free(rv); free(c.slot); free(c.last_seen.p);
}

/* ---- A7 labels: connected components stand-in for mcl + label_dct :1918-1944 */
typedef struct { uint64_t code, v; int64_t id; } nodeent;
static int cmp_node(const void *a, const void *b) {
    const nodeent *x = a, *y = b;
    if (x->code != y->code) return x->code < y->code ? -1 : 1;
    if (x->v != y->v) return x->v < y->v ? -1 : 1;
    return 0;
}
static int64_t uf_find(int64_t *p, int64_t x) { while (p[x] != x) { p[x] = p[p[x]]; x = p[x]; } return x; }
typedef struct { int64_t size, minnode, root; } compent;
static int cmp_comp(const void *a, const void *b) {
    const compent *x = a, *y = b;
    if (x->size != y->size) return x->size > y->size ? -1 : 1;
    return x->minnode < y->minnode ? -1 : x->minnode > y->minnode;
}
static int64_t node_lookup(const pgo_result *r, uint64_t code, uint64_t v) {
    int64_t lo = 0, hi = r->n_nodes;
    while (lo < hi) {
        int64_t mid = (lo + hi) / 2;
        if (r->node_code[mid] < code || (r->node_code[mid] == code && r->node_v[mid] < v)) lo = mid + 1; else hi = mid;
    }
    if (lo < r->n_nodes && r->node_code[lo] == code && r->node_v[lo] == v) return lo;
    return -1;
}
static void stage_labels(pgo_result *r) {
    int64_t E = r->e_c0.n;
    nodeent *tmp = malloc((size_t)(2 * E + 1) * sizeof(nodeent));
    for (int64_t e = 0; e < E; e++) {
        tmp[2 * e] = (nodeent){ r->e_c0.p[e], r->e_v0.p[e], 0 };
        tmp[2 * e + 1] = (nodeent){ r->e_c1.p[e], r->e_v1.p[e], 0 };
    }
    qsort(tmp, (size_t)(2 * E), sizeof(nodeent), cmp_node);
    int64_t n = 0;
    for (int64_t i = 0; i < 2 * E; i++) if (i == 0 || cmp_node(&tmp[i], &tmp[i - 1]) != 0) tmp[n++] = tmp[i];
    r->n_nodes = n;
    r->node_code = malloc((size_t)(n + 1) * 8); r->node_v = malloc((size_t)(n + 1) * 8); r->node_label = malloc((size_t)(n + 1) * 8);
    for (int64_t i = 0; i < n; i++) { r->node_code[i] = tmp[i].code; r->node_v[i] = tmp[i].v; }
    free(tmp);
    int64_t *par = malloc((size_t)(n + 1) * 8);
    for (int64_t i = 0; i < n; i++) par[i] = i;
    for (int64_t e = 0; e < E; e++) {
        int64_t a = uf_find(par, node_lookup(r, r->e_c0.p[e], r->e_v0.p[e]));
        int64_t b = uf_find(par, node_lookup(r, r->e_c1.p[e], r->e_v1.p[e]));
        if (a != b) par[a > b ? a : b] = a > b ? b : a;     /* root = smallest node index */
    }
    int64_t *csize = calloc((size_t)(n + 1), 8);
    for (int64_t i = 0; i < n; i++) csize[uf_find(par, i)]++;
    compent *comps = malloc((size_t)(n + 1) * sizeof(compent));
    int64_t nc = 0;
    for (int64_t i = 0; i < n; i++) if (par[i] == i) comps[nc++] = (compent){ csize[i], i, i };
    qsort(comps, (size_t)nc, sizeof(compent), cmp_comp);
    int64_t *lab_of_root = csize;   /* reuse */
    for (int64_t c = 0; c < nc; c++) lab_of_root[comps[c].root] = c;
    for (int64_t i = 0; i < n; i++) r->node_label[i] = lab_of_root[uf_find(par, i)];
    r->n_comp = nc;
    free(par); free(csize); free(comps);
}

/* ---- A8 regions: seq2path_jit_ :1523-1573, seqs2path_jit_ :1830-1849 ----- */
typedef struct {
    pgo_result *r; int k;
    vec_i64 starts, labels;
} path_ctx;
static void path_occ(void *vctx, int64_t idx, uint64_t code, int hd, int nt) {
    path_ctx *c = vctx;
    uint64_t v6 = ((uint64_t)LASTC[hd] << 6) | (uint64_t)LASTC[nt];     /* offbit 6 here (Q7) */
    if (code == MINUS_ONE) return;            /* (-1, 32) is never a label_dct key */
    int64_t j = node_lookup(c->r, code, v6);  /* `kk in label_dct` :1549 */
    if (j < 0) return;
    int64_t label = c->r->node_label[j];
    if (c->starts.p[c->starts.n - 1] < idx) {
        int64_t pos = idx + c->k;
        if (c->labels.p[c->labels.n - 1] != label) { VPUSH(c->labels, label); VPUSH(c->starts, pos); }
        else c->starts.p[c->starts.n - 1] = pos;
    }
}
static void stage_paths(pgo_result *r, int k, int rc, uint64_t Ns) {
    path_ctx c; memset(&c, 0, sizeof c); c.r = r; c.k = k;
    uint64_t N = 0; uint8_t *rv = NULL; int64_t rvcap = 0;
    for (int64_t i = 0; i < r->R.n_rec; i++) {
        const uint8_t *s = r->R.seq.p + r->R.seq_off.p[i];
        int64_t n = r->R.seq_off.p[i + 1] - r->R.seq_off.p[i];
        for (int strand = 0; strand < (rc ? 2 : 1); strand++) {
            c.starts.n = 0; c.labels.n = 0; VPUSH(c.starts, 0); VPUSH(c.labels, -1);
            if (strand == 0) occurrences(s, n, k, path_occ, &c);
            else {
                if (n > rvcap) { rvcap = n; rv = realloc(rv, (size_t)n + 1); }
                reverse_strand(s, n, rv);
                occurrences(rv, n, k, path_occ, &c);
            }
            for (int64_t j = 1; j < c.starts.n; j++) {
                int64_t st = c.starts.p[j - 1], ed = c.starts.p[j];
                VPUSH(r->row_rec, i); VPUSH(r->row_lab, c.labels.p[j]);
                if (strand == 0) { VPUSH(r->row_st, st); VPUSH(r->row_ed, ed); VPUSH(r->row_strand, 1); }
                else { VPUSH(r->row_st, n - ed); VPUSH(r->row_ed, n - st); VPUSH(r->row_strand, -1); }   /* :1843-1844 */
            }
        }
        N += (uint64_t)n;
        if (N > Ns) break;
    }
    free(rv); free(c.starts.p); free(c.labels.p);
}

/* ---- public C API (ctypes) ---------------------------------------------- */
/* stages: 1 = dBG only, 2 = + rdBG, 3 = + edges, 4 = + labels and rows.
 * c_flags: the reference's -c (bit1 = rc in dBG stage, bit0 = rc in edge/path stages) :2110,2141.
 * path_offset: seqs2path_jit_ passes isfasta (=1) in the offset slot :1833.
 * edge_offbit: 5 reproduces the head version (F7); 6 the older variants. */
pgo_result *pgo_run(const uint8_t *fasta, int64_t n, int k, int c_flags, uint64_t Ns, int stages, int edge_offbit) {
    init_tables();
    if (k < 1) k = 1;
    if (k > 27) k = 27;                      /* :1236, :1855 */
    pgo_result *r = calloc(1, sizeof *r);
    g_ub_count = 0;
    parse_records(&r->R, fasta, n, 0);
    double t0 = now();
    stage_dbg(r, k, (c_flags >> 1) & 1, Ns);
    r->t_dbg = now() - t0;
    r->dbg_n = export_sorted(&r->dbg, &r->dbg_keys, &r->dbg_vals, &r->dbg_cnts);
    if (stages >= 2) {
        t0 = now(); stage_rdbg(r); r->t_rdbg = now() - t0;
        r->rdbg_n = export_sorted(&r->rdbg, &r->rdbg_keys, &r->rdbg_vals, NULL);
    }
    if (stages >= 3) { t0 = now(); stage_edges(r, k, c_flags & 1, Ns, edge_offbit); r->t_edge = now() - t0; }
    if (stages >= 4) {
        t0 = now();
        stage_labels(r);
        if (n > 0 && fasta[0] == 10) {       /* offset=1 quirk: a leading blank line hides the first header */
            records_free(&r->R); parse_records(&r->R, fasta, n, 1);
        }
        stage_paths(r, k, c_flags & 1, Ns);
        r->t_label = now() - t0;
    }
    r->ub_count = g_ub_count;
    return r;
}

void pgo_free(pgo_result *r) {
    if (!r) return;
    records_free(&r->R);
    if (r->dbg.keys) oakht_free(&r->dbg);
    if (r->rdbg.keys) oakht_free(&r->rdbg);
    free(r->dbg_keys); free(r->dbg_vals); free(r->dbg_cnts); free(r->rdbg_keys); free(r->rdbg_vals);
    free(r->e_c0.p); free(r->e_v0.p); free(r->e_c1.p); free(r->e_v1.p); free(r->e_w.p);
    free(r->node_code); free(r->node_v); free(r->node_label);
    free(r->row_rec.p); free(r->row_st.p); free(r->row_ed.p); free(r->row_lab.p); free(r->row_strand.p);
    free(r);
}

int64_t pgo_n_records(const pgo_result *r) { return r->R.n_rec; }
const int64_t *pgo_hdr_off(const pgo_result *r) { return r->R.hdr_off.p; }
const int64_t *pgo_hdr_len(const pgo_result *r) { return r->R.hdr_len.p; }
const int64_t *pgo_seq_off(const pgo_result *r) { return r->R.seq_off.p; }
const uint8_t *pgo_seq(const pgo_result *r) { return r->R.seq.p; }
int64_t pgo_n_inserts(const pgo_result *r) { return r->n_ins; }
int64_t pgo_ub_count(const pgo_result *r) { return r->ub_count; }
int64_t pgo_dbg_size(const pgo_result *r) { return r->dbg_n; }
const uint64_t *pgo_dbg_keys(const pgo_result *r) { return r->dbg_keys; }
const uint16_t *pgo_dbg_vals(const pgo_result *r) { return r->dbg_vals; }
const uint8_t *pgo_dbg_cnts(const pgo_result *r) { return r->dbg_cnts; }
/* raw oakht image of the dBG, slot order as the reference lays it out (for _db.npz interop) */
int64_t pgo_dbg_capacity(const pgo_result *r) { return r->dbg.capacity; }
const uint64_t *pgo_dbg_slot_keys(const pgo_result *r) { return r->dbg.keys; }
const uint16_t *pgo_dbg_slot_vals(const pgo_result *r) { return r->dbg.values; }
const uint8_t *pgo_dbg_slot_cnts(const pgo_result *r) { return r->dbg.counts; }
int64_t pgo_rdbg_size(const pgo_result *r) { return r->rdbg_n; }
const uint64_t *pgo_rdbg_keys(const pgo_result *r) { return r->rdbg_keys; }
const uint16_t *pgo_rdbg_vals(const pgo_result *r) { return r->rdbg_vals; }
int64_t pgo_n_edges(const pgo_result *r) { return r->e_c0.n; }
const uint64_t *pgo_edge_c0(const pgo_result *r) { return r->e_c0.p; }
const uint64_t *pgo_edge_v0(const pgo_result *r) { return r->e_v0.p; }
const uint64_t *pgo_edge_c1(const pgo_result *r) { return r->e_c1.p; }
const uint64_t *pgo_edge_v1(const pgo_result *r) { return r->e_v1.p; }
const int64_t *pgo_edge_w(const pgo_result *r) { return r->e_w.p; }
int64_t pgo_n_nodes(const pgo_result *r) { return r->n_nodes; }
int64_t pgo_n_components(const pgo_result *r) { return r->n_comp; }
const uint64_t *pgo_node_code(const pgo_result *r) { return r->node_code; }
const uint64_t *pgo_node_v(const pgo_result *r) { return r->node_v; }
const int64_t *pgo_node_label(const pgo_result *r) { return r->node_label; }
int64_t pgo_n_rows(const pgo_result *r) { return r->row_rec.n; }
const int64_t *pgo_row_rec(const pgo_result *r) { return r->row_rec.p; }
const int64_t *pgo_row_start(const pgo_result *r) { return r->row_st.p; }
const int64_t *pgo_row_end(const pgo_result *r) { return r->row_ed.p; }
const int32_t *pgo_row_strand(const pgo_result *r) { return r->row_strand.p; }
const int64_t *pgo_row_label(const pgo_result *r) { return r->row_lab.p; }
double pgo_time(const pgo_result *r, int stage) { return stage == 1 ? r->t_dbg : stage == 2 ? r->t_rdbg : stage == 3 ? r->t_edge : r->t_label; }
