// table_dev.cuh - device-side pieces shared by the table kernels (dbg_table.cu) and the path kernels
// (path_graph.cu): slot upsert / lookup, record lookup, shared-memory staging of the packed stream.
#pragma once
#include "kmer_core.cuh"

constexpr int K2_THREADS = 256;                 // one 32-base word per thread
constexpr int K2_TILE_WORDS = K2_THREADS;       // 8192 bases per CTA tile
constexpr uint32_t PG_MAX_PROBE = 1u << 16;

// Home slot = TOP bits of the 64-bit mix: the high bits of a slot index are then hash bits too, so
// "region of the table" == "hash prefix" for every capacity (K2a buckets records by that prefix before
// the table is even sized); the owner rank of the multi-GPU split comes from the LOW bits instead.
// rmask: probing wraps inside the aligned block of rmask + 1 slots the home slot lies in (pg_table.region_bits; the
// whole table when 0), so a region of a table built in shared memory (region_build.cu) holds ALL the keys that hash into it.
// hmask: region tables round the home slot down to a group of PG_REGION_GROUP slots (K3s reads a whole group per probe
// step), so the linear-probing invariant "no free slot between home and the key" is stated from the group's first slot.
// Region semantics hold whenever 0 < region_bits <= log2(capacity): a table of exactly ONE region is built by K3s / K3s-c
// like any other, so every later upsert must start from the same group-aligned home (tests/test_table_geometry.py).
#define PG_REGION_GROUP 4
// hkind: which code the placement hash is taken of (pg_table.hash_kind): 0 = the base-5 key itself, 1 = its 2-bit form
// (tables built from compact records, compact_build.cu; generic upserts and look-ups then pay a base-5 -> 2-bit conversion)
struct TableView { uint64_t *slots; uint64_t capmask; int64_t *stats; int shift; uint64_t tag; uint64_t rmask; uint64_t hmask; int hkind; int k; };
__host__ __device__ __forceinline__ uint64_t tv_next(const TableView &t, uint64_t s) { return (s & ~t.rmask) | ((s + 1) & t.rmask); }
inline uint64_t pg_tag(const pg_table *t) { return (uint64_t)(uint32_t)t->epoch << PG_TAG_SHIFT; }
__host__ __device__ __forceinline__ uint64_t tv_home(const TableView &t, uint64_t key) {
    const uint64_t h = t.hkind ? pg_hash_kind1(key, t.k) : pg_mix64(key);
    return (h >> t.shift) & t.hmask;
}
inline TableView make_view(const pg_table *t) {
    int bits = 0; while ((1ll << bits) < t->capacity) bits++;
    const uint64_t capmask = (uint64_t)t->capacity - 1;
    const bool region = t->region_bits > 0 && t->region_bits <= bits;
    const uint64_t rmask = region ? ((1ull << t->region_bits) - 1ull) : capmask;
    const uint64_t hmask = region ? ~(uint64_t)(PG_REGION_GROUP - 1) : ~0ull;
    return TableView{t->d_slots, capmask, t->d_stats, 64 - bits, pg_tag(t), rmask, hmask, t->hash_kind ? 1 : 0, t->k};
}

// Merge one update into a slot whose key already matches; cv = the value word last seen.
__device__ __forceinline__ void slot_merge(uint64_t *p, uint64_t cv, uint32_t masks, uint32_t inc) {
    uint32_t *v = reinterpret_cast<uint32_t *>(p + 1);
    if (((uint32_t)cv & masks) != masks) pg_red_or32(v, masks);
    if ((uint32_t)(cv >> 32) < 255u) pg_red_add32(v + 1, inc);       // counts clamp at 255 upstream (:551)
}
// Continue an upsert from slot s whose raw contents (lo, hi) were already loaded.
// returns the slot index the key lives in (claimed if absent), or -1 when probing gives up
__device__ __forceinline__ int64_t table_upsert_from(const TableView &t, uint64_t s, uint64_t lo, uint64_t hi, uint64_t key,
                                                     uint32_t masks, uint32_t inc, uint32_t &n_claimed) {
    const uint32_t max_probe = t.rmask + 1 < PG_MAX_PROBE ? (uint32_t)(t.rmask + 1) : PG_MAX_PROBE;
    for (uint32_t probe = 0; probe < max_probe; probe++) {
        uint64_t *p = t.slots + 2 * s;
        if (probe) pg_ld_slot_raw(p, lo, hi);
        if ((hi & ~PG_VAL_MASK) != t.tag) {
            // not of this generation = free: replace whatever it holds by key + first masks + first count + tag
            // in ONE 128-bit CAS against the contents just seen
            uint64_t olo, ohi;
            pg_cas128(p, lo, hi, key, (uint64_t)masks | ((uint64_t)inc << 32) | t.tag, olo, ohi);
            if (olo == lo && ohi == hi) { n_claimed++; return (int64_t)s; }
            lo = olo; hi = ohi;              // lost the race: the slot is live now, look at its key
        }
        if (lo == key) { slot_merge(p, hi & PG_VAL_MASK, masks, inc); return (int64_t)s; }
        s = tv_next(t, s);
    }
    atomicExch(reinterpret_cast<unsigned long long *>(t.stats + PG_STAT_OVERFLOW), 1ull);
    return -1;
}
__device__ __forceinline__ int64_t table_upsert(const TableView &t, uint64_t key, uint32_t masks, uint32_t inc, uint32_t &n_claimed) {
    uint64_t s = tv_home(t, key), lo, hi;
    pg_ld_slot_raw(t.slots + 2 * s, lo, hi);
    return table_upsert_from(t, s, lo, hi, key, masks, inc, n_claimed);
}
// Store {key, val} whole (no masks/count semantics): claims a free slot, or ORs val into the slot that already
// holds the key.  Used where every key arrives once (K4) or arrives with its final value (gathered tables).
__device__ __forceinline__ bool table_put_or(const TableView &t, uint64_t key, uint64_t val) {
    uint64_t s = tv_home(t, key);
    for (uint32_t probe = 0; probe < PG_MAX_PROBE; probe++) {
        uint64_t *p = t.slots + 2 * s, lo, hi;
        pg_ld_slot_raw(p, lo, hi);
        if ((hi & ~PG_VAL_MASK) != t.tag) {
            uint64_t olo, ohi;
            pg_cas128(p, lo, hi, key, (val & PG_VAL_MASK) | t.tag, olo, ohi);
            if (olo == lo && ohi == hi) return true;
            lo = olo; hi = ohi;
        }
        if (lo == key) {
            if ((hi & val & PG_VAL_MASK) != (val & PG_VAL_MASK))
                atomicOr(reinterpret_cast<unsigned long long *>(p + 1), (unsigned long long)(val & PG_VAL_MASK));
            return true;
        }
        s = (s + 1) & t.capmask;
    }
    atomicExch(reinterpret_cast<unsigned long long *>(t.stats + PG_STAT_OVERFLOW), 1ull);
    return false;
}
// one atomicAdd per warp: slots claimed by this kernel -> PG_STAT_USED (distinct keys, kept by the inserts)
__device__ __forceinline__ void publish_claims(const TableView &t, uint32_t n_claimed) {
    n_claimed = __reduce_add_sync(0xffffffffu, n_claimed);
    if ((threadIdx.x & 31) == 0 && n_claimed)
        atomicAdd(reinterpret_cast<unsigned long long *>(t.stats + PG_STAT_USED), (unsigned long long)n_claimed);
}

// largest r in [-1, n_rec) with seq_off[r] <= g   (r = -1: g precedes the first record)
__device__ __forceinline__ int64_t find_record(const int64_t *__restrict__ seq_off, int64_t n_rec, int64_t g) {
    int64_t lo = 0, hi = n_rec;   // first index with seq_off[idx] > g
    while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if (__ldg(seq_off + mid) <= g) lo = mid + 1; else hi = mid;
    }
    return lo - 1;
}

// Stage the packed words [w0-2, w0+K2_TILE_WORDS+2) of a tile in shared memory with 128-bit loads.
__device__ __forceinline__ void stage_tile(const uint64_t *__restrict__ pk2, const uint32_t *__restrict__ amb,
                                           int64_t w0, int64_t n_words, uint64_t *s_pk, uint32_t *s_am) {
    // pk2: (K2_TILE_WORDS + 4) u64 = 130 uint4 ; amb: (K2_TILE_WORDS + 4) u32 = 65 uint4 ; w0 is even -> 16-B aligned
    const uint4 *gp = reinterpret_cast<const uint4 *>(pk2 + (w0 - 2));
    const uint4 *ga = reinterpret_cast<const uint4 *>(amb + (w0 - 4));
    for (int i = threadIdx.x; i < (K2_TILE_WORDS + 4) / 2; i += K2_THREADS) {
        int64_t w = w0 - 2 + 2 * i;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (w >= 0 && w + 1 < n_words) v = __ldg(gp + i);
        reinterpret_cast<uint4 *>(s_pk)[i] = v;
    }
    for (int i = threadIdx.x; i < (K2_TILE_WORDS + 8) / 4; i += K2_THREADS) {
        int64_t w = w0 - 4 + 4 * i;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (w >= 0 && w + 3 < n_words) v = __ldg(ga + i);
        reinterpret_cast<uint4 *>(s_am)[i] = v;
    }
}

