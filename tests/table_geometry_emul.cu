// table_geometry_emul.cu - host-side check of the dBG table's placement rule (tests/test_table_geometry.py).
// make_view / tv_home / tv_next (table_dev.cuh) are what every generic upsert and look-up probes with; the shared-memory
// region kernels (K3s region_build.cu, K3s-c compact_build.cu) place keys by a rule of their own.  The two must agree for
// every geometry the builder produces, or a key placed by a region kernel is claimed a second time by a later upsert.
// Compiled for sm_100a because table_dev.cuh uses __reduce_add_sync; only the host code here ever runs.
#include <cstring>
#include <vector>
#include "../pangenome_b200/csrc/table_dev.cuh"

namespace {

pg_table geometry(int bits, int region_bits, int hash_kind, int k) {
    pg_table t;
    memset(&t, 0, sizeof t);
    t.capacity = 1ll << bits; t.epoch = 1; t.region_bits = region_bits; t.hash_kind = hash_kind; t.k = k;
    t.mode = PG_MODE_CANONICAL;
    return t;
}

// The placement hash as the region kernels take it: K3s mixes the base-5 key; K3s-c mixes the 2-bit code with
// pg_mix64_top (the same top 31 bits as pg_mix64), and k3s_wide_insert places a key without a 2-bit form by mix64(~key).
uint64_t region_hash(int hash_kind, int k, uint64_t key) {
    if (!hash_kind) return pg_mix64(key);
    uint64_t x2;
    return pg_code2_of5(key, k, x2) ? pg_mix64_top(x2) : pg_mix64(~key);
}

// The region kernels' home: region r = the top (bits - region_bits) hash bits (the bucket K2a / K2c sort the record
// into), slot g = the next region_bits bits rounded down to a group of PG_REGION_GROUP (K3s: r * NS + g).
uint64_t region_home(int bits, int region_bits, uint64_t h) {
    const uint64_t ns = 1ull << region_bits;
    const uint64_t r = region_bits < bits ? h >> (64 - (bits - region_bits)) : 0;
    const uint64_t g = (h >> (64 - bits)) & (ns - 1) & ~(uint64_t)(PG_REGION_GROUP - 1);
    return r * ns + g;
}

}  // namespace

// out: capmask, rmask, hmask, shift of make_view for a table of 2^bits slots
extern "C" void tg_view(int bits, int region_bits, int hash_kind, int k, uint64_t *out) {
    const pg_table t = geometry(bits, region_bits, hash_kind, k);
    const TableView v = make_view(&t);
    out[0] = v.capmask; out[1] = v.rmask; out[2] = v.hmask; out[3] = (uint64_t)v.shift;
}

// Per key: tv_home; the region kernels' home (only meaningful while 0 < region_bits <= bits); and the unmasked home
// (top `bits` bits of the hash tv_home takes), which is the rule of a table without regions.
extern "C" void tg_homes(int bits, int region_bits, int hash_kind, int k, const uint64_t *keys, int64_t n, uint64_t *tv,
                         uint64_t *region, uint64_t *flat) {
    const pg_table t = geometry(bits, region_bits, hash_kind, k);
    const TableView v = make_view(&t);
    for (int64_t i = 0; i < n; i++) {
        tv[i] = tv_home(v, keys[i]);
        const uint64_t h = hash_kind ? pg_hash_kind1(keys[i], k) : pg_mix64(keys[i]);
        flat[i] = h >> (64 - bits);
        region[i] = region_bits > 0 && region_bits <= bits ? region_home(bits, region_bits, region_hash(hash_kind, k, keys[i])) : flat[i];
    }
}

// Place `keys` into a host slot array the way K3s / K3s-c do (home group; a key already in the group is found, else
// the first free slot of the group is claimed; else the next group, wrapping inside the region), then look every key
// up with the generic probe (tv_home, tv_next until a free slot) and replay the generic upsert (table_upsert_from's
// rule: claim the first free slot met).  stats: [0] keys the region rule found no room for, [1] keys placed outside
// their home group, [2] keys whose probe wrapped past the region's end, [3] keys the look-up missed, [4] keys the
// replayed upserts claimed a second slot for (a duplicate key) or found no room for.  Returns stats[3] + stats[4].
extern "C" int64_t tg_place_lookup(int bits, int region_bits, int hash_kind, int k, const uint64_t *keys, int64_t n,
                                   int64_t *stats) {
    const pg_table t = geometry(bits, region_bits, hash_kind, k);
    const TableView v = make_view(&t);
    const uint64_t ns = 1ull << region_bits;
    std::vector<uint64_t> slots((size_t)1 << bits, PG_EMPTY);
    for (int i = 0; i < 5; i++) stats[i] = 0;
    for (int64_t i = 0; i < n; i++) {
        const uint64_t key = keys[i];
        const uint64_t home = region_home(bits, region_bits, region_hash(hash_kind, k, key));
        const uint64_t base = home & ~(ns - 1);
        uint64_t g = home & (ns - 1);
        bool placed = false;
        for (uint64_t probe = 0; probe < ns / PG_REGION_GROUP && !placed; probe++) {
            int match = -1, free_ = -1;
            for (int j = PG_REGION_GROUP - 1; j >= 0; j--) {
                const uint64_t s = slots[base + g + j];
                if (s == key) match = j;
                if (s == PG_EMPTY) free_ = j;
            }
            const int j = match >= 0 ? match : free_;
            if (j >= 0) {
                slots[base + g + j] = key;
                placed = true;
                if (probe) stats[1]++;
                if (base + g < home) stats[2]++;
            }
            g = (g + PG_REGION_GROUP) & (ns - 1);
        }
        if (!placed) stats[0]++;
    }
    const uint64_t max_probe = v.rmask + 1 < PG_MAX_PROBE ? v.rmask + 1 : PG_MAX_PROBE;
    for (int pass = 0; pass < 2; pass++) {         // 0: look-up, 1: upsert
        for (int64_t i = 0; i < n; i++) {
            uint64_t s = tv_home(v, keys[i]);
            bool found = false;
            for (uint64_t probe = 0; probe < max_probe; probe++) {
                if (slots[s] == keys[i]) { found = true; break; }
                if (slots[s] == PG_EMPTY) {
                    if (pass) { slots[s] = keys[i]; stats[4]++; found = true; }
                    break;
                }
                s = tv_next(v, s);
            }
            if (!found) stats[3 + pass]++;
        }
    }
    return stats[3] + stats[4];
}
