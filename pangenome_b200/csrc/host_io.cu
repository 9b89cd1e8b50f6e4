// host_io.cu - host-side text writers for the side files the reference leaves next to its input
// (seq2graph, kmer_numba.py:1893-1904 writes <qry>_rdbg_weight.xyz line by line from Python; `mcl`
// writes <xyz>.mcl).  Plain C++ on the host: formatting millions of short lines is the slowest part
// of the drop-in CLI when done in Python.
#include <stdio.h>
#include <string.h>
#include <vector>
#include "common.cuh"

namespace {
// buffered writer that remembers a short write: a full disk must not leave a truncated side file behind a PG_OK
struct OutFile {
    FILE *f; bool ok;
    explicit OutFile(const char *path) : f(fopen(path, "wb")), ok(f != nullptr) {}
    void write(const char *p, size_t n) { if (ok && n && fwrite(p, 1, n, f) != n) ok = false; }
    bool close() { if (f) { if (fclose(f) != 0) ok = false; f = nullptr; } return ok; }
    ~OutFile() { if (f) fclose(f); }
};
inline char *put_u64(char *p, uint64_t v) {
    char tmp[24]; int n = 0;
    do { tmp[n++] = (char)('0' + v % 10); v /= 10; } while (v);
    while (n) *p++ = tmp[--n];
    return p;
}
}  // namespace

// "%d_%d\t%d_%d\t%d\n" per edge, in the order given (the caller sorts by first-insertion ordinal)
extern "C" int pg_host_write_xyz(const char *path, const uint64_t *c0, const uint32_t *v0, const uint64_t *c1,
                                 const uint32_t *v1, const uint32_t *w, int64_t n) {
    OutFile f(path);
    if (!f.ok) return pg_fail(PG_ERR_INVALID, "pg_host_write_xyz: cannot open %s", path);
    std::vector<char> buf(1 << 22);
    char *p = buf.data(), *end = buf.data() + buf.size() - 128;
    for (int64_t i = 0; i < n; i++) {
        p = put_u64(p, c0[i]); *p++ = '_'; p = put_u64(p, v0[i]); *p++ = '\t';
        p = put_u64(p, c1[i]); *p++ = '_'; p = put_u64(p, v1[i]); *p++ = '\t';
        p = put_u64(p, w[i]); *p++ = '\n';
        if (p > end) { f.write(buf.data(), (size_t)(p - buf.data())); p = buf.data(); }
    }
    f.write(buf.data(), (size_t)(p - buf.data()));
    if (!f.close()) return pg_fail(PG_ERR_INVALID, "pg_host_write_xyz: short write to %s (disk full?)", path);
    return PG_OK;
}

// one tab-separated line of node names "code_v5" per label; nodes must arrive sorted by (label, code, v5)
extern "C" int pg_host_write_mcl(const char *path, const uint64_t *code, const uint32_t *v5, const int64_t *label, int64_t n) {
    OutFile f(path);
    if (!f.ok) return pg_fail(PG_ERR_INVALID, "pg_host_write_mcl: cannot open %s", path);
    std::vector<char> buf(1 << 22);
    char *p = buf.data(), *end = buf.data() + buf.size() - 128;
    for (int64_t i = 0; i < n; i++) {
        if (i) *p++ = (label[i] != label[i - 1]) ? '\n' : '\t';
        p = put_u64(p, code[i]); *p++ = '_'; p = put_u64(p, v5[i]);
        if (p > end) { f.write(buf.data(), (size_t)(p - buf.data())); p = buf.data(); }
    }
    if (n) *p++ = '\n';
    f.write(buf.data(), (size_t)(p - buf.data()));
    if (!f.close()) return pg_fail(PG_ERR_INVALID, "pg_host_write_mcl: short write to %s (disk full?)", path);
    return PG_OK;
}

// ---- `_db.npz` interop (kmer_numba.py dump :243-261 / load_on_disk :289-335) --------------------
// The reference stores its dBG as the raw arrays of its open-addressing table `oakht`; to hand a
// GPU-built dBG to the reference's `-d` option the entries must be laid out the way its `pointer()`
// (:521-538) will probe for them: prime capacity, FNV-1a over the low 4 key bytes (:400-411),
// quadratic probing j = (j0 + t*t) % M.  The reference computes the hash in int64 and numba's % is
// Python's floor modulo, so j0 = signed hash mod M in [0, M): for hashes with bit 63 set this is not
// the unsigned remainder.  Host code: this is file-format work, not the hot path.
namespace {
bool oak_isprime(int64_t n) {
    if (n <= 1 || n % 2 == 0 || n % 3 == 0) return false;
    for (int64_t i = 5; i * i <= n; i += 6) if (n % i == 0 || n % (i + 2) == 0) return false;
    return true;
}
int64_t oak_find_prime(int64_t n) { for (;; n++) if (oak_isprime(n)) return n; }
inline uint64_t oak_fnv4(uint64_t v) {
    uint64_t a = 0xcbf29ce484222325ull;
    for (int i = 0; i < 4; i++) { a ^= (v & 0xff); a *= 0x100000001b3ull; v >>= 8; }
    return a;
}
}  // namespace

// capacity the reference's table has after inserting n distinct keys: starts at prime >= 2^20
// (init_dict ignores its capacity argument, :1121) and grows x1.62 whenever size/capacity > 0.75
extern "C" int64_t pg_host_oakht_capacity(int64_t n_entries) {
    int64_t cap = oak_find_prime(1 << 20);
    while ((double)n_entries / (double)cap > 0.75) cap = oak_find_prime((int64_t)((double)cap * 1.62));
    return cap;
}

extern "C" int pg_host_build_oakht(const uint64_t *keys, const uint16_t *vals, const uint8_t *cnts, int64_t n, int64_t cap,
                                   uint64_t *okeys, uint16_t *ovals, uint8_t *ocnts) {
    if (n < 0 || cap < 1 || n > cap || !okeys || !ovals || !ocnts) return pg_fail(PG_ERR_INVALID, "pg_host_build_oakht: bad arguments");
    memset(okeys, 0, (size_t)cap * 8); memset(ovals, 0, (size_t)cap * 2); memset(ocnts, 0, (size_t)cap);
    for (int64_t i = 0; i < n; i++) {
        int64_t j = (int64_t)oak_fnv4(keys[i]) % cap;
        if (j < 0) j += cap;
        const int64_t j0 = j;
        for (int64_t t = 0; t < cap; t++) {
            if (ocnts[j] == 0 || okeys[j] == keys[i]) break;
            j = (j0 + t * t) % cap;
        }
        if (ocnts[j] != 0 && okeys[j] != keys[i]) return pg_fail(PG_ERR_CAPACITY, "pg_host_build_oakht: probe sequence exhausted");
        okeys[j] = keys[i]; ovals[j] = vals[i]; ocnts[j] = cnts[i] ? cnts[i] : 1;
    }
    return PG_OK;
}
