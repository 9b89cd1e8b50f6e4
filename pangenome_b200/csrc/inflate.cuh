// inflate.cuh - raw-DEFLATE (RFC 1951) decoder and CRC-32 for one BGZF member, host + device.
//
// One member is decoded by a group of `PgLanes` cooperating threads: a warp on the device (bgzf_inflate.cu),
// a single thread in the CPU harness (tests/inflate_emul.cu), from the same source.  Every lane runs the SAME
// bit reader and symbol decoder on the same compressed bytes, so control flow stays uniform across the warp and
// the decoded symbol never has to be broadcast: the loads are same-address (one transaction) and the redundant
// lanes cost issue slots the warp would spend waiting anyway.  The lanes split the work that has no serial
// dependency: filling the Huffman look-up tables, match and stored-block copies, and the CRC-32 of the output.
// Lane 0 alone writes literals and builds the per-block code tables (counting sort of the code lengths).
//
// All input is untrusted.  The decoder reads only src[0, src_len) and writes only dst[0, dst_len); every
// malformed stream ends in a PG_INF_* error code (include/pgdbg.h), never in an out-of-bounds access.  Code
// validation follows zlib's inflate: over-subscribed codes are rejected, incomplete literal/length and distance
// codes are accepted only as a single code of length 1, an incomplete code-length code is rejected.
#pragma once
#include <stdint.h>
#include "../../include/pgdbg.h"

#ifndef PG_HD
#define PG_HD __host__ __device__ __forceinline__
#endif

#define PG_INF_LIT_LB 10      // first-level look-up bits of the literal/length code (longer codes: canonical walk)
#define PG_INF_DIST_LB 8      // ... of the distance code

// Per-member scratch: shared memory on the device (about 3.7 KB per warp)
struct PgInflateWs {
    uint16_t lit_lut[1 << PG_INF_LIT_LB];   // entry = symbol << 4 | code length; 0 = not resolved in LB bits
    uint16_t dist_lut[1 << PG_INF_DIST_LB];
    uint16_t lit_sym[288];                   // symbols ordered by (code length, value): canonical code order
    uint16_t dist_sym[32];                   // also holds the 19-symbol code-length code while a header is read
    uint16_t lit_cnt[16];                    // codes per length
    uint16_t dist_cnt[16];
    uint8_t lens[320];                       // code lengths of the block being set up (HLIT + HDIST <= 316)
    uint32_t crc_part[32];                   // per-lane CRC-32 of the output segments
    int32_t err;                             // lane 0's verdict, read by every lane after a sync
    int32_t fixed_loaded;                    // the tables hold the fixed code (reused by later fixed blocks)
};

// A group of lanes decoding one member: a warp on the device, one thread on the host
struct PgLanes {
    int lane, n;
    PG_HD void sync() const {
#ifdef __CUDA_ARCH__
        __syncwarp();
#endif
    }
};

// ---- CRC-32 (gzip: reflected polynomial 0xEDB88320, initial and final xor 0xFFFFFFFF) ----------------------------
PG_HD uint32_t pg_crc_entry(uint32_t i) {
    uint32_t c = i;
    for (int k = 0; k < 8; k++) c = (c & 1) ? (c >> 1) ^ 0xEDB88320u : c >> 1;
    return c;
}
// a(x) * b(x) mod P(x), reflected bit order (zlib's multmodp)
PG_HD uint32_t pg_crc_mulmod(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = (b & 1) ? (b >> 1) ^ 0xEDB88320u : b >> 1;
    }
    return p;
}
// x^(8 n) mod P(x): the operator that appends n zero bytes
PG_HD uint32_t pg_crc_x8n(int64_t n) {
    uint32_t p = 1u << 31, t = 1u << 30;           // 1, x
    for (int i = 0; i < 3; i++) t = pg_crc_mulmod(t, t);   // x^8
    while (n) {
        if (n & 1) p = pg_crc_mulmod(t, p);
        t = pg_crc_mulmod(t, t);
        n >>= 1;
    }
    return p;
}
// crc(A || B) from crc(A), crc(B) and |B| (zlib's crc32_combine)
PG_HD uint32_t pg_crc_combine(uint32_t crc_a, uint32_t crc_b, int64_t len_b) {
    return pg_crc_mulmod(pg_crc_x8n(len_b), crc_a) ^ crc_b;
}

// CRC-32 of buf[0, n): every lane takes one contiguous segment, lane 0 chains the segment CRCs
PG_HD uint32_t pg_crc32_lanes(const uint8_t *buf, int64_t n, const uint32_t *tab, PgInflateWs *ws, PgLanes L) {
    const int64_t seg = (n + L.n - 1) / L.n;
    int64_t a = (int64_t)L.lane * seg, b = a + seg;
    if (a > n) a = n;
    if (b > n) b = n;
    uint32_t c = 0xFFFFFFFFu;
    for (int64_t i = a; i < b; i++) c = tab[(c ^ buf[i]) & 0xFF] ^ (c >> 8);
    ws->crc_part[L.lane] = c ^ 0xFFFFFFFFu;
    L.sync();
    if (L.lane == 0) {
        uint32_t crc = ws->crc_part[0];
        if (L.n > 1 && seg > 0) {
            const uint32_t shift = pg_crc_x8n(seg);
            for (int l = 1; l < L.n; l++) {
                const int64_t la = (int64_t)l * seg;
                if (la >= n) break;
                const int64_t len = (la + seg <= n) ? seg : n - la;
                crc = (len == seg ? pg_crc_mulmod(shift, crc) : pg_crc_mulmod(pg_crc_x8n(len), crc)) ^ ws->crc_part[l];
            }
        }
        ws->crc_part[0] = crc;
    }
    L.sync();
    const uint32_t crc = ws->crc_part[0];
    L.sync();
    return crc;
}

// ---- bit reader: least significant bit first, refilled byte by byte, never past `end` ----------------------------
struct PgBits {
    const uint8_t *p;
    int64_t pos, end;    // next byte to load, end of the compressed bytes
    uint64_t buf;        // unread bits, bit 0 first
    int n;               // valid bits in buf
};

PG_HD void pg_bits_fill(PgBits &b) {
    while (b.n <= 56 && b.pos < b.end) { b.buf |= (uint64_t)b.p[b.pos++] << b.n; b.n += 8; }
}
// take k <= 32 bits; false when the input has fewer left
PG_HD bool pg_bits_take(PgBits &b, int k, uint32_t &v) {
    if (b.n < k) pg_bits_fill(b);
    if (b.n < k) return false;
    v = (uint32_t)(b.buf & ((1ull << k) - 1));
    b.buf >>= k;
    b.n -= k;
    return true;
}

// ---- Huffman codes ---------------------------------------------------------------------------------------------
// Counting sort of the code lengths into canonical order; validation as zlib's inflate_table.  Lane 0 only.
// kind 0: code-length code (must be complete), 1: literal/length or distance code (incomplete only as one 1-bit code)
PG_HD int pg_huff_build(const uint8_t *lens, int n, uint16_t *cnt, uint16_t *sym, int kind) {
    for (int l = 0; l < 16; l++) cnt[l] = 0;
    for (int s = 0; s < n; s++) cnt[lens[s]]++;
    int max = 0;
    for (int l = 1; l < 16; l++) if (cnt[l]) max = l;
    if (max == 0) return kind == 0 ? PG_INF_ERR_CODE : PG_OK;   // no codes: any use is an invalid-code error
    int left = 1;
    for (int l = 1; l < 16; l++) {
        left <<= 1;
        left -= cnt[l];
        if (left < 0) return PG_INF_ERR_CODE;                    // over-subscribed
    }
    if (left > 0 && (kind == 0 || max != 1)) return PG_INF_ERR_CODE;   // incomplete
    uint16_t offs[16];
    offs[1] = 0;
    for (int l = 1; l < 15; l++) offs[l + 1] = (uint16_t)(offs[l] + cnt[l]);
    for (int s = 0; s < n; s++) if (lens[s]) sym[offs[lens[s]]++] = (uint16_t)s;
    return PG_OK;
}

// One canonical-code walk over at most `maxlen` bits of `bits` (bit 0 first).  Returns symbol << 4 | length, 0 when no
// code of at most maxlen bits matches.
PG_HD uint32_t pg_huff_walk(const uint16_t *cnt, const uint16_t *sym, uint32_t bits, int maxlen) {
    int code = 0, first = 0, index = 0;
    for (int len = 1; len <= maxlen; len++) {
        code |= (int)(bits & 1);
        bits >>= 1;
        const int count = cnt[len];
        if (code - first < count) return ((uint32_t)sym[index + (code - first)] << 4) | (uint32_t)len;
        index += count;
        first += count;
        first <<= 1;
        code <<= 1;
    }
    return 0;
}

// first-level table: entry i resolves the code that bits i (LB of them, bit 0 first) begin with; the lanes split it
PG_HD void pg_huff_lut(const uint16_t *cnt, const uint16_t *sym, uint16_t *lut, int lb, PgLanes L) {
    for (int i = L.lane; i < (1 << lb); i += L.n) lut[i] = (uint16_t)pg_huff_walk(cnt, sym, (uint32_t)i, lb);
}

// decode one symbol; -1 = invalid code, -2 = input ends inside it.  The caller has filled the bit buffer.
PG_HD int pg_huff_decode(PgBits &b, const uint16_t *lut, int lb, const uint16_t *cnt, const uint16_t *sym) {
    uint32_t e = lut[b.buf & ((1u << lb) - 1)];
    if (e == 0) e = pg_huff_walk(cnt, sym, (uint32_t)(b.buf & 0x7FFF), 15);
    const int len = (int)(e & 15);
    if (len == 0) return -1;
    if (len > b.n) return -2;
    b.buf >>= len;
    b.n -= len;
    return (int)(e >> 4);
}

// ---- the decoder -----------------------------------------------------------------------------------------------
PG_HD void pg_inf_setup_tables(PgInflateWs *ws, int nlit, PgLanes L) {
    // lane 0 has written lens[0, nlit + ndist) and built the counts/symbols; every lane fills its share of the tables
    pg_huff_lut(ws->lit_cnt, ws->lit_sym, ws->lit_lut, PG_INF_LIT_LB, L);
    pg_huff_lut(ws->dist_cnt, ws->dist_sym, ws->dist_lut, PG_INF_DIST_LB, L);
    L.sync();
}

// Code lengths of a dynamic block (RFC 1951 3.2.7) -> ws tables.  Returns PG_OK or PG_INF_ERR_*, the same in every lane.
PG_HD int pg_inf_dynamic(PgBits &b, PgInflateWs *ws, PgLanes L) {
    uint32_t hlit, hdist, hclen;
    if (!pg_bits_take(b, 5, hlit) || !pg_bits_take(b, 5, hdist) || !pg_bits_take(b, 4, hclen)) return PG_INF_ERR_TRUNCATED;
    const int nlit = (int)hlit + 257, ndist = (int)hdist + 1, ncl = (int)hclen + 4;
    if (nlit > 286 || ndist > 30) return PG_INF_ERR_CODE;
    const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    uint8_t cl[19];
    for (int i = 0; i < 19; i++) cl[i] = 0;
    for (int i = 0; i < ncl; i++) {
        uint32_t v;
        if (!pg_bits_take(b, 3, v)) return PG_INF_ERR_TRUNCATED;
        cl[order[i]] = (uint8_t)v;
    }
    L.sync();                                       // every lane is done with the previous block's tables
    if (L.lane == 0) ws->err = pg_huff_build(cl, 19, ws->dist_cnt, ws->dist_sym, 0);
    L.sync();
    int err = ws->err;
    if (err) return err;
    int i = 0, prev = 0;
    while (i < nlit + ndist) {
        pg_bits_fill(b);
        const uint32_t e = pg_huff_walk(ws->dist_cnt, ws->dist_sym, (uint32_t)(b.buf & 0x7F), 7);
        const int len = (int)(e & 15);
        if (len == 0) return PG_INF_ERR_CODE;
        if (len > b.n) return PG_INF_ERR_TRUNCATED;
        b.buf >>= len;
        b.n -= len;
        const int s = (int)(e >> 4);
        int val, rep;
        uint32_t x;
        if (s < 16) {
            val = s; rep = 1; prev = s;
        } else if (s == 16) {
            if (i == 0) return PG_INF_ERR_CODE;       // repeat with no previous length
            if (!pg_bits_take(b, 2, x)) return PG_INF_ERR_TRUNCATED;
            val = prev; rep = 3 + (int)x;
        } else if (s == 17) {
            if (!pg_bits_take(b, 3, x)) return PG_INF_ERR_TRUNCATED;
            val = 0; rep = 3 + (int)x; prev = 0;
        } else {
            if (!pg_bits_take(b, 7, x)) return PG_INF_ERR_TRUNCATED;
            val = 0; rep = 11 + (int)x; prev = 0;
        }
        if (i + rep > nlit + ndist) return PG_INF_ERR_CODE;
        if (L.lane == 0) for (int r = 0; r < rep; r++) ws->lens[i + r] = (uint8_t)val;
        i += rep;
    }
    L.sync();
    if (L.lane == 0) {
        err = ws->lens[256] == 0 ? PG_INF_ERR_CODE : pg_huff_build(ws->lens, nlit, ws->lit_cnt, ws->lit_sym, 1);
        if (!err) err = pg_huff_build(ws->lens + nlit, ndist, ws->dist_cnt, ws->dist_sym, 1);
        ws->err = err;
        ws->fixed_loaded = 0;
    }
    L.sync();
    err = ws->err;
    if (err) return err;
    pg_inf_setup_tables(ws, nlit, L);
    return PG_OK;
}

PG_HD int pg_inf_fixed(PgInflateWs *ws, PgLanes L) {
    L.sync();
    if (ws->fixed_loaded) return PG_OK;
    if (L.lane == 0) {
        for (int s = 0; s < 288; s++) ws->lens[s] = (uint8_t)(s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8);
        for (int s = 0; s < 32; s++) ws->lens[288 + s] = 5;
        pg_huff_build(ws->lens, 288, ws->lit_cnt, ws->lit_sym, 1);          // both codes are complete: cannot fail
        pg_huff_build(ws->lens + 288, 32, ws->dist_cnt, ws->dist_sym, 1);
        ws->fixed_loaded = 1;
    }
    L.sync();
    pg_inf_setup_tables(ws, 288, L);
    return PG_OK;
}

// Inflate the raw-DEFLATE stream src[0, src_len) into dst[0, dst_len).  On PG_OK: *produced = output bytes,
// *consumed = input bytes up to the end of the final block (rounded up to a byte).  Errors: PG_INF_ERR_*.
PG_HD int pg_inflate_raw(const uint8_t *src, int64_t src_len, uint8_t *dst, int64_t dst_len, PgInflateWs *ws, PgLanes L,
                         int64_t *produced, int64_t *consumed) {
    PgBits b;
    b.p = src; b.pos = 0; b.end = src_len; b.buf = 0; b.n = 0;
    int64_t op = 0;
    if (L.lane == 0) ws->fixed_loaded = 0;
    L.sync();
    uint32_t last = 0;
    do {
        uint32_t type;
        if (!pg_bits_take(b, 1, last) || !pg_bits_take(b, 2, type)) return PG_INF_ERR_TRUNCATED;
        if (type == 0) {
            // stored: skip to a byte boundary, LEN and its complement, LEN bytes copied as they are
            const int drop = b.n & 7;
            b.buf >>= drop;
            b.n -= drop;
            uint32_t len, nlen;
            if (!pg_bits_take(b, 16, len) || !pg_bits_take(b, 16, nlen)) return PG_INF_ERR_TRUNCATED;
            if ((len ^ 0xFFFFu) != nlen) return PG_INF_ERR_STORED;
            b.pos -= b.n >> 3;                       // the whole bytes still buffered are unread input
            b.buf = 0;
            b.n = 0;
            if ((int64_t)len > b.end - b.pos) return PG_INF_ERR_TRUNCATED;
            if ((int64_t)len > dst_len - op) return PG_INF_ERR_OVERFLOW;
            L.sync();
            for (int64_t j = L.lane; j < (int64_t)len; j += L.n) dst[op + j] = src[b.pos + j];
            b.pos += len;
            op += len;
            continue;
        }
        int err = type == 1 ? pg_inf_fixed(ws, L) : type == 2 ? pg_inf_dynamic(b, ws, L) : PG_INF_ERR_BLOCK;
        if (err) return err;
        for (;;) {
            pg_bits_fill(b);
            const int s = pg_huff_decode(b, ws->lit_lut, PG_INF_LIT_LB, ws->lit_cnt, ws->lit_sym);
            if (s < 0) return s == -1 ? PG_INF_ERR_SYMBOL : PG_INF_ERR_TRUNCATED;
            if (s < 256) {
                if (op >= dst_len) return PG_INF_ERR_OVERFLOW;
                if (L.lane == 0) dst[op] = (uint8_t)s;
                op++;
                continue;
            }
            if (s == 256) break;
            const int ls = s - 257;
            if (ls >= 29) return PG_INF_ERR_SYMBOL;
            int len;
            uint32_t x;
            if (ls < 8) {
                len = ls + 3;
            } else if (ls == 28) {
                len = 258;
            } else {
                const int e = (ls - 4) >> 2;
                if (!pg_bits_take(b, e, x)) return PG_INF_ERR_TRUNCATED;
                len = ((4 + (ls & 3)) << e) + 3 + (int)x;
            }
            const int ds = pg_huff_decode(b, ws->dist_lut, PG_INF_DIST_LB, ws->dist_cnt, ws->dist_sym);
            if (ds < 0) return ds == -1 ? PG_INF_ERR_SYMBOL : PG_INF_ERR_TRUNCATED;
            if (ds >= 30) return PG_INF_ERR_SYMBOL;
            int64_t dist;
            if (ds < 4) {
                dist = ds + 1;
            } else {
                const int e = (ds >> 1) - 1;
                if (!pg_bits_take(b, e, x)) return PG_INF_ERR_TRUNCATED;
                dist = ((int64_t)(2 + (ds & 1)) << e) + 1 + x;
            }
            if (dist > op) return PG_INF_ERR_DISTANCE;
            if ((int64_t)len > dst_len - op) return PG_INF_ERR_OVERFLOW;
            // out[op + j] = out[op - dist + j mod dist]: every source byte lies before op, so the lanes copy in any order
            L.sync();
            const uint8_t *from = dst + op - dist;
            if (dist >= len) {
                for (int j = L.lane; j < len; j += L.n) dst[op + j] = from[j];
            } else {
                for (int j = L.lane; j < len; j += L.n) dst[op + j] = from[j % (int)dist];
            }
            op += len;
        }
    } while (!last);
    L.sync();
    *produced = op;
    *consumed = b.pos - (b.n >> 3);
    return PG_OK;
}

PG_HD uint32_t pg_le32(const uint8_t *p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

// One BGZF member gz[0, gz_len) (gzip header with the BC extra field, raw DEFLATE, CRC-32, ISIZE) into exactly
// out[0, out_len).  Returns PG_OK or PG_INF_ERR_*, the same in every lane.
PG_HD int pg_bgzf_member(const uint8_t *gz, int64_t gz_len, uint8_t *out, int64_t out_len, const uint32_t *crc_tab,
                         PgInflateWs *ws, PgLanes L) {
    if (gz_len < 12 + 8) return PG_INF_ERR_HEADER;
    if (gz[0] != 0x1f || gz[1] != 0x8b || gz[2] != 8 || gz[3] != 4) return PG_INF_ERR_HEADER;
    const int64_t data = 12 + (int64_t)(gz[10] | (gz[11] << 8));
    if (data > gz_len - 8) return PG_INF_ERR_HEADER;
    const uint32_t crc = pg_le32(gz + gz_len - 8), isize = pg_le32(gz + gz_len - 4);
    if ((int64_t)isize != out_len) return PG_INF_ERR_LENGTH;
    int64_t produced = 0, consumed = 0;
    const int err = pg_inflate_raw(gz + data, gz_len - 8 - data, out, out_len, ws, L, &produced, &consumed);
    if (err) return err;
    if (produced != out_len || consumed != gz_len - 8 - data) return PG_INF_ERR_LENGTH;
    return pg_crc32_lanes(out, out_len, crc_tab, ws, L) == crc ? PG_OK : PG_INF_ERR_CRC;
}
