// deflate.cuh - raw-DEFLATE (RFC 1951) encoder for one independent chunk, host + device.
//
// The `_db.npz` members are images of an open-addressing table: empty slots are runs of zero bytes, live slots are
// close to random bytes.  Matches at distance 1 (runs) capture nearly all the redundancy (zlib's Z_RLE does as well as
// its level 6 on such images), so the parse is local and data-parallel:
//   - every maximal run of equal bytes of length L >= 4 becomes one literal and matches at distance 1 covering the
//     other L - 1 bytes, in pieces of 258 split deterministically (pg_def_piece); shorter runs are literals;
//   - one histogram per chunk, one Huffman code per chunk (two-queue construction over the symbols sorted by
//     (frequency, symbol), lengths limited with the JPEG Annex K.3 adjustment), so the output is a function of the
//     chunk's bytes alone;
//   - the chunk becomes the smallest of one dynamic block, one fixed block or one stored block.  A chunk that is not the
//     member's last ends byte-aligned (a stored block is aligned already; a Huffman block is followed by an empty stored
//     block, 00 00 ff ff), so chunks concatenate into one valid stream and each decodes on its own.
//
// A chunk is encoded by a group of `PgDefLanes` cooperating threads: a CTA on the device (npz_dump.cu), one thread in
// the CPU harness (tests/deflate_emul.cu), from the same source.  Lanes split the chunk into contiguous segments; a
// lane owns every run that STARTS in its segment.  Code construction is lane 0's; the bit offsets of the segments are
// a prefix sum, and each lane ORs its bits into the zeroed output words, so the bytes do not depend on the lane count.
#pragma once
#include <stdint.h>
#include "inflate.cuh"

#define PG_DEF_MAX_CHUNK 65535    // one stored block per chunk: at most 5 bytes of overhead
#define PG_DEF_MAX_LANES 256
#define PG_DEF_NLIT 286
#define PG_DEF_NDIST 30
#define PG_DEF_NCL 19
#define PG_DEF_MODE_DYNAMIC 2     // BTYPE values
#define PG_DEF_MODE_FIXED 1
#define PG_DEF_MODE_STORED 0

struct PgDefLanes {
    int lane, n;
    PG_HD void sync() const {
#ifdef __CUDA_ARCH__
        __syncthreads();
#endif
    }
};

// Per-chunk scratch: shared memory on the device (about 9 KB)
struct PgDeflateWs {
    uint32_t lit_freq[PG_DEF_NLIT];
    uint32_t dist_freq[PG_DEF_NDIST];
    uint32_t cl_freq[PG_DEF_NCL];
    uint8_t lit_len[PG_DEF_NLIT];
    uint8_t dist_len[PG_DEF_NDIST];
    uint8_t cl_len[PG_DEF_NCL];
    uint16_t lit_code[PG_DEF_NLIT];      // canonical codes, bit-reversed for LSB-first output
    uint16_t dist_code[PG_DEF_NDIST];
    uint16_t cl_code[PG_DEF_NCL];
    // code construction (one alphabet at a time)
    uint32_t tf[288];                    // frequencies, with symbols forced in so that every code has >= 2 symbols
    uint16_t order[288];                 // used symbols sorted by (frequency, symbol)
    uint32_t iw[288];                    // weights of the internal nodes
    uint16_t parent[576];                // leaves 0..m-1 (sorted order), internal nodes m..2m-2
    uint16_t depth[576];
    uint16_t bits[300];                  // leaves per depth (a Huffman tree over <= 288 leaves is at most 287 deep)
    uint16_t cl_tok[PG_DEF_NLIT + PG_DEF_NDIST];   // code-length tokens: symbol | extra << 5
    uint32_t part[PG_DEF_MAX_LANES];     // per-lane bit counts, then bit offsets
    int32_t ntok, nlit, ndist, nclen, mode, used;
    int64_t hdr_bits, size;
};

PG_HD void pg_or32(uint32_t *p, uint32_t v) {
#ifdef __CUDA_ARCH__
    atomicOr(p, v);
#else
    *p |= v;
#endif
}
PG_HD void pg_add32(uint32_t *p, uint32_t v) {
#ifdef __CUDA_ARCH__
    atomicAdd(p, v);
#else
    *p += v;
#endif
}

// LSB-first bit writer that ORs whole 32-bit words into a zeroed buffer: writers of neighbouring bit ranges share at
// most their boundary words, which the atomic OR merges
struct PgBitOut {
    uint32_t *w;
    int64_t word;
    uint64_t acc;
    int nb;
    PG_HD void init(uint32_t *out, int64_t bitpos) { w = out; word = bitpos >> 5; nb = (int)(bitpos & 31); acc = 0; }
    PG_HD void put(uint32_t v, int k) {        // k <= 32, v < 2^k
        acc |= (uint64_t)v << nb;
        nb += k;
        if (nb >= 32) { pg_or32(w + word, (uint32_t)acc); word++; acc >>= 32; nb -= 32; }
    }
    PG_HD void flush() { if (nb > 0) pg_or32(w + word, (uint32_t)acc); }
};

PG_HD int pg_def_log2(uint32_t v) {
#ifdef __CUDA_ARCH__
    return 31 - __clz(v);
#else
    return 31 - __builtin_clz(v);
#endif
}

// match length 3..258 -> length symbol - 257 (0..28), its extra bits and their value
PG_HD void pg_def_lencode(int len, int &ls, int &eb, uint32_t &ev) {
    const int v = len - 3;
    if (v < 8) { ls = v; eb = 0; ev = 0; return; }
    if (len == 258) { ls = 28; eb = 0; ev = 0; return; }
    const int e = pg_def_log2((uint32_t)v) - 2;
    ls = 4 * e + 4 + ((v >> e) & 3);
    eb = e;
    ev = (uint32_t)(v - ((4 + (ls & 3)) << e));
}
PG_HD int pg_def_len_extra(int ls) { return (ls < 8 || ls == 28) ? 0 : (ls - 4) >> 2; }

// The pieces a run's match span of M = L - 1 bytes is cut into: 258 while at least 261 are left (a piece may not leave
// fewer than 3), then one piece of the rest, or - for 259 / 260 left - rest - 3 and 3.  Returns the length of the piece
// that starts at offset o of the span, 0 when none does.
PG_HD int pg_def_piece(int64_t M, int64_t o) {
    const int64_t k = M >= 261 ? (M - 261) / 258 + 1 : 0;
    const int64_t rest = M - 258 * k;                        // 3..260
    if (o < 258 * k) return (o % 258 == 0) ? 258 : 0;
    if (o == 258 * k) return (int)(rest <= 258 ? rest : rest - 3);
    if (rest > 258 && o == 258 * k + rest - 3) return 3;
    return 0;
}

// Visit the tokens of the runs that start in this lane's segment of in[0, n), in stream order: f.lit(byte), f.match(len)
template <class F>
PG_HD void pg_def_walk(const uint8_t *in, int64_t n, PgDefLanes L, F &f) {
    const int64_t seg = (n + L.n - 1) / L.n;
    int64_t i = (int64_t)L.lane * seg, b = i + seg;
    if (b > n) b = n;
    while (i < b && i > 0 && in[i] == in[i - 1]) i++;       // the tail of a run an earlier lane owns
    while (i < b) {
        const uint8_t c = in[i];
        int64_t e = i + 1;
        while (e < n && in[e] == c) e++;
        const int64_t len = e - i;
        if (len < 4) {
            for (int64_t j = 0; j < len; j++) f.lit(c);
        } else {
            f.lit(c);
            const int64_t M = len - 1;
            for (int64_t o = 0; o < M;) {
                const int p = pg_def_piece(M, o);
                f.match(p);
                o += p;
            }
        }
        i = e;
    }
}

struct PgDefHist {
    PgDeflateWs *ws;
    PG_HD void lit(uint8_t c) { pg_add32(&ws->lit_freq[c], 1); }
    PG_HD void match(int len) {
        int ls, eb; uint32_t ev;
        pg_def_lencode(len, ls, eb, ev);
        pg_add32(&ws->lit_freq[257 + ls], 1);
        pg_add32(&ws->dist_freq[0], 1);
    }
};

// fixed code (RFC 1951 3.2.6): code value and length of a literal/length symbol, not yet bit-reversed
PG_HD void pg_def_fixed(int s, uint32_t &code, int &len) {
    if (s < 144) { code = 0x30 + s; len = 8; }
    else if (s < 256) { code = 0x190 + (s - 144); len = 9; }
    else if (s < 280) { code = s - 256; len = 7; }
    else { code = 0xC0 + (s - 280); len = 8; }
}
PG_HD uint32_t pg_def_rev(uint32_t v, int len) {
    uint32_t r = 0;
    for (int i = 0; i < len; i++) { r = (r << 1) | (v & 1); v >>= 1; }
    return r;
}

struct PgDefCount {
    const PgDeflateWs *ws;
    int fixed;
    int64_t bits;
    PG_HD int lit_bits(int s) const {
        if (!fixed) return ws->lit_len[s];
        uint32_t c; int l; pg_def_fixed(s, c, l); return l;
    }
    PG_HD void lit(uint8_t c) { bits += lit_bits(c); }
    PG_HD void match(int len) {
        int ls, eb; uint32_t ev;
        pg_def_lencode(len, ls, eb, ev);
        bits += lit_bits(257 + ls) + eb + (fixed ? 5 : ws->dist_len[0]);
    }
};

struct PgDefEmit {
    const PgDeflateWs *ws;
    int fixed;
    PgBitOut o;
    PG_HD void sym(int s) {
        if (fixed) { uint32_t c; int l; pg_def_fixed(s, c, l); o.put(pg_def_rev(c, l), l); }
        else o.put(ws->lit_code[s], ws->lit_len[s]);
    }
    PG_HD void lit(uint8_t c) { sym(c); }
    PG_HD void match(int len) {
        int ls, eb; uint32_t ev;
        pg_def_lencode(len, ls, eb, ev);
        sym(257 + ls);
        if (eb) o.put(ev, eb);
        if (fixed) o.put(0, 5);                              // distance symbol 0 (distance 1): five zero bits
        else o.put(ws->dist_code[0], ws->dist_len[0]);
    }
};

// Length-limited Huffman code lengths len[0, n) for freq[0, n) (limit <= 15).  Every lane calls it.
PG_HD void pg_def_tree(const uint32_t *freq, int n, int limit, uint8_t *len, PgDeflateWs *ws, PgDefLanes L) {
    if (L.lane == 0) {
        int used = 0;
        for (int s = 0; s < n; s++) { ws->tf[s] = freq[s]; used += freq[s] > 0; }
        for (int s = 0; s < n && used < 2; s++)            // a code needs two symbols (one alone is incomplete)
            if (ws->tf[s] == 0) { ws->tf[s] = 1; used++; }
        ws->used = used;
    }
    L.sync();
    for (int s = L.lane; s < n; s += L.n) {                // rank sort by (frequency, symbol)
        const uint32_t f = ws->tf[s];
        if (f == 0) { len[s] = 0; continue; }
        int r = 0;
        for (int t = 0; t < n; t++) {
            const uint32_t g = ws->tf[t];
            r += g != 0 && (g < f || (g == f && t < s));
        }
        ws->order[r] = (uint16_t)s;
    }
    L.sync();
    if (L.lane == 0) {
        const int m = ws->used;
        // two-queue Huffman: leaves in sorted order, internal nodes in creation order (non-decreasing weights);
        // on equal weights the leaf is taken first
        int li = 0, ii = 0, ni = 0;
        for (int k = 0; k < m - 1; k++) {
            int pick[2];
            uint32_t w = 0;
            for (int q = 0; q < 2; q++) {
                const bool leaf = li < m && (ii >= ni || ws->tf[ws->order[li]] <= ws->iw[ii]);
                if (leaf) { w += ws->tf[ws->order[li]]; pick[q] = li++; }
                else { w += ws->iw[ii]; pick[q] = m + ii++; }
            }
            ws->parent[pick[0]] = ws->parent[pick[1]] = (uint16_t)(m + ni);
            ws->iw[ni++] = w;
        }
        const int root = 2 * m - 2;
        ws->depth[root] = 0;
        for (int v = root - 1; v >= 0; v--) ws->depth[v] = (uint16_t)(ws->depth[ws->parent[v]] + 1);
        int maxd = 0;
        for (int d = 0; d < 300; d++) ws->bits[d] = 0;
        for (int v = 0; v < m; v++) { ws->bits[ws->depth[v]]++; if (ws->depth[v] > maxd) maxd = ws->depth[v]; }
        // JPEG Annex K.3: move pairs of the deepest leaves up until no code is longer than the limit (stays complete)
        for (int i = maxd; i > limit; i--) {
            while (ws->bits[i] > 0) {
                int j = i - 2;
                while (ws->bits[j] == 0) j--;
                ws->bits[i] -= 2;
                ws->bits[i - 1] += 1;
                ws->bits[j + 1] += 2;
                ws->bits[j] -= 1;
            }
        }
        // the longest codes to the least frequent symbols
        int v = 0;
        for (int d = maxd < limit ? maxd : limit; d >= 1; d--)
            for (int c = 0; c < ws->bits[d]; c++) len[ws->order[v++]] = (uint8_t)d;
    }
    L.sync();
}

// canonical codes (RFC 1951 3.2.2), bit-reversed for LSB-first output.  Lane 0.
PG_HD void pg_def_codes(const uint8_t *len, int n, uint16_t *code) {
    uint16_t cnt[16], next[16];
    for (int l = 0; l < 16; l++) cnt[l] = 0;
    for (int s = 0; s < n; s++) cnt[len[s]]++;
    cnt[0] = 0;
    uint32_t c = 0;
    for (int l = 1; l < 16; l++) { c = (c + cnt[l - 1]) << 1; next[l] = (uint16_t)c; }
    for (int s = 0; s < n; s++) if (len[s]) code[s] = (uint16_t)pg_def_rev(next[len[s]]++, len[s]);
}

// Encode in[0, n) (n <= PG_DEF_MAX_CHUNK) as described above into out (4-byte aligned, at least n + 8 bytes).  `last`:
// the member's final chunk (sets BFINAL).  Returns the chunk's compressed size in bytes, the same in every lane.
PG_HD int64_t pg_deflate_chunk(const uint8_t *in, int64_t n, bool last, uint8_t *out, PgDeflateWs *ws, PgDefLanes L) {
    for (int s = L.lane; s < PG_DEF_NLIT; s += L.n) ws->lit_freq[s] = 0;
    for (int s = L.lane; s < PG_DEF_NDIST; s += L.n) ws->dist_freq[s] = 0;
    L.sync();
    PgDefHist h{ws};
    pg_def_walk(in, n, L, h);
    if (L.lane == 0) ws->lit_freq[256] = 1;                  // end of block
    L.sync();
    pg_def_tree(ws->lit_freq, PG_DEF_NLIT, 15, ws->lit_len, ws, L);
    pg_def_tree(ws->dist_freq, PG_DEF_NDIST, 15, ws->dist_len, ws, L);
    if (L.lane == 0) {
        int nlit = PG_DEF_NLIT, ndist = PG_DEF_NDIST;
        while (nlit > 257 && ws->lit_len[nlit - 1] == 0) nlit--;
        while (ndist > 1 && ws->dist_len[ndist - 1] == 0) ndist--;
        // run-length code of the nlit + ndist code lengths (16: repeat previous 3-6, 17: 3-10 zeros, 18: 11-138 zeros)
        for (int s = 0; s < PG_DEF_NCL; s++) ws->cl_freq[s] = 0;
        int nt = 0;
        const int tot = nlit + ndist;
        for (int i = 0; i < tot;) {
            const int v = i < nlit ? ws->lit_len[i] : ws->dist_len[i - nlit];
            int r = 1;
            while (i + r < tot && (i + r < nlit ? ws->lit_len[i + r] : ws->dist_len[i + r - nlit]) == v) r++;
            i += r;
            if (v == 0) {
                while (r >= 11) { const int t = r < 138 ? r : 138; ws->cl_tok[nt++] = (uint16_t)(18 | (t - 11) << 5); r -= t; }
                if (r >= 3) { ws->cl_tok[nt++] = (uint16_t)(17 | (r - 3) << 5); r = 0; }
            } else {
                ws->cl_tok[nt++] = (uint16_t)v; r--;
                while (r >= 3) { const int t = r < 6 ? r : 6; ws->cl_tok[nt++] = (uint16_t)(16 | (t - 3) << 5); r -= t; }
            }
            while (r > 0) { ws->cl_tok[nt++] = (uint16_t)v; r--; }
        }
        for (int t = 0; t < nt; t++) ws->cl_freq[ws->cl_tok[t] & 31]++;
        ws->ntok = nt; ws->nlit = nlit; ws->ndist = ndist;
    }
    L.sync();
    pg_def_tree(ws->cl_freq, PG_DEF_NCL, 7, ws->cl_len, ws, L);
    if (L.lane == 0) {
        const uint8_t corder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        int nclen = PG_DEF_NCL;
        while (nclen > 4 && ws->cl_len[corder[nclen - 1]] == 0) nclen--;
        ws->nclen = nclen;
        int64_t hdr = 3 + 5 + 5 + 4 + 3 * nclen;
        for (int t = 0; t < ws->ntok; t++) {
            const int s = ws->cl_tok[t] & 31;
            hdr += ws->cl_len[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0);
        }
        int64_t dyn = 0, fix = 0;
        for (int s = 0; s < PG_DEF_NLIT; s++) {
            const uint32_t f = ws->lit_freq[s];
            if (!f) continue;
            uint32_t c; int l;
            pg_def_fixed(s, c, l);
            const int eb = s > 256 ? pg_def_len_extra(s - 257) : 0;
            dyn += (int64_t)f * (ws->lit_len[s] + eb);
            fix += (int64_t)f * (l + eb);
        }
        dyn += (int64_t)ws->dist_freq[0] * ws->dist_len[0];
        fix += (int64_t)ws->dist_freq[0] * 5;
        const int64_t dyn_end = hdr + dyn, fix_end = 3 + fix;   // end-of-block included (counted in lit_freq[256])
        // a last chunk pads to a byte; any other appends an empty stored block (3 bits, pad, 4 bytes)
        const int64_t dyn_bytes = last ? (dyn_end + 7) / 8 : (dyn_end + 3 + 7) / 8 + 4;
        const int64_t fix_bytes = last ? (fix_end + 7) / 8 : (fix_end + 3 + 7) / 8 + 4;
        const int64_t sto_bytes = n + 5;
        if (dyn_bytes <= fix_bytes && dyn_bytes <= sto_bytes) { ws->mode = PG_DEF_MODE_DYNAMIC; ws->size = dyn_bytes; ws->hdr_bits = hdr; }
        else if (fix_bytes <= sto_bytes) { ws->mode = PG_DEF_MODE_FIXED; ws->size = fix_bytes; ws->hdr_bits = 3; }
        else { ws->mode = PG_DEF_MODE_STORED; ws->size = sto_bytes; ws->hdr_bits = 0; }
        if (ws->mode == PG_DEF_MODE_DYNAMIC) {
            pg_def_codes(ws->lit_len, PG_DEF_NLIT, ws->lit_code);
            pg_def_codes(ws->dist_len, PG_DEF_NDIST, ws->dist_code);
            pg_def_codes(ws->cl_len, PG_DEF_NCL, ws->cl_code);
        }
    }
    L.sync();
    const int mode = ws->mode;
    const int64_t size = ws->size;
    if (mode == PG_DEF_MODE_STORED) {
        if (L.lane == 0) {
            out[0] = last ? 1 : 0;                                 // BFINAL, BTYPE 00, padding
            out[1] = (uint8_t)(n & 0xFF); out[2] = (uint8_t)(n >> 8);
            out[3] = (uint8_t)(~n & 0xFF); out[4] = (uint8_t)((~n >> 8) & 0xFF);
        }
        for (int64_t j = L.lane; j < n; j += L.n) out[5 + j] = in[j];
        L.sync();
        return size;
    }
    uint32_t *w = (uint32_t *)out;
    for (int64_t j = L.lane; j < (size + 3) / 4; j += L.n) w[j] = 0;
    const int fixed = mode == PG_DEF_MODE_FIXED;
    PgDefCount cnt{ws, fixed, 0};
    pg_def_walk(in, n, L, cnt);
    ws->part[L.lane] = (uint32_t)cnt.bits;
    L.sync();
    if (L.lane == 0) {
        uint32_t acc = (uint32_t)ws->hdr_bits;
        for (int l = 0; l < L.n; l++) { const uint32_t b = ws->part[l]; ws->part[l] = acc; acc += b; }
        PgBitOut o;
        o.init(w, 0);
        o.put(last ? 1 : 0, 1);
        o.put((uint32_t)mode, 2);
        if (!fixed) {
            const uint8_t corder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
            o.put((uint32_t)(ws->nlit - 257), 5);
            o.put((uint32_t)(ws->ndist - 1), 5);
            o.put((uint32_t)(ws->nclen - 4), 4);
            for (int i = 0; i < ws->nclen; i++) o.put(ws->cl_len[corder[i]], 3);
            for (int t = 0; t < ws->ntok; t++) {
                const int s = ws->cl_tok[t] & 31, x = ws->cl_tok[t] >> 5;
                o.put(ws->cl_code[s], ws->cl_len[s]);
                if (s == 16) o.put((uint32_t)x, 2);
                else if (s == 17) o.put((uint32_t)x, 3);
                else if (s == 18) o.put((uint32_t)x, 7);
            }
        }
        o.flush();
        // end of block, then the byte-aligning empty stored block of a chunk that is not the last
        PgDefEmit e{ws, fixed, PgBitOut()};
        e.o.init(w, acc);
        e.sym(256);
        if (!last) {
            const int64_t at = acc + (fixed ? 7 : ws->lit_len[256]) + 3;
            e.o.put(0, 3);
            const int pad = (int)((8 - (at & 7)) & 7);
            if (pad) e.o.put(0, pad);
            e.o.put(0, 16);
            e.o.put(0xFFFF, 16);
        }
        e.o.flush();
    }
    L.sync();
    PgDefEmit e{ws, fixed, PgBitOut()};
    e.o.init(w, ws->part[L.lane]);
    pg_def_walk(in, n, L, e);
    e.o.flush();
    L.sync();
    return size;
}
