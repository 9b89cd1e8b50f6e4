// inflate_emul.cu - the BGZF decoder core (pangenome_b200/csrc/inflate.cuh) compiled for the CPU: one lane per member
// instead of a warp, otherwise the same source the kernel runs.  Lets tests/test_inflate_host.py check every decoding
// rule against zlib without a GPU.
#include <stdint.h>
#include <vector>
#include "../pangenome_b200/csrc/inflate.cuh"

namespace {
const uint32_t *crc_table() {
    static uint32_t tab[256];
    static bool done = false;
    if (!done) {
        for (uint32_t i = 0; i < 256; i++) tab[i] = pg_crc_entry(i);
        done = true;
    }
    return tab;
}
}  // namespace

// raw DEFLATE src[slen] -> dst[dlen]; out[0] = produced, out[1] = consumed, out[2] = CRC-32 of dst[0, produced)
extern "C" int emul_inflate_raw(const uint8_t *src, int64_t slen, uint8_t *dst, int64_t dlen, int64_t *out) {
    PgInflateWs ws;
    PgLanes L{0, 1};
    int64_t produced = 0, consumed = 0;
    const int err = pg_inflate_raw(src, slen, dst, dlen, &ws, L, &produced, &consumed);
    out[0] = produced;
    out[1] = consumed;
    out[2] = err ? 0 : pg_crc32_lanes(dst, produced, crc_table(), &ws, L);
    return err;
}

// one BGZF member gz[glen] -> exactly out[olen]
extern "C" int emul_bgzf_member(const uint8_t *gz, int64_t glen, uint8_t *out, int64_t olen) {
    PgInflateWs ws;
    return pg_bgzf_member(gz, glen, out, olen, crc_table(), &ws, PgLanes{0, 1});
}

// the CRC-32 of buf[n] as the kernel's 32 lanes compute it: per-segment CRCs chained by pg_crc_combine
extern "C" uint32_t emul_crc32_segments(const uint8_t *buf, int64_t n, int lanes) {
    const uint32_t *tab = crc_table();
    const int64_t seg = (n + lanes - 1) / lanes;
    uint32_t crc = 0;
    for (int l = 0; l < lanes; l++) {
        int64_t a = l * seg, b = a + seg;
        if (a > n) a = n;
        if (b > n) b = n;
        uint32_t c = 0xFFFFFFFFu;
        for (int64_t i = a; i < b; i++) c = tab[(c ^ buf[i]) & 0xFF] ^ (c >> 8);
        c ^= 0xFFFFFFFFu;
        crc = l == 0 ? c : pg_crc_combine(crc, c, b - a);
    }
    return crc;
}
