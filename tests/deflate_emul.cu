// deflate_emul.cu - the chunk encoder core (pangenome_b200/csrc/deflate.cuh) compiled for the CPU: one lane per chunk
// instead of a CTA, otherwise the same source the kernel runs.  Lets tests/test_deflate_host.py check the encoder against
// zlib and the repo's own decoder without a GPU, and gives the GPU tests the bytes the kernel must reproduce.
#include <stdint.h>
#include <string.h>
#include <vector>
#include "../pangenome_b200/csrc/deflate.cuh"

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

// One member src[n] cut into chunks of `chunk` bytes -> out (capacity: n + 5 per chunk + 8).  sizes[i] / crcs[i]: the
// compressed size and CRC-32 of chunk i (arrays of max(1, ceil(n / chunk)) entries).  Returns the member's compressed
// size; *crc = CRC-32 of src, chained from the chunk CRCs with pg_crc_combine.
extern "C" int64_t emul_deflate(const uint8_t *src, int64_t n, int64_t chunk, uint8_t *out, int64_t *sizes, uint32_t *crcs,
                                uint32_t *crc) {
    if (chunk < 1 || chunk > PG_DEF_MAX_CHUNK) return -1;
    const int64_t nchunks = n ? (n + chunk - 1) / chunk : 1;
    std::vector<uint32_t> slot((size_t)(chunk + 8 + 3) / 4);
    PgDeflateWs ws;
    PgInflateWs iws;
    int64_t pos = 0;
    uint32_t all = 0;
    for (int64_t c = 0; c < nchunks; c++) {
        const int64_t a = c * chunk, len = (n - a) < chunk ? (n - a) : chunk;
        const int64_t size = pg_deflate_chunk(src + a, len, c == nchunks - 1, (uint8_t *)slot.data(), &ws, PgDefLanes{0, 1});
        memcpy(out + pos, slot.data(), (size_t)size);
        pos += size;
        sizes[c] = size;
        crcs[c] = pg_crc32_lanes(src + a, len, crc_table(), &iws, PgLanes{0, 1});
        all = c == 0 ? crcs[c] : pg_crc_combine(all, crcs[c], len);
    }
    *crc = all;
    return pos;
}
