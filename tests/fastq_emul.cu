// Host build of the FASTQ pack's per-chunk logic (pangenome_b200/csrc/fastq_chunk.cuh), run in the kernels' order:
// tile aggregates for phase 0, a scan over the tiles, then every chunk again from its entry phase.  Tiles are
// `tile` bytes (a multiple of 32) so a test can put tile boundaries anywhere.  nvcc -O2 --shared -Xcompiler -fPIC.
#include <cstring>
#include <vector>
#include "../pangenome_b200/csrc/fastq_chunk.cuh"

static void load32(const uint8_t *p, int64_t n, int64_t off, uint32_t w[8]) {
    uint8_t b[32] = {0};
    for (int i = 0; i < 32 && off + i < n; i++) b[i] = p[off + i];
    memcpy(w, b, 32);
}

// Outputs: sym[n_bases] = 2-bit digit | amb << 2 of every base in stream order; hdr / seq_off / sep / qual per record
// start (all header-line starts, blank trailing groups included); counts = {records, bases, line ends, content end}.
// Returns 0, or -1 if the tile aggregates disagree with the second pass.
extern "C" int64_t emul_fq_pack(const uint8_t *p, int64_t n, int64_t tile, uint8_t *sym, int64_t *hdr, int64_t *seq_off,
                                int64_t *sep, int64_t *qual, int64_t cap, int64_t *counts) {
    const int64_t ntiles = (n + tile - 1) / tile;
    std::vector<uint32_t> tseq(4 * ntiles), trec(4 * ntiles), tnl(ntiles);
    int64_t content_end = 0;
    for (int64_t t = 0; t < ntiles; t++) {                        // pass A
        uint32_t lines = 0;
        for (int64_t off = t * tile; off < (t + 1) * tile; off += 32) {
            uint32_t w[8];
            load32(p, n, off, w);
            const Cls32 c = classify32<true>(w, n - off);
            const uint32_t inf = fq_infile32(n - off);
            const uint32_t prev = off == 0 ? 1u : (off - 1 < n ? (uint32_t)(p[off - 1] == '\n') : 1u);
            const FqChunkCount k = fq_chunk_count(c.nl, inf, fq_line_starts32(c.nl, prev, inf), lines & 3u);
            for (int j = 0; j < 4; j++) { tseq[4 * t + j] += k.seq[j]; trec[4 * t + j] += k.rec[j]; }
            lines += pg_popc(c.nl & inf);
            for (int i = 0; i < 32 && off + i < n; i++) if (p[off + i] != '\n') content_end = off + i + 1;
        }
        tnl[t] = lines;
    }
    uint64_t seq = 0, rec = 0, nl = 0;
    for (int64_t t = 0; t < ntiles; t++) {                        // pass B (sequential) + pass C
        const uint32_t ph = (uint32_t)(nl & 3u);
        const uint64_t seq_end = seq + fq_bases_at(&tseq[4 * t], ph), rec_end = rec + fq_recs_at(&trec[4 * t], ph);
        uint32_t lines = 0;
        for (int64_t off = t * tile; off < (t + 1) * tile; off += 32) {
            uint32_t w[8];
            load32(p, n, off, w);
            const Cls32 c = classify32<false>(w, n - off);
            const uint32_t inf = fq_infile32(n - off);
            const uint32_t prev = off == 0 ? 1u : (off - 1 < n ? (uint32_t)(p[off - 1] == '\n') : 1u);
            const FqRoles r = fq_roles32(c.nl, (ph + lines) & 3u);
            const uint32_t ls = fq_line_starts32(c.nl, prev, inf);
            const uint32_t seqmask = fq_role_mask(r, 1) & ~c.nl & inf, hs = ls & fq_role_mask(r, 0);
            const uint32_t s2 = ls & fq_role_mask(r, 2), s3 = ls & fq_role_mask(r, 3);
            for (int i = 0; i < 32; i++) {
                const uint32_t bit = 1u << i;
                if (hs & bit) {
                    if ((int64_t)rec < cap) { hdr[rec] = off + i; seq_off[rec] = (int64_t)seq; }
                    rec++;
                } else if ((s2 | s3) & bit) {
                    const int64_t g = (int64_t)rec - 1;
                    if (g >= 0 && g < cap) ((s2 & bit) ? sep : qual)[g] = off + i;
                }
                if (seqmask & bit) {
                    const uint32_t d = ((i < 16 ? c.dig_lo : c.dig_hi) >> (2 * (i & 15))) & 3u;
                    sym[seq++] = (uint8_t)(d | (((c.amb >> i) & 1u) << 2));
                }
            }
            lines += pg_popc(c.nl & inf);
        }
        if (seq != seq_end || rec != rec_end) return -1;
        nl += lines;
    }
    if ((int64_t)rec <= cap) seq_off[rec] = (int64_t)seq;
    counts[0] = (int64_t)rec; counts[1] = (int64_t)seq; counts[2] = (int64_t)nl; counts[3] = content_end;
    return 0;
}

extern "C" int emul_fq_kind(int hdr_byte, int sep_byte, int64_t qual_start, int64_t qual_end, int64_t seq_len) {
    return fq_record_kind(hdr_byte, sep_byte, qual_start, qual_end, seq_len);
}
