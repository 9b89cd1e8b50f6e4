// fastq_chunk.cuh - the line-role logic of the FASTQ pack (fastq_pack.cu), written as host+device functions so
// tests/fastq_emul.cu can check it on the CPU.
//
// A FASTQ record is four lines: header ('@'), sequence, separator ('+'), quality.  The role of a line is its index in
// the file mod 4, so the role of a byte is (line ends before it) mod 4: a byte belongs to the line it ends.  What a
// span of bytes hands on is its line-end count mod 4 - the phase - which composes by addition, so a tile's entry phase
// is a plain prefix sum of line-end counts.  Line ends are classify32's `nl` mask: real '\n' bytes plus the last byte
// of the input (a line without a final newline still ends there, as for FASTA).
#pragma once
#include "fasta_chunk.cuh"

// exclusive prefix XOR over the 32 bits of x: bit i = parity of the set bits below i
PG_HD uint32_t fq_pxor_excl32(uint32_t x) {
    x ^= x << 1; x ^= x << 2; x ^= x << 4; x ^= x << 8; x ^= x << 16;
    return x << 1;
}

// Role of every byte of a 32-byte chunk whose first byte lies in a line of role `phase` (0..3): two bit planes, role
// of byte i = lo_i + 2 hi_i.  A 2-bit counter of the line ends below each byte, added to the phase.
struct FqRoles { uint32_t lo, hi; };
PG_HD FqRoles fq_roles32(uint32_t nl, uint32_t phase) {
    const uint32_t c0 = fq_pxor_excl32(nl);              // bit 0 of the count: parity of the line ends below
    const uint32_t c1 = fq_pxor_excl32(nl & c0);         // bit 1 flips at every second line end
    const uint32_t e0 = (phase & 1u) ? 0xFFFFFFFFu : 0u, e1 = (phase & 2u) ? 0xFFFFFFFFu : 0u;
    FqRoles r;
    r.lo = c0 ^ e0;
    r.hi = c1 ^ e1 ^ (c0 & e0);
    return r;
}
PG_HD uint32_t fq_role_mask(const FqRoles &r, uint32_t role) {
    return ((role & 1u) ? r.lo : ~r.lo) & ((role & 2u) ? r.hi : ~r.hi);
}

// bytes of the chunk that lie inside the input; left = input bytes from the chunk's first byte on (may be <= 0)
PG_HD uint32_t fq_infile32(int64_t left) { return left >= 32 ? 0xFFFFFFFFu : (left > 0 ? (1u << left) - 1u : 0u); }

// bytes of the chunk that start a line; prev_nl = 1 when the byte before the chunk ends a line or the chunk starts the input
PG_HD uint32_t fq_line_starts32(uint32_t nl, uint32_t prev_nl, uint32_t infile) { return ((nl << 1) | (prev_nl & 1u)) & infile; }

// What one chunk contributes for each entry phase e of its TILE (the chunk's own phase is e + lines before it in the
// tile): bases and record starts, as the counts for tile phase 0 rotated.  seq[j] / rec[j] = bases / header-line starts
// whose role is j when the chunk is entered at phase 0.
struct FqChunkCount { uint32_t seq[4], rec[4]; };
PG_HD FqChunkCount fq_chunk_count(uint32_t nl, uint32_t infile, uint32_t ls, uint32_t phase) {
    const FqRoles r = fq_roles32(nl, phase);
    const uint32_t base = ~nl & infile;
    FqChunkCount c;
#pragma unroll
    for (uint32_t j = 0; j < 4; j++) {
        const uint32_t m = fq_role_mask(r, j);
        c.seq[j] = pg_popc(base & m);
        c.rec[j] = pg_popc(ls & m);
    }
    return c;
}
// bases / record starts of a span whose counts for phase 0 are seq[] / rec[], entered at phase e
PG_HD uint32_t fq_sel4(const uint32_t v[4], uint32_t j) { return j == 0 ? v[0] : (j == 1 ? v[1] : (j == 2 ? v[2] : v[3])); }
PG_HD uint32_t fq_bases_at(const uint32_t seq[4], uint32_t e) { return fq_sel4(seq, (1u - e) & 3u); }
PG_HD uint32_t fq_recs_at(const uint32_t rec[4], uint32_t e) { return fq_sel4(rec, (0u - e) & 3u); }

// Malformed-record kinds (pg_fastq_scan_pack's d_status[1])
enum { FQ_OK = 0, FQ_BAD_HEADER = 1, FQ_BAD_SEPARATOR = 2, FQ_BAD_QUALITY_LENGTH = 3, FQ_TRUNCATED = 4 };

// The check of record g, from what the pack recorded: its header-line byte, the first byte of its separator line (when
// that line exists), the start of its quality line and the end of that line (exclusive, without the '\n'), the length of
// its sequence line.  Lines that do not exist are passed as sep_byte < 0 / qual_start < 0.
PG_HD int fq_record_kind(int hdr_byte, int sep_byte, int64_t qual_start, int64_t qual_end, int64_t seq_len) {
    if (hdr_byte != '@') return FQ_BAD_HEADER;
    if (sep_byte < 0) return FQ_TRUNCATED;
    if (sep_byte != '+') return FQ_BAD_SEPARATOR;
    if (qual_start < 0) return FQ_TRUNCATED;
    if (qual_end - qual_start != seq_len) return FQ_BAD_QUALITY_LENGTH;
    return FQ_OK;
}
