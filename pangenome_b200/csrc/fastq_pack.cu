// fastq_pack.cu - the FASTQ pack: what K1 (fasta_pack.cu) produces for a FASTA file, produced from a FASTQ file.
//
// A FASTQ file F is packed exactly as the FASTA file fasta(F) - every record written as its header line with '>' for
// '@' and its sequence line - would be: the same 2-bit / 1-bit planes, seq_off and counts[0..1]; hdr_off holds the
// offsets of the '@' lines of F.  Every byte of a sequence line but its '\n' is a base (so '\r' is one, Q9); header,
// separator and quality lines give no bases.  The role of a line is its index mod 4 (fastq_chunk.cuh), and five
// launches over the 16 KB tiles of K1x do the work:
//   A  fq_tile_aggs  per tile: line ends, and for each of the 4 entry phases its bases and record starts (one uint4),
//                    plus the position of its last byte that is not a '\n'
//   B  fq_scan       one CTA: each tile's entry phase (a sum of line ends mod 4), base rank and record rank
//   C  fq_pack       every tile again: byte roles from the phase, 2-bit / 1-bit pack staged in shared memory and stored
//                    as whole words (K1x's write-out), the record index, and the start of every separator and quality line
//   D  fq_check      per record: '@' header, '+' separator, quality length = sequence length, four lines present
//   E  fq_finish     one thread: the first bad record into d_status, or the record count without the trailing blank
//                    lines into d_counts[0]
// Validation is part of the launch, so a malformed file ends in d_status and never in a fault: every read and write is
// bounded by nbytes and cap_records.
#include "fastq_chunk.cuh"

namespace {

constexpr int FQ_THREADS = 512;
constexpr int FQ_TILE = FQ_THREADS * 32;                 // 16 KB, one 32-byte chunk per thread
constexpr int FQ_NW = FQ_THREADS / 32;
constexpr int FQ_PKW = (FQ_TILE + 32) / 16 + 2;          // staged pk2 words per tile
constexpr int FQ_AMW = (FQ_TILE + 32) / 32 + 2;
constexpr int FQB_THREADS = 1024;

struct FqEntry { uint64_t seq, rec; uint32_t phase, pad; };
// launch-wide values in the workspace: written by fq_scan, read by fq_check / fq_finish
struct FqState { unsigned long long content_end, n_lines, bad, n_real; };

__device__ __forceinline__ void fq_load32(const uint8_t *p, int64_t nbytes, int64_t off, uint32_t w[8]) {
    const int64_t left = nbytes - off;
    if (left >= 32) {
        const uint4 a = __ldg(reinterpret_cast<const uint4 *>(p + off)), b = __ldg(reinterpret_cast<const uint4 *>(p + off) + 1);
        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
    } else {
        uint64_t q[4] = {0, 0, 0, 0};
        for (int i = 0; i < (int)left; i++) {            // the ragged chunk(s) at the end of the input
            const uint64_t v = (uint64_t)p[off + i] << (8 * (i & 7));
            if (i < 8) q[0] |= v; else if (i < 16) q[1] |= v; else if (i < 24) q[2] |= v; else q[3] |= v;
        }
#pragma unroll
        for (int i = 0; i < 4; i++) { w[2 * i] = (uint32_t)q[i]; w[2 * i + 1] = (uint32_t)(q[i] >> 32); }
    }
}
// the byte before the chunk ends a line (or the chunk starts the input): lane 0 looks, the others take the neighbour's bit 31
__device__ __forceinline__ uint32_t fq_prev_nl(const uint8_t *p, int64_t nbytes, int64_t off, uint32_t nl) {
    uint32_t v = __shfl_up_sync(0xffffffffu, nl >> 31, 1);
    if ((threadIdx.x & 31) == 0) v = off == 0 ? 1u : (off - 1 < nbytes ? (uint32_t)(p[off - 1] == '\n') : 1u);
    return v;
}
// exclusive block-wide sum (NT threads); s_w: NT / 32 words.  Two barriers; s_w may be reused after it returns.
template <int NT, typename T>
__device__ __forceinline__ T fq_block_excl(T v, T *s_w, T &total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const T y = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += y; }
    if (lane == 31) s_w[warp] = inc;
    __syncthreads();
    T w = lane < NT / 32 ? s_w[lane] : (T)0, winc = w;
#pragma unroll
    for (int d = 1; d < NT / 32; d <<= 1) { const T y = __shfl_up_sync(0xffffffffu, winc, d); if (lane >= d) winc += y; }
    const T base = __shfl_sync(0xffffffffu, winc - w, warp);
    total = __shfl_sync(0xffffffffu, winc, NT / 32 - 1);
    __syncthreads();
    return base + inc - v;
}

__global__ void __launch_bounds__(FQ_THREADS)
fq_tile_aggs(const uint8_t *__restrict__ fq, int64_t nbytes, int64_t ntiles, uint4 *__restrict__ agg_cnt, uint4 *__restrict__ agg_meta) {
    __shared__ uint32_t s_w[FQ_NW];
    __shared__ uint32_t s_cnt[4], s_real, s_last;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        if (threadIdx.x < 4) s_cnt[threadIdx.x] = 0;
        if (threadIdx.x == 0) { s_real = 0; s_last = 0; }
        const int64_t off = tile * FQ_TILE + (int64_t)threadIdx.x * 32;
        uint32_t w[8];
        fq_load32(fq, nbytes, off, w);
        const int64_t left = nbytes - off;
        const Cls32 c = classify32<true>(w, left);
        const uint32_t infile = fq_infile32(left);
        const uint32_t nlc = pg_popc(c.nl & infile);
        uint32_t tile_nl;
        const uint32_t lines = fq_block_excl<FQ_THREADS>(nlc, s_w, tile_nl);       // barriers inside: the zeroed sums are visible
        const uint32_t ls = fq_line_starts32(c.nl, fq_prev_nl(fq, nbytes, off, c.nl), infile);
        const FqChunkCount k = fq_chunk_count(c.nl, infile, ls, lines & 3u);
        uint32_t content = ~c.nl & infile;                   // bytes that are not '\n': the last byte of the input is a line
        if (left > 0 && left <= 32 && fq[nbytes - 1] != '\n') content |= 1u << (left - 1);   // end in c.nl whatever it is
        uint32_t rnl = c.real_nl, last = content ? threadIdx.x * 32u + (uint32_t)pg_msb(content) + 1u : 0u;
        rnl = __reduce_add_sync(0xffffffffu, rnl);
        last = __reduce_max_sync(0xffffffffu, last);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t v = __reduce_add_sync(0xffffffffu, k.seq[j] | (k.rec[j] << 16));   // both halves stay below 2^15
            if ((threadIdx.x & 31) == 0 && v) atomicAdd(&s_cnt[j], v);
        }
        if ((threadIdx.x & 31) == 0) {
            if (rnl) atomicAdd(&s_real, rnl);
            if (last) atomicMax(&s_last, last);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            agg_cnt[tile] = make_uint4(s_cnt[0], s_cnt[1], s_cnt[2], s_cnt[3]);
            agg_meta[tile] = make_uint4(tile_nl, s_real, s_last, 0u);
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(FQB_THREADS)
fq_scan(const uint4 *__restrict__ agg_cnt, const uint4 *__restrict__ agg_meta, int64_t ntiles, int64_t nbytes,
        FqEntry *__restrict__ entries, uint32_t *__restrict__ pk2, uint32_t *__restrict__ amb, int64_t *__restrict__ seq_off,
        int64_t cap_records, int64_t *__restrict__ counts, FqState *__restrict__ st) {
    __shared__ unsigned long long s_w[FQB_THREADS / 32];
    __shared__ unsigned long long s_last;
    const int t = threadIdx.x;
    const int64_t per = (ntiles + FQB_THREADS - 1) / FQB_THREADS;
    const int64_t lo = (int64_t)t * per < ntiles ? (int64_t)t * per : ntiles, hi = lo + per < ntiles ? lo + per : ntiles;
    if (t == 0) s_last = 0;
    unsigned long long nl = 0, real = 0, last = 0;
    for (int64_t i = lo; i < hi; i++) {
        const uint4 m = agg_meta[i];
        nl += m.x; real += m.y;
        if (m.z) last = (unsigned long long)(i * FQ_TILE + m.z);
    }
    unsigned long long n_lines, n_real_nl;
    const unsigned long long lines_before = fq_block_excl<FQB_THREADS>(nl, s_w, n_lines);
    fq_block_excl<FQB_THREADS>(real, s_w, n_real_nl);
    if (last) atomicMax(&s_last, last);
    // this thread's tiles at their entry phases
    uint32_t ph = (uint32_t)(lines_before & 3u);
    unsigned long long bases = 0, recs = 0;
    for (int64_t i = lo; i < hi; i++) {
        const uint4 k = agg_cnt[i];
        const uint32_t seq[4] = {k.x & 0xFFFFu, k.y & 0xFFFFu, k.z & 0xFFFFu, k.w & 0xFFFFu};
        const uint32_t rec[4] = {k.x >> 16, k.y >> 16, k.z >> 16, k.w >> 16};
        bases += fq_bases_at(seq, ph); recs += fq_recs_at(rec, ph);
        ph = (ph + agg_meta[i].x) & 3u;
    }
    unsigned long long tot_bases, tot_recs;
    unsigned long long seq = fq_block_excl<FQB_THREADS>(bases, s_w, tot_bases);
    unsigned long long rec = fq_block_excl<FQB_THREADS>(recs, s_w, tot_recs);      // its barriers also publish s_last
    ph = (uint32_t)(lines_before & 3u);
    for (int64_t i = lo; i < hi; i++) {
        FqEntry e; e.seq = seq; e.rec = rec; e.phase = ph; e.pad = 0;
        entries[i] = e;
        pk2[seq >> 4] = 0; amb[seq >> 5] = 0;                 // words shared between neighbouring tiles (the tiles OR into them)
        const uint4 k = agg_cnt[i];
        const uint32_t sq[4] = {k.x & 0xFFFFu, k.y & 0xFFFFu, k.z & 0xFFFFu, k.w & 0xFFFFu};
        const uint32_t rc[4] = {k.x >> 16, k.y >> 16, k.z >> 16, k.w >> 16};
        seq += fq_bases_at(sq, ph); rec += fq_recs_at(rc, ph);
        ph = (ph + agg_meta[i].x) & 3u;
    }
    if (t == 0) {
        counts[0] = (int64_t)tot_recs;                        // header-line starts, trailing blank lines included: fq_finish
        counts[1] = (int64_t)tot_bases;                       // takes those off once the index is complete
        counts[2] = (int64_t)n_real_nl;
        counts[3] = nbytes == 0 ? 1 : 0;
        if ((int64_t)tot_recs <= cap_records) seq_off[tot_recs] = (int64_t)tot_bases;
        for (int i = 0; i < 16; i++) { pk2[(tot_bases >> 4) + i] = 0; amb[(tot_bases >> 5) + i] = 0; }   // padding the k-mer kernels may read
        st->content_end = s_last; st->n_lines = n_lines; st->bad = ~0ull; st->n_real = 0;
    }
}

__global__ void __launch_bounds__(FQ_THREADS)
fq_pack(const uint8_t *__restrict__ fq, int64_t nbytes, int64_t ntiles, const FqEntry *__restrict__ entries,
        uint32_t *__restrict__ pk2, uint32_t *__restrict__ amb, int64_t *__restrict__ hdr_off, int64_t *__restrict__ seq_off,
        int64_t cap_records, int64_t *__restrict__ sep_start, int64_t *__restrict__ qual_start) {
    __shared__ uint32_t s_w[FQ_NW];
    __shared__ uint32_t s_pk[FQ_PKW];
    __shared__ uint32_t s_am[FQ_AMW];
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const FqEntry e = entries[tile];
        const int64_t off = tile * FQ_TILE + (int64_t)threadIdx.x * 32;
        uint32_t w[8];
        fq_load32(fq, nbytes, off, w);                       // loads in flight while the staging is cleared
        for (int i = threadIdx.x; i < FQ_PKW; i += FQ_THREADS) s_pk[i] = 0;
        for (int i = threadIdx.x; i < FQ_AMW; i += FQ_THREADS) s_am[i] = 0;
        const int64_t left = nbytes - off;
        const Cls32 c = classify32<false>(w, left);
        const uint32_t infile = fq_infile32(left);
        uint32_t unused;
        const uint32_t lines = fq_block_excl<FQ_THREADS>(pg_popc(c.nl & infile), s_w, unused);   // barriers: staging zeroed
        const FqRoles r = fq_roles32(c.nl, (e.phase + lines) & 3u);
        const uint32_t ls = fq_line_starts32(c.nl, fq_prev_nl(fq, nbytes, off, c.nl), infile);
        const uint32_t seqmask = fq_role_mask(r, 1) & ~c.nl & infile;
        const uint32_t hs = ls & fq_role_mask(r, 0), s2 = ls & fq_role_mask(r, 2), s3 = ls & fq_role_mask(r, 3);
        // ranks: bases | record starts << 16 before this chunk
        uint32_t total;
        const uint32_t excl = fq_block_excl<FQ_THREADS>(pg_popc(seqmask) | (pg_popc(hs) << 16), s_w, total);
        const uint32_t rank = excl & 0xFFFFu, hrank = excl >> 16;
        const uint32_t a0 = (uint32_t)(e.seq & 31);
        // ---- pack the two 16-byte halves into the shared-memory staging (as k1x_pack)
        uint32_t r2 = rank;
#pragma unroll
        for (int half = 0; half < 2; half++) {
            const uint32_t sm = (seqmask >> (16 * half)) & 0xFFFFu, n = pg_popc(sm);
            if (n) {
                uint32_t d = pext16_2bit(half ? c.dig_hi : c.dig_lo, sm);
                const uint32_t m = pext16_1bit((c.amb >> (16 * half)) & 0xFFFFu, sm);
                if (n < 16) d &= (1u << (2 * n)) - 1u;
                const uint32_t q = a0 + r2, sh = 2 * (q & 15);
                atomicOr(&s_pk[q >> 4], d << sh);
                if (sh && (d >> (32 - sh))) atomicOr(&s_pk[(q >> 4) + 1], d >> (32 - sh));
                if (m) {
                    const uint32_t sh1 = q & 31;
                    atomicOr(&s_am[q >> 5], m << sh1);
                    if (sh1 > 16 && (m >> (32 - sh1))) atomicOr(&s_am[(q >> 5) + 1], m >> (32 - sh1));
                }
            }
            r2 += n;
        }
        if (hs | s2 | s3) {   // line starts of the record index: about one chunk in three on 150 bp reads
            uint32_t x = hs | s2 | s3;
            while (x) {
                const int j = pg_ctz(x); x &= x - 1;
                const uint32_t below = (1u << j) - 1u;
                const int64_t g = (int64_t)(e.rec + hrank + pg_popc(hs & below)) - ((hs >> j) & 1u ? 0 : 1);
                if (g < 0 || g >= cap_records) continue;
                if ((hs >> j) & 1u) {
                    hdr_off[g] = off + j;
                    seq_off[g] = (int64_t)(e.seq + rank + pg_popc(seqmask & below));
                } else if ((s2 >> j) & 1u) {
                    sep_start[g] = off + j;
                } else {
                    qual_start[g] = off + j;
                }
            }
        }
        __syncthreads();
        // ---- write-out: words fully owned by this tile are stored, shared boundary words are OR-ed
        const uint32_t end = a0 + (total & 0xFFFFu);
        uint32_t *gpk = pk2 + ((e.seq >> 5) << 1);
        uint32_t *gam = amb + (e.seq >> 5);
        const uint32_t npk = (end + 15) >> 4, nam = (end + 31) >> 5;
        for (uint32_t x = threadIdx.x; x < npk; x += FQ_THREADS) {
            const uint32_t v = s_pk[x];
            if (16 * x >= a0 && 16 * (x + 1) <= end) gpk[x] = v;
            else if (v) atomicOr(&gpk[x], v);
        }
        for (uint32_t x = threadIdx.x; x < nam; x += FQ_THREADS) {
            const uint32_t v = s_am[x];
            if (32 * x >= a0 && 32 * (x + 1) <= end) gam[x] = v;
            else if (v) atomicOr(&gam[x], v);
        }
        __syncthreads();
    }
}

// Record g is a record when its header line starts before the last byte that is not a '\n'; the groups of four lines
// after that are the blank lines a file may end with.  Only the last group can lack lines (n_lines says which).
__global__ void __launch_bounds__(256)
fq_check(const uint8_t *__restrict__ fq, int64_t nbytes, const int64_t *__restrict__ hdr_off, const int64_t *__restrict__ seq_off,
         const int64_t *__restrict__ sep_start, const int64_t *__restrict__ qual_start, int64_t cap_records,
         const int64_t *__restrict__ counts, FqState *__restrict__ st) {
    const int64_t n_raw = counts[0];
    if (n_raw > cap_records) return;                         // truncated index: the caller packs again with room for it
    const unsigned long long content_end = st->content_end, n_lines = st->n_lines;
    for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < n_raw; g += (int64_t)gridDim.x * blockDim.x) {
        const int64_t h = hdr_off[g];
        if ((unsigned long long)h >= content_end) continue;
        atomicMax(&st->n_real, (unsigned long long)(g + 1));
        const bool has_sep = n_lines > (unsigned long long)(4 * g + 2), has_qual = n_lines > (unsigned long long)(4 * g + 3);
        const int64_t q = has_qual ? qual_start[g] : -1;
        const int64_t q_end = g + 1 < n_raw ? hdr_off[g + 1] - 1 : (fq[nbytes - 1] == '\n' ? nbytes - 1 : nbytes);
        const int kind = fq_record_kind(fq[h], has_sep ? (int)fq[sep_start[g]] : -1, q, q_end, seq_off[g + 1] - seq_off[g]);
        if (kind != FQ_OK) atomicMin(&st->bad, ((unsigned long long)g << 3) | (unsigned long long)kind);
    }
}

__global__ void fq_finish(const int64_t *__restrict__ hdr_off, int64_t *__restrict__ seq_off, int64_t cap_records,
                          int64_t *__restrict__ counts, const FqState *__restrict__ st, int64_t *__restrict__ status) {
    status[0] = -1; status[1] = FQ_OK;
    if (counts[0] > cap_records) return;
    if (st->bad != ~0ull) {
        const int64_t g = (int64_t)(st->bad >> 3);
        status[0] = hdr_off[g]; status[1] = (int64_t)(st->bad & 7u);
        counts[0] = 0; counts[1] = 0; seq_off[0] = 0;        // nothing to build from
        return;
    }
    counts[0] = (int64_t)st->n_real;                           // blank groups hold no bases: seq_off[n_real] = counts[1]
}

struct FqLayout { size_t state, agg_cnt, agg_meta, entries, sep, qual, end; };
FqLayout fq_layout(int64_t nbytes, int64_t cap_records) {
    const size_t nt = (size_t)((nbytes + FQ_TILE - 1) / FQ_TILE < 1 ? 1 : (nbytes + FQ_TILE - 1) / FQ_TILE);
    const size_t cap = (size_t)(cap_records < 1 ? 1 : cap_records);
    FqLayout l;
    l.state = 0;
    l.agg_cnt = 256;
    l.agg_meta = l.agg_cnt + nt * sizeof(uint4);
    l.entries = l.agg_meta + nt * sizeof(uint4);
    l.sep = l.entries + nt * sizeof(FqEntry);
    l.qual = l.sep + cap * sizeof(int64_t);
    l.end = l.qual + cap * sizeof(int64_t);
    return l;
}

}  // namespace

extern "C" int64_t pg_fastq_workspace_bytes(int64_t nbytes, int64_t cap_records) {
    return (int64_t)fq_layout(nbytes < 0 ? 0 : nbytes, cap_records).end;
}

extern "C" int pg_fastq_scan_pack(const uint8_t *d_fastq, int64_t nbytes, uint32_t *d_pk2, uint32_t *d_amb, int64_t cap_bases,
                                  int64_t *d_hdr_off, int64_t *d_seq_off, int64_t cap_records, int64_t *d_counts,
                                  int64_t *d_status, void *d_ws, int64_t ws_bytes, pg_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (nbytes < 0 || !d_pk2 || !d_amb || !d_hdr_off || !d_seq_off || !d_counts || !d_status || !d_ws || cap_records < 0)
        return pg_fail(PG_ERR_INVALID, "pg_fastq_scan_pack: null buffer or negative size");
    if (nbytes > 0 && !d_fastq) return pg_fail(PG_ERR_INVALID, "pg_fastq_scan_pack: d_fastq is null");
    if (cap_bases < nbytes) return pg_fail(PG_ERR_CAPACITY, "pg_fastq_scan_pack: cap_bases %lld < nbytes %lld",
                                           (long long)cap_bases, (long long)nbytes);
    const FqLayout l = fq_layout(nbytes, cap_records);
    if (ws_bytes < (int64_t)l.end)
        return pg_fail(PG_ERR_WORKSPACE, "pg_fastq_scan_pack: workspace %lld < %lld", (long long)ws_bytes, (long long)l.end);
    if ((reinterpret_cast<uintptr_t>(d_fastq) & 15) != 0 || (reinterpret_cast<uintptr_t>(d_ws) & 15) != 0)
        return pg_fail(PG_ERR_INVALID, "pg_fastq_scan_pack: d_fastq and d_ws must be 16-byte aligned");
    char *w = reinterpret_cast<char *>(d_ws);
    FqState *st = reinterpret_cast<FqState *>(w + l.state);
    uint4 *agg_cnt = reinterpret_cast<uint4 *>(w + l.agg_cnt), *agg_meta = reinterpret_cast<uint4 *>(w + l.agg_meta);
    FqEntry *ent = reinterpret_cast<FqEntry *>(w + l.entries);
    int64_t *sep = reinterpret_cast<int64_t *>(w + l.sep), *qual = reinterpret_cast<int64_t *>(w + l.qual);
    const int64_t ntiles = (nbytes + FQ_TILE - 1) / FQ_TILE;
    const int grid = (int)(ntiles < (1ll << 20) ? (ntiles < 1 ? 1 : ntiles) : (1ll << 20));
    if (ntiles > 0) fq_tile_aggs<<<grid, FQ_THREADS, 0, stream>>>(d_fastq, nbytes, ntiles, agg_cnt, agg_meta);
    fq_scan<<<1, FQB_THREADS, 0, stream>>>(agg_cnt, agg_meta, ntiles, nbytes, ent, d_pk2, d_amb, d_seq_off, cap_records, d_counts, st);
    if (ntiles > 0) {
        fq_pack<<<grid, FQ_THREADS, 0, stream>>>(d_fastq, nbytes, ntiles, ent, d_pk2, d_amb, d_hdr_off, d_seq_off, cap_records, sep, qual);
        const int64_t cg = (cap_records + 255) / 256, cmax = (int64_t)pg_num_sms() * 8;
        fq_check<<<(int)(cg < 1 ? 1 : (cg < cmax ? cg : cmax)), 256, 0, stream>>>(d_fastq, nbytes, d_hdr_off, d_seq_off, sep, qual,
                                                                                  cap_records, d_counts, st);
    }
    fq_finish<<<1, 1, 0, stream>>>(d_hdr_off, d_seq_off, cap_records, d_counts, st, d_status);
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}
