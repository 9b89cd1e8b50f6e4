// compact_build.cu - the streaming dBG build on COMPACT (8-byte) update records: K2a-c -> K2c-c -> K3s-c.
//
// Why: every stage after the extraction is a stream of update records - K2a writes them, K2c reads and re-writes them once
// per partition level, K3s reads them - and at 16 bytes {base-5 key, masks, increment} they are 3.2 of the ~4 GB a
// config-2 build moves.  An interior position (the k-mer, the base before and the base after it are ACGT inside one
// record - all but ~2(k+16) positions per record of a genome) needs 2k <= 54 bits of 2-bit code plus 4 bits of
// (previous, next) base, one strand bit and one palindrome bit: 8 bytes (kmer_core.cuh, pg_crec_pack).  That halves the
// traffic of K2a's write-out, K2c and K3s' read, AND takes the base-5 arithmetic out of the extraction: both strands'
// codes roll with shifts instead of two 64-bit multiply chains per position (kmer_numba.py:975-988, 1064-1082 restated in
// the 2-bit domain; the base-5 key the reference's table holds is produced once per DISTINCT key, when K3s-c writes a
// finished region to HBM).
//
//   K2a-c  thread = 16 positions.  Interior: bucket = top bits of mix64(2-bit key), rank inside the tile's run from the
//          histogram atomic, scan, every record stored at its sorted position of an 8-byte shared-memory staging,
//          linear copy-out (the multisplit of multisplit.cu without the tile sort's permutation and gather passes,
//          which were half of K2a's instructions).  With a compile-time k the two windows of a position are constant
//          funnel shifts of three digit words, so the records are derived twice (before and after the scan) rather
//          than held.  Everything else (record edges with '#', '$' and Q1, ambiguity codes): the generic per-position
//          path of partition.cu, emitted as 16-byte WIDE records straight into the build's wide spill.  Across GPUs
//          (PEER) the bucket is the owner rank and the runs are stored into the owners' receive buffers over NVLink.
//   K2c-c  register-held multisplit of 8-byte records, 16 per thread, one level of <= 2^8 ways per launch; K2b-c: the
//          same kernel on what arrived from the other ranks (one segment per source -> hash-prefix buckets).
//   K3s-c  one CTA per 4096-slot region: the region lives in shared memory keyed by the 2-bit code; the value words come
//          from the 16-entry table by the record's context bits; the region is converted to base-5 keys (6 table
//          look-ups per live slot) as the LAST round writes it to HBM.  Between the rounds of a multi-round build the
//          2-bit keys stay in HBM under PG_C_HBM_FLAG (a key with an ambiguity digit keeps its base-5 form and gets
//          PG_WIDE_FLAG in shared memory).  The wide spill is upserted afterwards with L2 atomics.
//
// The table this produces is placed by the hash of the 2-bit code (pg_table.hash_kind = 1, table_dev.cuh tv_home), probes
// inside 4096-slot regions like every region-built table, and holds exactly the slots the 16-byte path would: same keys,
// masks, counts (tests/test_gpu_builder.py compares both with the oracle).
#include "tile_sort.cuh"

namespace {

struct CBuckets {
    uint2 *records; unsigned long long *counts; int64_t part_cap; int bits;
    uint4 *wide; unsigned long long *wide_count; int64_t wide_cap;
    // fused exchange (K2a-c across GPUs): bucket = OWNER rank; bucket o is written straight into rank o's receive buffers
    // over NVLink, at the slice reserved for source rank my_rank - compact records at peers[o] + my_rank * part_cap, wide
    // ones at wide_peers[o] + my_rank * wide_cap, counted in counts[o] / wide_count[o]
    uint2 *const *peers; uint4 *const *wide_peers; int my_rank;
};

constexpr uint32_t C_NONE = 0xFFFFFFFFu;

__device__ __forceinline__ void wide_emit(const CBuckets &b, uint64_t key5, uint32_t masks, uint32_t inc) {
    const unsigned long long at = atomicAdd(b.wide_count, 1ull);
    if ((int64_t)at < b.wide_cap) b.wide[at] = make_uint4((uint32_t)key5, (uint32_t)(key5 >> 32), masks, inc);
}
// the same towards the owner rank of the key (fused exchange)
__device__ __noinline__ void wide_emit_owner(uint4 *const *wide_peers, unsigned long long *wide_counts, int64_t wide_cap, int my_rank,
                                             uint32_t owner, uint64_t key5, uint32_t masks, uint32_t inc) {
    const unsigned long long at = atomicAdd(wide_counts + owner, 1ull);
    if ((int64_t)at < wide_cap) wide_peers[owner][(int64_t)my_rank * wide_cap + (int64_t)at] = make_uint4((uint32_t)key5, (uint32_t)(key5 >> 32), masks, inc);
}
__device__ __noinline__ void wide_emit_compact_owner(uint4 *const *wide_peers, unsigned long long *wide_counts, int64_t wide_cap, int my_rank,
                                                     uint32_t owner, uint64_t rec, int k) {
    const uint32_t ctx = (uint32_t)(rec >> PG_C_KEYBITS);
    uint32_t masks, inc;
    pg_crec_vals(ctx, pg_vlut_entry(ctx & 15u), masks, inc);
    wide_emit_owner(wide_peers, wide_counts, wide_cap, my_rank, owner, pg_code5_of2_loop(rec & PG_C_KEYMASK, k), masks, inc);
}
// a compact record whose bucket is full travels on as a wide one (rare: hash skew)
__device__ __noinline__ void wide_emit_compact(uint4 *wide, unsigned long long *wide_count, int64_t wide_cap, uint64_t rec, int k) {
    const uint32_t ctx = (uint32_t)(rec >> PG_C_KEYBITS);
    uint32_t masks, inc;
    pg_crec_vals(ctx, pg_vlut_entry(ctx & 15u), masks, inc);
    const uint64_t key5 = pg_code5_of2_loop(rec & PG_C_KEYMASK, k);
    const unsigned long long at = atomicAdd(wide_count, 1ull);
    if ((int64_t)at < wide_cap) wide[at] = make_uint4((uint32_t)key5, (uint32_t)(key5 >> 32), masks, inc);
}
__device__ __forceinline__ uint2 ld_stream8(const uint2 *p) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream8_l2first(uint2 *p, uint64_t v, uint64_t pol) {
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.v2.u32 [%0], {%1,%2}, %3;"
                 ::"l"(p), "r"((uint32_t)v), "r"((uint32_t)(v >> 32)), "l"(pol) : "memory");
}

// Scan of a tile's bucket histogram, room reservation in the output buckets, per-bucket destination pointers: steps 2 of
// the register-held multisplit, shared by K2a-c and K2c-c.  Call with all threads after the barrier that follows the
// histogram atomics; ends with a barrier.  counts / obase: the output buckets' counters and records (already offset to the
// slice this tile writes).
template <int T>
__device__ __forceinline__ void tile_offsets(int fan, uint32_t *s_hist, uint32_t *s_off, uint32_t *s_end, unsigned long long *s_base,
                                             uint2 **s_dst, uint32_t *s_chunk, uint32_t *s_nrec, unsigned long long *counts,
                                             uint2 *obase, int64_t part_cap, uint2 *const *peers = nullptr, int my_rank = 0) {
    const int lane = threadIdx.x & 31;
    for (int base = 0; base < fan; base += T) {
        const int i = base + threadIdx.x;
        const uint32_t h = i < fan ? s_hist[i] : 0;
        if (i < fan) s_base[i] = h ? atomicAdd(counts + i, (unsigned long long)h) : 0ull;
        uint32_t inc = h;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += y; }
        if (i < fan) s_off[i] = inc - h;
        if (lane == 31) s_chunk[i >> 5] = inc;            // chunks past `fan` hold 0
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        const int nchunk = (fan + 31) >> 5;
        uint32_t v = (int)threadIdx.x < nchunk ? s_chunk[threadIdx.x] : 0, inc = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += y; }
        s_chunk[threadIdx.x] = inc - v;
        if (threadIdx.x == 31) *s_nrec = inc;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < fan; i += T) {
        const uint32_t off = s_off[i] + s_chunk[i >> 5], h = s_hist[i];
        const int64_t b = (int64_t)s_base[i];
        int64_t room = part_cap - b;
        if (room < 0) room = 0;
        s_off[i] = off;
        s_end[i] = off + (room < (int64_t)h ? (uint32_t)room : h);
        s_dst[i] = (peers ? peers[i] + (int64_t)my_rank * part_cap : obase + (int64_t)i * part_cap) + (b - (int64_t)off);
    }
    __syncthreads();
}

// step 4: linear copy-out of the sorted staging, consecutive threads consecutive records of a run
template <int T>
__device__ __forceinline__ void tile_copy_out(uint32_t nrec, const uint64_t *s_sorted, const uint16_t *s_spid, const uint32_t *s_end,
                                              uint2 *const *s_dst, uint64_t pol) {
    for (uint32_t p0 = threadIdx.x; p0 < nrec; p0 += 4 * T) {
        uint64_t r[4]; uint32_t pid[4];
#pragma unroll
        for (int j = 0; j < 4; j++) if (p0 + j * T < nrec) { r[j] = s_sorted[p0 + j * T]; pid[j] = s_spid[p0 + j * T]; }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t p = p0 + j * T;
            if (p < nrec && p < s_end[pid[j]]) st_stream8_l2first(s_dst[pid[j]] + p, r[j], pol);
        }
    }
}

// ---- K2a-c ---------------------------------------------------------------------------------------------------------
struct CPartArgs {
    const uint64_t *pk2; const uint32_t *amb; int64_t n_words;
    const int64_t *seq_off; int64_t n_rec, g_begin, g_end; int k; uint64_t pow5km1;
    int64_t t_first, n_tiles;
    CBuckets out;
    uint64_t *sample_keys; uint64_t sample_mask; unsigned long long *sample_count;      // 1/256 key-space sample (partition.cu)
    const int64_t *d_counts; int64_t cap_records;                                       // device-side arguments (partition.cu)
};

__device__ __noinline__ void sample_key_c(uint64_t *sample_keys, uint64_t sample_mask, unsigned long long *sample_count, uint64_t key, uint64_t h) {
    uint64_t s = (h >> 16) & sample_mask;
    for (uint64_t probe = 0; probe <= sample_mask; probe++) {
        const uint64_t ck = sample_keys[s];
        if (ck == key) return;
        if (ck == PG_EMPTY) {
            const uint64_t old = atomicCAS(reinterpret_cast<unsigned long long *>(sample_keys + s), (unsigned long long)PG_EMPTY, (unsigned long long)key);
            if (old == PG_EMPTY) { atomicAdd(sample_count, 1ull); return; }
            if (old == key) return;
        }
        s = (s + 1) & sample_mask;
    }
    atomicAdd(sample_count, 1ull << 40);     // set full: poison the estimate so the host falls back to the upper bound
}

// KT: compile-time k (pg_interior_visit_ck: no rolling state, constant funnel shifts) or 0 = the k of the arguments.
// The records are derived twice - bucket + rank before the scan, the record itself after it - instead of held in 32
// registers across the barriers: with a compile-time k a window costs two funnel shifts, and the kernel is bound by the
// latency of its dependent chains at 24 warps per SM, not by its instruction count (holding the records measured 0.349 ms
// against 0.332 ms; ranks from ballots / MATCH.ANY + per-warp counters instead of the histogram atomic: 0.72 / 0.76 ms).
// PEER: the fused exchange - bucket = owner rank = LOW bits of the full mix (disjoint from the slot bits, which are the top
// ones), runs stored into the owners' receive buffers over NVLink.
template <int T, bool SAMPLE, int KT, int MINB, bool PEER>
__global__ void __launch_bounds__(T, MINB)
k2a_partition_c(CPartArgs a) {
    constexpr int TILE = T * KP_G;
    if (a.d_counts) {      // all records of the packed stream, bounds read from the device (as k2a_partition)
        const int64_t n_rec = a.d_counts[0];
        if (n_rec > a.cap_records) {          // the record index was truncated: poison the wide spill, the host falls back
            if (blockIdx.x == 0 && threadIdx.x == 0) *a.out.wide_count = 1ull << 62;
            return;
        }
        a.n_rec = n_rec;
        const int64_t s0 = n_rec > 0 ? a.seq_off[0] : 0, s1 = n_rec > 0 ? a.seq_off[n_rec] : 0;
        const int64_t lo = s0 + a.g_begin, hi = s0 + a.g_end;
        a.g_begin = lo < s1 ? lo : s1;
        a.g_end = (a.g_end < 0 || hi > s1) ? s1 : hi;
        a.n_words = ((s1 + 31) >> 5) + 4;
        a.t_first = a.g_begin / TILE;
        a.n_tiles = a.g_end > a.g_begin ? (a.g_end + TILE - 1) / TILE - a.t_first : 0;
    }
    extern __shared__ __align__(16) unsigned char smem[];
    const int fan = 1 << a.out.bits;
    uint64_t *s_sorted = reinterpret_cast<uint64_t *>(smem);                                    // TILE records
    unsigned long long *s_base = reinterpret_cast<unsigned long long *>(s_sorted + TILE);       // fan
    uint2 **s_dst = reinterpret_cast<uint2 **>(s_base + fan);                                   // fan
    uint32_t *s_hist = reinterpret_cast<uint32_t *>(s_dst + fan);                               // fan
    uint32_t *s_off = s_hist + fan, *s_end = s_off + fan;                                       // fan each
    uint16_t *s_spid = reinterpret_cast<uint16_t *>(s_end + fan);                               // TILE: bucket of a sorted position
    __shared__ uint32_t s_chunk[32];
    __shared__ uint32_t s_nrec;
    const uint64_t pol = pg_policy_evict_first();
    const int k = KT ? KT : a.k;
    const int shift = 64 - a.out.bits;

    for (int64_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        __syncthreads();                                  // the previous tile's copy-out is done with the staging and the tables
        for (int i = threadIdx.x; i < fan; i += T) s_hist[i] = 0;
        __syncthreads();
        // ---- 1. this thread's 16 positions.  Interior: bucket + rank of every compact record (the records themselves are
        // re-derived after the scan: two shifts each, cheaper than 32 registers held across the barriers); anything else
        // goes straight to the wide spill
        uint32_t pr[KP_G];                                // bucket | rank << 10
#pragma unroll
        for (int q = 0; q < KP_G; q++) pr[q] = C_NONE;
        const int64_t g0 = (a.t_first + tile) * TILE + (int64_t)threadIdx.x * KP_G;
        PgWindow w;
        const int j0 = (int)(g0 & 31);
        bool interior = false;
        if (g0 < a.g_end && g0 + KP_G > a.g_begin) {
            const int64_t wi = g0 >> 5;
            w.prv = wi > 0 ? __ldg(a.pk2 + wi - 1) : 0; w.cur = __ldg(a.pk2 + wi); w.nxt = wi + 1 < a.n_words ? __ldg(a.pk2 + wi + 1) : 0;
            w.aprv = wi > 0 ? __ldg(a.amb + wi - 1) : 0; w.acur = __ldg(a.amb + wi); w.anxt = wi + 1 < a.n_words ? __ldg(a.amb + wi + 1) : 0;
            int64_t r = find_record(a.seq_off, a.n_rec, g0);
            int64_t rs = r >= 0 ? __ldg(a.seq_off + r) : 0, re = __ldg(a.seq_off + r + 1);
            interior = pg_is_interior(w, g0, KP_G, k, rs, re, r >= 0, a.g_begin, a.g_end);
            if (interior) {
                auto rank = [&](int q, uint64_t F2, uint64_t R2, uint32_t) {
                    const uint64_t key = F2 < R2 ? F2 : R2;
                    uint64_t h;
                    if (SAMPLE || PEER) {
                        h = pg_mix64(key);
                        if (SAMPLE) { if (((h >> 8) & 0xFFu) == 0) sample_key_c(a.sample_keys, a.sample_mask, a.sample_count, key, h); }
                    } else {
                        h = pg_mix64_top(key);
                    }
                    const uint32_t pid = PEER ? (uint32_t)h & (uint32_t)(fan - 1) : (a.out.bits ? (uint32_t)(h >> shift) : 0u);
                    pr[q] = pid | (atomicAdd(&s_hist[pid], 1u) << 10);
                };
                if (KT) pg_interior_visit_ck<(KT ? KT : 27)>(w, j0, rank);
                else pg_interior_visit_c<KP_G>(w, j0, k, rank);
            } else {
                // generic path: record edges, ambiguity codes, range ends (all the quirks) -> wide records
                uint64_t F, R;
                pg_codes_init(w, j0, k, F, R);
#pragma unroll 1
                for (int q = 0; q < KP_G; q++) {
                    const int64_t g = g0 + q;
                    const int j = j0 + q;
                    bool ok = false;
                    if (g < a.g_end) {
                        while (r + 1 < a.n_rec && g >= re) { r++; rs = re; re = __ldg(a.seq_off + r + 1); }
                        ok = g >= a.g_begin && r >= 0 && g + k <= re;
                    }
                    if (ok) {
                        uint32_t vf, vr;
                        pg_occ_vals(w, j, g - rs, re - rs, k, vf, vr);
                        const PgUpdate u = pg_canonical_update_w(F, R, vf | (vr << 16));
                        if (PEER) wide_emit_owner(a.out.wide_peers, a.out.wide_count, a.out.wide_cap, a.out.my_rank,
                                                  (uint32_t)pg_hash_kind1(u.key, k) & (uint32_t)(fan - 1), u.key, u.masks, u.inc);
                        else wide_emit(a.out, u.key, u.masks, u.inc);
                    }
                    pg_codes_roll(w, j, k, a.pow5km1, F, R);
                }
            }
        }
        __syncthreads();
        // ---- 2. offsets in the tile, room in the output buckets
        tile_offsets<T>(fan, s_hist, s_off, s_end, s_base, s_dst, s_chunk, &s_nrec, a.out.counts, a.out.records, a.out.part_cap,
                        PEER ? a.out.peers : nullptr, a.out.my_rank);
        // ---- 3. every record to its sorted position
        if (interior) {
            uint32_t ovf = 0;       // records past their bucket's room (rare: hash skew) are handled after the loop, off the common path
            auto place = [&](int q, uint64_t F2, uint64_t R2, uint32_t ctx4) {
                const uint32_t pid = pr[q] & 1023u;
                const uint32_t p = s_off[pid] + (pr[q] >> 10);
                s_sorted[p] = pg_crec_pack(F2, R2, ctx4);
                s_spid[p] = (uint16_t)pid;
                if (p >= s_end[pid]) ovf |= 1u << q;
            };
            if (KT) pg_interior_visit_ck<(KT ? KT : 27)>(w, j0, place);
            else pg_interior_visit_c<KP_G>(w, j0, k, place);
            if (ovf) {
                auto spill = [&](int q, uint64_t F2, uint64_t R2, uint32_t ctx4) {
                    if (!(ovf & (1u << q))) return;
                    if (PEER) wide_emit_compact_owner(a.out.wide_peers, a.out.wide_count, a.out.wide_cap, a.out.my_rank, pr[q] & 1023u,
                                                      pg_crec_pack(F2, R2, ctx4), k);
                    else wide_emit_compact(a.out.wide, a.out.wide_count, a.out.wide_cap, pg_crec_pack(F2, R2, ctx4), k);
                };
                pg_interior_visit_c<KP_G>(w, j0, k, spill);
            }
        }
        __syncthreads();
        // ---- 4. linear copy-out
        tile_copy_out<T>(s_nrec, s_sorted, s_spid, s_end, s_dst, pol);
    }
}

// ---- K2c-c ---------------------------------------------------------------------------------------------------------
// sliced (the kernel's SLICED): segment s of `in` writes buckets [s << bits, ...) of `out` by hash bits [in.bits, in.bits + bits)
// (K2c-c); else every segment writes the same 2^bits buckets by the TOP bits (K2b-c: what arrived from the other ranks)
struct CSplitArgs { CBuckets in, out; int bits; int k; int64_t *stats; int sliced; };

constexpr int MSC_LOADS = 8;                 // 16-byte loads per thread = 16 records

template <int T, bool SLICED>
__global__ void __launch_bounds__(T, T == 256 ? 3 : (T == 512 ? 2 : 1))
k2c_multisplit_c(CSplitArgs a) {
    constexpr int TILE = T * MSC_LOADS * 2;
    extern __shared__ __align__(16) unsigned char smem[];
    const int fan = 1 << a.bits;
    const int n_seg = 1 << a.in.bits;
    uint64_t *s_sorted = reinterpret_cast<uint64_t *>(smem);                                    // TILE records
    unsigned long long *s_base = reinterpret_cast<unsigned long long *>(s_sorted + TILE);       // fan
    uint2 **s_dst = reinterpret_cast<uint2 **>(s_base + fan);                                   // fan
    uint32_t *s_tile0 = reinterpret_cast<uint32_t *>(s_dst + fan);                              // n_seg + 1: prefix of tiles per segment
    uint32_t *s_hist = s_tile0 + n_seg + 1;                                                     // fan
    uint32_t *s_off = s_hist + fan, *s_end = s_off + fan;                                       // fan each
    uint16_t *s_spid = reinterpret_cast<uint16_t *>(s_end + fan);                               // TILE
    __shared__ uint32_t s_chunk[32];
    __shared__ uint32_t s_nrec;
    const uint64_t pol = pg_policy_evict_first();
    const int lane = threadIdx.x & 31;

    auto seg_count = [&](int s) -> long long {      // a count above the capacity: the surplus went to the wide spill
        const long long c = (long long)a.in.counts[s];
        return c > a.in.part_cap ? a.in.part_cap : (c < 0 ? 0 : c);
    };
    for (int s = threadIdx.x; s < n_seg; s += T) s_tile0[s + 1] = (uint32_t)((seg_count(s) + TILE - 1) / TILE);
    if (threadIdx.x == 0) s_tile0[0] = 0;
    __syncthreads();
    if (threadIdx.x < 32) {
        uint32_t carry = 0;
        for (int base = 0; base < n_seg; base += 32) {
            const int i = base + threadIdx.x;
            uint32_t v = i < n_seg ? s_tile0[i + 1] : 0, inc = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += y; }
            if (i < n_seg) s_tile0[i + 1] = carry + inc;
            carry += __shfl_sync(0xffffffffu, inc, 31);
        }
    }
    __syncthreads();
    const uint32_t n_tiles = s_tile0[n_seg];
    // K2b-c into one bucket (a one-region table per rank: a.bits == 0) would shift by 64, which is undefined; the fan
    // mask of 0 sends every record to bucket 0 whatever the shift, so it is clamped to 63
    const int shift_ = 64 - (SLICED ? a.in.bits : 0) - a.bits;
    const int shift = shift_ < 64 ? shift_ : 63;

    int seg = 0;
    for (uint32_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        while (s_tile0[seg + 1] <= tile) seg++;       // a CTA's tiles only move forward through the segments
        const long long i0 = (long long)(tile - s_tile0[seg]) * TILE;
        const long long left = seg_count(seg) - i0;                      // records of this tile: min(left, TILE)
        const uint4 *src = reinterpret_cast<const uint4 *>(a.in.records + (int64_t)seg * a.in.part_cap + i0);    // part_cap and TILE are even
        __syncthreads();
        for (int i = threadIdx.x; i < fan; i += T) s_hist[i] = 0;
        __syncthreads();
        // ---- 1. load (two records per 16-byte load), bucket, rank
        uint4 v[MSC_LOADS];
        uint32_t pr[2 * MSC_LOADS];
#pragma unroll
        for (int q = 0; q < MSC_LOADS; q++) {
            const int slot = q * T + threadIdx.x;
            if (2 * slot < left) v[q] = pg_ld_stream_l2first(src + slot, pol);
        }
#pragma unroll
        for (int q = 0; q < MSC_LOADS; q++) {
            const int slot = q * T + threadIdx.x;
#pragma unroll
            for (int h = 0; h < 2; h++) {
                pr[2 * q + h] = C_NONE;
                if (2 * slot + h < left) {
                    const uint64_t rc = h ? ((uint64_t)v[q].z | ((uint64_t)v[q].w << 32)) : ((uint64_t)v[q].x | ((uint64_t)v[q].y << 32));
                    const uint32_t pid = (uint32_t)(pg_mix64_top(rc & PG_C_KEYMASK) >> shift) & (uint32_t)(fan - 1);
                    pr[2 * q + h] = pid | (atomicAdd(&s_hist[pid], 1u) << 10);
                }
            }
        }
        __syncthreads();
        // ---- 2. offsets in the tile, room in this segment's slice of the output buckets
        const int64_t slice = SLICED ? ((int64_t)seg << a.bits) : 0;
        tile_offsets<T>(fan, s_hist, s_off, s_end, s_base, s_dst, s_chunk, &s_nrec, a.out.counts + slice,
                        a.out.records + slice * a.out.part_cap, a.out.part_cap);
        // ---- 3. every record to its sorted position (one past its bucket's room: remembered, handled off the common path)
        uint32_t ovf = 0;
#pragma unroll
        for (int q = 0; q < MSC_LOADS; q++) {
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const uint32_t x = pr[2 * q + h];
                if (x == C_NONE) continue;
                const uint32_t pid = x & 1023u;
                const uint32_t p = s_off[pid] + (x >> 10);
                reinterpret_cast<uint2 *>(s_sorted)[p] = h ? make_uint2(v[q].z, v[q].w) : make_uint2(v[q].x, v[q].y);
                s_spid[p] = (uint16_t)pid;
                if (p >= s_end[pid]) ovf |= 1u << (2 * q + h);
            }
        }
        if (ovf) {
#pragma unroll
            for (int q = 0; q < MSC_LOADS; q++) {
#pragma unroll
                for (int h = 0; h < 2; h++)
                    if (ovf & (1u << (2 * q + h)))
                        wide_emit_compact(a.out.wide, a.out.wide_count, a.out.wide_cap,
                                          h ? ((uint64_t)v[q].z | ((uint64_t)v[q].w << 32)) : ((uint64_t)v[q].x | ((uint64_t)v[q].y << 32)), a.k);
            }
        }
        __syncthreads();
        // ---- 4. linear copy-out
        tile_copy_out<T>(s_nrec, s_sorted, s_spid, s_end, s_dst, pol);
    }
}

template <int T>
int launch_split_c(const CSplitArgs &a, cudaStream_t st) {
    const int fan = 1 << a.bits, n_seg = 1 << a.in.bits;
    const int tile = T * MSC_LOADS * 2;
    const int smem = tile * 8 + fan * 16 + (n_seg + 1) * 4 + 3 * fan * 4 + tile * 2 + 16;
    const int64_t max_tiles = (int64_t)n_seg * ((a.in.part_cap + tile - 1) / tile);
    int per_sm = 227 * 1024 / (smem + 1024 + 256);
    const int cap_sm = T == 256 ? 3 : (T == 512 ? 2 : 1);
    if (per_sm > cap_sm) per_sm = cap_sm;
    if (per_sm < 1) return pg_fail(PG_ERR_INVALID, "pg_records_resplit_c: %d bytes of shared memory do not fit an SM", smem);
    const int64_t maxg = (int64_t)pg_num_sms() * per_sm;
    int grid = (int)(max_tiles < maxg ? max_tiles : maxg);
    if (grid < 1) grid = 1;
    if (a.sliced) {
        PG_CUDA(cudaFuncSetAttribute(k2c_multisplit_c<T, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        k2c_multisplit_c<T, true><<<grid, T, smem, st>>>(a);
    } else {
        PG_CUDA(cudaFuncSetAttribute(k2c_multisplit_c<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        k2c_multisplit_c<T, false><<<grid, T, smem, st>>>(a);
    }
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}

// ---- K3s-c ---------------------------------------------------------------------------------------------------------
struct CRegionArgs { TableView t; CBuckets b; int n_regions; };

__device__ __forceinline__ uint4 lds128c(const void *p) {      // re-issued every time: the slots change under the other threads' atomics
    uint4 r;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "r"((uint32_t)__cvta_generic_to_shared(p)) : "memory");
    return r;
}

// Same probe scheme as k3s_region_build (region_build.cu): groups of four slots per step, match / free masks from bit
// tricks, one CAS site.  Differences: records are 8 bytes, the shared-memory key is the 2-bit code (or PG_WIDE_FLAG | base-5
// key for a key that has no 2-bit form, met only when a later round reloads a region the wide spill wrote into), the value
// word comes from the 16-entry table, and the write-out converts to the base-5 key the table holds in HBM.
// Between the rounds of a multi-round build the table holds ACGT-only keys in their 2-bit form under PG_C_HBM_FLAG (bit 63;
// base-5 codes stay below 2^63): a later round then reloads a region without converting 2^RB keys back (27 divisions by 5
// each - on BASELINE config 4 at 2 GPUs that doubled K3s-c), and only the LAST round writes the base-5 keys the
// reference's table holds.  The wide upserts between rounds follow the same convention (k3s_wide_insert, compact_mode).
#define PG_C_HBM_FLAG 0x8000000000000000ull
// FP: probe on 16-bit FINGERPRINTS.  The kernel is bound by shared-memory wavefronts, almost half of them the two 16-byte
// loads (four 8-byte keys) of a probe step, which random addresses stretch to ~10 wavefronts each.  With FP a probe step
// loads the group's four 16-bit tags (one 8-byte load), compares them in SWAR form and reads a key (8 bytes) only where a
// tag matches; tag 0 = free.  The 64-bit CAS on the key stays the one source of truth: a claim writes the key first and the
// tag after it, so a reader can meet a slot whose tag is still 0 although its key is set - its CAS then fails and tells
// it the key (its own: found; another: that slot is taken, on to the next free one).
__device__ __forceinline__ uint32_t haszero16(uint32_t x) { return (x - 0x00010001u) & ~x & 0x80008000u; }
__device__ __forceinline__ uint2 lds64c(const void *p) {
    uint2 r;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "r"((uint32_t)__cvta_generic_to_shared(p)) : "memory");
    return r;
}
template <bool FIRST, bool LAST, int THREADS, int RPT, bool FP>
__global__ void __launch_bounds__(THREADS, THREADS == 1024 ? 2 : 3)
k3s_region_build_c(CRegionArgs a) {
    constexpr int NS = 1 << 12;
    constexpr uint32_t CNT_MAX = (1u << 22) - 1u;
    extern __shared__ __align__(16) unsigned char smem[];
    uint64_t *s_key = reinterpret_cast<uint64_t *>(smem);
    uint32_t *s_mask = reinterpret_cast<uint32_t *>(s_key + NS);
    uint32_t *s_cnt = s_mask + NS;
    uint16_t *s_fp = reinterpret_cast<uint16_t *>(s_cnt + NS);          // FP only: NS tags
    const int tag_shift = a.t.shift - 16;                               // the 16 hash bits below the slot index
    __shared__ uint16_t s_lut5[PG_LUT5_SIZE];
    __shared__ uint32_t s_vlut[16];
    const TableView &t = a.t;
    uint4 *const slots = reinterpret_cast<uint4 *>(t.slots);
    uint32_t n_claimed = 0;
    for (int i = threadIdx.x; i < PG_LUT5_SIZE; i += THREADS) s_lut5[i] = (uint16_t)pg_lut5_entry(i);
    if (threadIdx.x < 16) s_vlut[threadIdx.x] = pg_vlut_entry(threadIdx.x);

    auto init_slot = [&](int64_t r, int s) {
        uint64_t key = PG_EMPTY; uint32_t m = 0, c = 0;
        if (!FIRST) {
            const uint4 g = slots[r * NS + s];
            const uint64_t hi = (uint64_t)g.z | ((uint64_t)g.w << 32);
            if ((hi & ~PG_VAL_MASK) == t.tag) {
                // what an earlier round left: a 2-bit key under PG_C_HBM_FLAG, or the base-5 key of a k-mer with an
                // ambiguity digit (it has no 2-bit form: PG_WIDE_FLAG in shared memory)
                const uint64_t kh = (uint64_t)g.x | ((uint64_t)g.y << 32);
                key = (kh & PG_C_HBM_FLAG) ? (kh & ~PG_C_HBM_FLAG) : (kh | PG_WIDE_FLAG);
                m = g.z; c = g.w & CNT_MAX;
            }
        }
        s_key[s] = key; s_mask[s] = m; s_cnt[s] = c;
        if (FP) {       // a key without a 2-bit form never equals a compact record's: any non-zero tag will do
            uint32_t tg = 0;
            if (!FIRST && key != PG_EMPTY) tg = (key & PG_WIDE_FLAG) ? 1u : (((uint32_t)(pg_mix64_top(key) >> tag_shift) & 0xFFFFu) | 1u);
            s_fp[s] = (uint16_t)tg;
        }
    };

    int64_t r = blockIdx.x;
    if (r < a.n_regions)
        for (int s = threadIdx.x; s < NS; s += THREADS) init_slot(r, s);
    __syncthreads();
    for (; r < a.n_regions; r += gridDim.x) {
        unsigned long long c64 = a.b.counts[r];
        if (c64 > (unsigned long long)a.b.part_cap) c64 = (unsigned long long)a.b.part_cap;     // the surplus sits in the wide spill
        const uint32_t c = (uint32_t)c64;
        const uint2 *src = a.b.records + r * a.b.part_cap;
        for (uint32_t base = 0; base < c; base += RPT * THREADS) {
            uint2 rec[RPT];
#pragma unroll
            for (int j = 0; j < RPT; j++) {
                const uint32_t i = base + j * THREADS + threadIdx.x;
                if (i < c) rec[j] = ld_stream8(src + i);
            }
#pragma unroll
            for (int j = 0; j < RPT; j++) {
                const bool act = base + j * THREADS + threadIdx.x < c;
                const uint32_t klo = rec[j].x, khi = rec[j].y & (uint32_t)(PG_C_KEYMASK >> 32);
                const uint32_t ctx = rec[j].y >> (PG_C_KEYBITS - 32);
                const uint64_t key = (uint64_t)klo | ((uint64_t)khi << 32);
                const uint64_t h = pg_mix64_top(key);
                uint32_t g = (uint32_t)(h >> t.shift) & (NS - 1) & ~(uint32_t)(PG_REGION_GROUP - 1);
                int s = -1;
                if (act && FP) {
                    const uint32_t tag = ((uint32_t)(h >> tag_shift) & 0xFFFFu) | 1u, tt = tag * 0x00010001u;
                    for (int probe = 0; probe < NS / PG_REGION_GROUP;) {
                        const uint2 tg = lds64c(s_fp + g);
                        // tags equal to mine (bit 15 / 31 of a word per slot; a flag above a true one may be spurious - every
                        // candidate is confirmed on its key)
                        uint32_t cm = (haszero16(tg.x ^ tt) >> 15 & 0x10001u) | ((haszero16(tg.y ^ tt) >> 15 & 0x10001u) << 2);
                        cm = (cm & 0xFu) | (cm >> 15 & 0xAu);              // slots 0..3 -> bits 0..3
                        bool found = false;
                        while (cm) {
                            const int j = __ffs(cm) - 1; cm &= cm - 1;
                            const uint2 kk = lds64c(s_key + g + j);
                            if (kk.x == klo && kk.y == khi) { s = (int)g + j; found = true; break; }
                        }
                        if (found) break;
                        uint32_t em = (haszero16(tg.x) >> 15 & 0x10001u) | ((haszero16(tg.y) >> 15 & 0x10001u) << 2);
                        em = (em & 0xFu) | (em >> 15 & 0xAu);              // the LOWEST flagged slot is always a true zero
                        // free slots of the group in ascending order.  A failed CAS says which key holds the slot: mine (found)
                        // or another one, whose tag is simply not out yet - skip it.  No re-reading, so no lane ever waits
                        // for another lane's tag store (two lanes of ONE warp racing for a slot would otherwise spin on each other).
                        while (em) {
                            const int e = (int)g + __ffs(em) - 1; em &= em - 1;
                            const unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long *>(s_key + e), (unsigned long long)PG_EMPTY,
                                                                     (unsigned long long)key);
                            if (old == PG_EMPTY) { *reinterpret_cast<volatile uint16_t *>(s_fp + e) = (uint16_t)tag; n_claimed++; s = e; found = true; break; }
                            if (old == key) { s = e; found = true; break; }
                        }
                        if (found) break;
                        g = (g + PG_REGION_GROUP) & (NS - 1); probe++;
                    }
                    if (s < 0) atomicExch(reinterpret_cast<unsigned long long *>(t.stats + PG_STAT_OVERFLOW), 1ull);
                }
                if (act && !FP) {
                    for (int probe = 0; probe < NS / PG_REGION_GROUP;) {
                        const uint4 a4 = lds128c(s_key + g), b4 = lds128c(s_key + g + 2);
                        const uint32_t mm = (uint32_t)(a4.x == klo && a4.y == khi) | ((uint32_t)(a4.z == klo && a4.w == khi) << 1) |
                                            ((uint32_t)(b4.x == klo && b4.y == khi) << 2) | ((uint32_t)(b4.z == klo && b4.w == khi) << 3);
                        if (mm) { s = (int)g + __ffs(mm) - 1; break; }
                        // free slots hold PG_EMPTY; a 2-bit code's high word is < 2^22 and PG_WIDE_FLAG | base-5 key < 2^63 + 5^27
                        const uint32_t em = (uint32_t)(a4.y == 0xFFFFFFFFu) | ((uint32_t)(a4.w == 0xFFFFFFFFu) << 1) |
                                            ((uint32_t)(b4.y == 0xFFFFFFFFu) << 2) | ((uint32_t)(b4.w == 0xFFFFFFFFu) << 3);
                        if (em) {
                            const int e = (int)g + __ffs(em) - 1;
                            const unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long *>(s_key + e), (unsigned long long)PG_EMPTY,
                                                                     (unsigned long long)key);
                            if (old == PG_EMPTY) { n_claimed++; s = e; break; }
                            if (old == key) { s = e; break; }
                            continue;             // another key took that slot first: look at the group again
                        }
                        g = (g + PG_REGION_GROUP) & (NS - 1); probe++;
                    }
                    if (s < 0)                // the region is full: the table is too small for this input
                        atomicExch(reinterpret_cast<unsigned long long *>(t.stats + PG_STAT_OVERFLOW), 1ull);
                }
                __syncwarp();
                if (s >= 0) {
                    uint32_t masks, inc;
                    pg_crec_vals(ctx, s_vlut[ctx & 15u], masks, inc);
                    atomicOr(s_mask + s, masks);
                    atomicAdd(s_cnt + s, inc);
                }
            }
        }
        __syncthreads();
        // ---- write the region out with base-5 keys (one 16-byte store per slot) and start the next one
        const int64_t nxt = r + gridDim.x;
        for (int s = threadIdx.x; s < NS; s += THREADS) {
            const uint64_t key = s_key[s];
            uint4 g = make_uint4(0u, 0u, 0u, 0u);
            if (key != PG_EMPTY) {
                const uint64_t key5 = (key & PG_WIDE_FLAG) ? (key & ~PG_WIDE_FLAG) : (LAST ? pg_code5_of2(key, s_lut5) : (key | PG_C_HBM_FLAG));
                const uint32_t cnt = s_cnt[s];
                g = make_uint4((uint32_t)key5, (uint32_t)(key5 >> 32), s_mask[s], (cnt < CNT_MAX ? cnt : CNT_MAX) | (uint32_t)(t.tag >> 32));
            }
            slots[r * NS + s] = g;
            if (nxt < a.n_regions) init_slot(nxt, s);
        }
        __syncthreads();
    }
    publish_claims(t, n_claimed);
}

// the wide spill: upserts with L2 atomics, probing confined to the regions (the same kernel region_build.cu runs on its spill)
__global__ void __launch_bounds__(256)
k3s_wide_insert(TableView t, const uint4 *__restrict__ wide, const unsigned long long *__restrict__ count, int64_t cap, int compact_mode) {
    unsigned long long c = *count;
    if (c > (unsigned long long)cap) {
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicExch(reinterpret_cast<unsigned long long *>(t.stats + PG_STAT_LOST), 1ull);
        c = (unsigned long long)cap;
    }
    uint32_t n_claimed = 0;
    for (unsigned long long i = blockIdx.x * 256ull + threadIdx.x; i < c; i += gridDim.x * 256ull) {
        const uint4 r = pg_ld_stream(wide + i);
        const uint64_t key5 = (uint64_t)r.x | ((uint64_t)r.y << 32);
        uint64_t x2;
        const bool pure = pg_code2_of5(key5, t.k, x2);
        // compact_mode: more rounds follow, ACGT-only keys live in the table in their flagged 2-bit form
        const uint64_t key = (compact_mode && pure) ? (x2 | PG_C_HBM_FLAG) : key5;
        const uint64_t h = pure ? pg_mix64(x2) : pg_mix64(~key5);           // == pg_hash_kind1(key5)
        const uint64_t s = (h >> t.shift) & t.hmask;
        uint64_t lo, hi;
        pg_ld_slot_raw(t.slots + 2 * s, lo, hi);
        table_upsert_from(t, s, lo, hi, key, r.z, r.w, n_claimed);
    }
    publish_claims(t, n_claimed);
}

int make_cbuckets(const pg_cbuckets *b, const char *who, CBuckets &o) {
    const bool peer = b && b->d_peer_bases != nullptr;
    if (!b || !b->d_counts || !b->d_wide_count || b->part_cap < 2 || (b->part_cap & 1) || b->wide_cap < 1 || b->bits < 0)
        return pg_fail(PG_ERR_INVALID, "%s: bad compact bucket set (even part_cap, wide_cap >= 1)", who);
    if (peer) {
        if (b->d_records || b->d_wide || !b->d_wide_peer_bases || b->bits > 6 || b->my_rank < 0 || b->my_rank >= (1 << b->bits))
            return pg_fail(PG_ERR_INVALID, "%s: a peer bucket set has d_peer_bases AND d_wide_peer_bases, no local buffers, bits = log2(ranks) <= 6", who);
    } else if (!b->d_records || !b->d_wide || ((reinterpret_cast<uintptr_t>(b->d_records) | reinterpret_cast<uintptr_t>(b->d_wide)) & 15)) {
        return pg_fail(PG_ERR_INVALID, "%s: bad compact bucket set (16-byte aligned buffers)", who);
    }
    o.records = reinterpret_cast<uint2 *>(b->d_records); o.counts = reinterpret_cast<unsigned long long *>(b->d_counts);
    o.part_cap = b->part_cap; o.bits = b->bits;
    o.wide = reinterpret_cast<uint4 *>(b->d_wide); o.wide_count = reinterpret_cast<unsigned long long *>(b->d_wide_count); o.wide_cap = b->wide_cap;
    o.peers = reinterpret_cast<uint2 *const *>(b->d_peer_bases); o.wide_peers = reinterpret_cast<uint4 *const *>(b->d_wide_peer_bases);
    o.my_rank = b->my_rank;
    return PG_OK;
}

int k2a_c_smem(int fan, int threads) { const int tile = threads * KP_G; return tile * 8 + fan * 16 + 3 * fan * 4 + tile * 2 + 16; }

}  // namespace

extern "C" int pg_kmer_partition_c(const pg_table *t, const uint32_t *d_pk2, const uint32_t *d_amb, const int64_t *d_seq_off,
                                   int64_t n_rec, int64_t g_begin, int64_t g_end, const int64_t *d_counts, int64_t cap_records,
                                   int64_t max_bases, const pg_cbuckets *out, uint64_t *d_sample_keys, int64_t sample_cap,
                                   int64_t *d_sample_count, pg_stream_t stream_) {
    if (!t || t->k < 1 || t->k > 27 || t->mode != PG_MODE_CANONICAL)
        return pg_fail(PG_ERR_INVALID, "pg_kmer_partition_c: bad table descriptor (k 1..27, PG_MODE_CANONICAL; only mode and k are used)");
    if (!d_pk2 || !d_amb || !d_seq_off || n_rec < 0 || g_begin < 0 || (!d_counts && g_end < g_begin) || (d_counts && (cap_records < 0 || max_bases < 0)))
        return pg_fail(PG_ERR_INVALID, "pg_kmer_partition_c: bad arguments");
    CPartArgs a;
    int rc = make_cbuckets(out, "pg_kmer_partition_c", a.out); if (rc) return rc;
    if (out->bits > 10) return pg_fail(PG_ERR_INVALID, "pg_kmer_partition_c: at most 2^10 buckets");
    cudaStream_t st = (cudaStream_t)stream_;
    const int fan = 1 << out->bits;
    const bool peer = a.out.peers != nullptr;
    PG_CUDA(cudaMemsetAsync(out->d_counts, 0, (size_t)fan * 8, st));
    PG_CUDA(cudaMemsetAsync(out->d_wide_count, 0, (size_t)(peer ? fan : 1) * 8, st));
    int64_t span = g_end - g_begin;                                     // grid sizing only in device-argument mode
    if (d_counts) { n_rec = 1; span = (g_end < 0 || g_end - g_begin > max_bases) ? max_bases - (g_begin < max_bases ? g_begin : max_bases) : g_end - g_begin; }
    if (n_rec == 0 || span <= 0) return PG_OK;
    a.pk2 = reinterpret_cast<const uint64_t *>(d_pk2); a.amb = d_amb; a.n_words = ((g_end + 31) >> 5) + 4;
    a.seq_off = d_seq_off; a.n_rec = n_rec; a.g_begin = g_begin; a.g_end = g_end; a.k = t->k; a.pow5km1 = pg_pow5(t->k - 1);
    const int T = peer ? 512 : 256;       // across GPUs 8192-position tiles: twice the run length per owner on NVLink
    const int tile = T * KP_G;
    a.t_first = g_begin / tile; a.n_tiles = (g_begin + span + tile - 1) / tile - a.t_first;
    a.d_counts = d_counts; a.cap_records = cap_records;
    a.sample_keys = nullptr; a.sample_mask = 0; a.sample_count = nullptr;
    if (d_sample_keys) {
        if (peer) return pg_fail(PG_ERR_INVALID, "pg_kmer_partition_c: no key sampling on the fused exchange");
        if (!d_sample_count || sample_cap < 2 || (sample_cap & (sample_cap - 1)))
            return pg_fail(PG_ERR_INVALID, "pg_kmer_partition_c: sample set needs a power-of-two capacity and a counter");
        a.sample_keys = d_sample_keys; a.sample_mask = (uint64_t)sample_cap - 1;
        a.sample_count = reinterpret_cast<unsigned long long *>(d_sample_count);
    }
    const int smem = k2a_c_smem(fan, T);
    static int per_sm_env = -1;
    if (per_sm_env < 0) { const char *e = getenv("PG_K2AC_CTAS"); per_sm_env = e ? atoi(e) : 0; }
    // 3 CTAs (80 registers) per SM measured 0.278 ms on config 2, 4 CTAs (64 registers, PG_K2AC_CTAS=4) 0.291 ms
    int per_sm = ctas_per_sm(smem, 512);
    const int want = per_sm_env > 0 ? per_sm_env : (peer ? 2 : 3);
    if (per_sm > want) per_sm = want;
    if (per_sm > 4) per_sm = 4;
    const int64_t maxg = (int64_t)pg_num_sms() * per_sm;
    int grid = (int)(a.n_tiles < maxg ? a.n_tiles : maxg);
    if (grid < 1) grid = 1;
#define K2AC_LAUNCH(TT, S, KT, MB, P)                                                                                       \
    do {                                                                                                                    \
        PG_CUDA(cudaFuncSetAttribute(k2a_partition_c<TT, S, KT, MB, P>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
        k2a_partition_c<TT, S, KT, MB, P><<<grid, TT, smem, st>>>(a);                                                       \
    } while (0)
    static int kt_env = -1;
    if (kt_env < 0) { const char *e = getenv("PG_K2AC_GENERIC"); kt_env = e ? atoi(e) : 0; }      // 1: always the runtime-k kernel
    const int kt = kt_env ? 0 : t->k;
    if (peer) {
        if (kt == 27) K2AC_LAUNCH(512, false, 27, 2, true); else if (kt == 21) K2AC_LAUNCH(512, false, 21, 2, true); else K2AC_LAUNCH(512, false, 0, 2, true);
    } else if (a.sample_keys) {
        if (kt == 27) K2AC_LAUNCH(256, true, 27, 3, false); else if (kt == 21) K2AC_LAUNCH(256, true, 21, 3, false); else K2AC_LAUNCH(256, true, 0, 3, false);
    } else if (per_sm >= 4) {
        if (kt == 27) K2AC_LAUNCH(256, false, 27, 4, false); else if (kt == 21) K2AC_LAUNCH(256, false, 21, 4, false); else K2AC_LAUNCH(256, false, 0, 3, false);
    } else {
        if (kt == 27) K2AC_LAUNCH(256, false, 27, 3, false); else if (kt == 21) K2AC_LAUNCH(256, false, 21, 3, false); else K2AC_LAUNCH(256, false, 0, 3, false);
    }
#undef K2AC_LAUNCH
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}

extern "C" int pg_records_resplit_c(const pg_cbuckets *in, int bits, const pg_cbuckets *out, int k, int64_t *d_table_stats, pg_stream_t stream_) {
    CSplitArgs a;
    int rc = make_cbuckets(in, "pg_records_resplit_c", a.in); if (rc) return rc;
    rc = make_cbuckets(out, "pg_records_resplit_c", a.out); if (rc) return rc;
    if (bits < 1 || bits > 10 || in->bits > 13 || out->bits != in->bits + bits || k < 1 || k > 27 || in->d_records == out->d_records)
        return pg_fail(PG_ERR_INVALID, "pg_records_resplit_c: bad geometry (bits 1..10, in->bits <= 13, out->bits == in->bits + bits, distinct buffers)");
    cudaStream_t st = (cudaStream_t)stream_;
    PG_CUDA(cudaMemsetAsync(out->d_counts, 0, (size_t)(1ll << out->bits) * 8, st));
    a.bits = bits; a.k = k; a.stats = d_table_stats; a.sliced = 1;
    static int thr_env = -1;
    if (thr_env < 0) { const char *e = getenv("PG_SPLITC_THREADS"); thr_env = e ? atoi(e) : 0; }
    const int fan = 1 << bits;
    int threads = fan <= 64 ? 256 : (fan <= 256 ? 512 : 1024);
    if (thr_env == 256 || thr_env == 512 || thr_env == 1024) threads = thr_env;
    if (threads == 256) return launch_split_c<256>(a, st);
    if (threads == 512) return launch_split_c<512>(a, st);
    return launch_split_c<1024>(a, st);
}

// K2b-c: what arrived from the other ranks - the 2^in->bits segments of `in`, one per source rank, each of in->part_cap
// records - into the 2^out->bits hash-prefix buckets of `out` (TOP bits of the mix)
extern "C" int pg_records_split_c(const pg_cbuckets *in, const pg_cbuckets *out, int k, int64_t *d_table_stats, pg_stream_t stream_) {
    CSplitArgs a;
    int rc = make_cbuckets(in, "pg_records_split_c", a.in); if (rc) return rc;
    rc = make_cbuckets(out, "pg_records_split_c", a.out); if (rc) return rc;
    if (a.in.peers || a.out.peers || in->bits > 6 || out->bits < 0 || out->bits > 10 || k < 1 || k > 27 || in->d_records == out->d_records)
        return pg_fail(PG_ERR_INVALID, "pg_records_split_c: bad geometry (local sets, <= 64 segments, 1..1024 buckets, distinct buffers)");
    cudaStream_t st = (cudaStream_t)stream_;
    PG_CUDA(cudaMemsetAsync(out->d_counts, 0, (size_t)(1ll << out->bits) * 8, st));
    a.bits = out->bits; a.k = k; a.stats = d_table_stats; a.sliced = 0;
    const int fan = 1 << a.bits;
    if (fan <= 64) return launch_split_c<256>(a, st);
    if (fan <= 256) return launch_split_c<512>(a, st);
    return launch_split_c<1024>(a, st);
}

// upsert one segment of wide records (what another rank's K2a-c sent for the keys this rank owns) with L2 atomics
extern "C" int pg_wide_insert(const pg_table *t, const uint64_t *d_wide, const int64_t *d_count, int64_t cap, int last_round, pg_stream_t stream_) {
    if (!t || !t->d_slots || !t->d_stats || t->capacity < 2 || (t->capacity & (t->capacity - 1)) || t->epoch < 1 || t->epoch > PG_EPOCH_MAX)
        return pg_fail(PG_ERR_INVALID, "pg_wide_insert: bad table");
    if (!d_wide || !d_count || cap < 1 || (reinterpret_cast<uintptr_t>(d_wide) & 15) || t->hash_kind != 1)
        return pg_fail(PG_ERR_INVALID, "pg_wide_insert: bad arguments (hash_kind 1 table, 16-byte aligned records)");
    k3s_wide_insert<<<pg_num_sms(), 256, 0, (cudaStream_t)stream_>>>(make_view(t), reinterpret_cast<const uint4 *>(d_wide),
                                                                     reinterpret_cast<const unsigned long long *>(d_count), cap, last_round ? 0 : 1);
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}

extern "C" int pg_region_build_c(const pg_table *t, const pg_cbuckets *b, int first_round, int last_round, pg_stream_t stream_) {
    if (!t || !t->d_slots || !t->d_stats || t->capacity < 2 || (t->capacity & (t->capacity - 1)) || t->epoch < 1 || t->epoch > PG_EPOCH_MAX)
        return pg_fail(PG_ERR_INVALID, "pg_region_build_c: bad table");
    if (t->region_bits != 12 || t->hash_kind != 1 || t->mode != PG_MODE_CANONICAL)
        return pg_fail(PG_ERR_INVALID, "pg_region_build_c: needs pg_table.region_bits 12, hash_kind 1 and PG_MODE_CANONICAL");
    int bits = 0; while ((1ll << bits) < t->capacity) bits++;
    CRegionArgs ra;
    int rc = make_cbuckets(b, "pg_region_build_c", ra.b); if (rc) return rc;
    if (bits < 12 || b->bits != bits - 12 || b->part_cap > 0x7FFFFFFF)
        return pg_fail(PG_ERR_INVALID, "pg_region_build_c: the bucket set must hold one bucket per 4096-slot region (bits %d, table 2^%d slots)", b->bits, bits);
    cudaStream_t st = (cudaStream_t)stream_;
    ra.t = make_view(t); ra.n_regions = 1 << b->bits;
    constexpr int smem = (1 << 12) * 16;
    static int cfg = -1;
    if (cfg < 0) { const char *e = getenv("PG_K3SC_CFG"); cfg = e ? atoi(e) : 0; }
    static int fp = -1;
    if (fp < 0) { const char *e = getenv("PG_K3SC_FP"); fp = e ? atoi(e) : 0; }      // measured 0.502 ms against 0.480 ms: off
#define K3SC_LAUNCH3(F, LA, T, R, PER, FPV)                                                                                 \
    do {                                                                                                                    \
        const int smem_ = smem + ((FPV) ? (1 << 12) * 2 : 0);                                                               \
        const int64_t maxg = (int64_t)pg_num_sms() * (PER);                                                                 \
        const int grid = (int)(ra.n_regions < maxg ? ra.n_regions : maxg);                                                  \
        PG_CUDA(cudaFuncSetAttribute(k3s_region_build_c<F, LA, T, R, FPV>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_)); \
        k3s_region_build_c<F, LA, T, R, FPV><<<grid, T, smem_, st>>>(ra);                                                   \
    } while (0)
#define K3SC_LAUNCH2(F, LA, T, R, PER) do { if (fp) K3SC_LAUNCH3(F, LA, T, R, PER, true); else K3SC_LAUNCH3(F, LA, T, R, PER, false); } while (0)
#define K3SC_LAUNCH(T, R, PER)                                                                                              \
    do {                                                                                                                    \
        if (first_round) { if (last_round) K3SC_LAUNCH2(true, true, T, R, PER); else K3SC_LAUNCH2(true, false, T, R, PER); } \
        else { if (last_round) K3SC_LAUNCH2(false, true, T, R, PER); else K3SC_LAUNCH2(false, false, T, R, PER); }          \
    } while (0)
    if (cfg == 2) K3SC_LAUNCH(1024, 2, 2);
    else K3SC_LAUNCH(512, 4, 3);
#undef K3SC_LAUNCH3
#undef K3SC_LAUNCH2
#undef K3SC_LAUNCH
    PG_CUDA(cudaGetLastError());
    k3s_wide_insert<<<pg_num_sms(), 256, 0, st>>>(ra.t, ra.b.wide, ra.b.wide_count, ra.b.wide_cap, last_round ? 0 : 1);
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}
