// npz_dump.cu - the `_db.npz` image on the GPU: oakht slot placement and the chunked DEFLATE of its members (sm_100a).
//
// Placement.  The reference's `oakht.pointer()` (kmer_numba.py:521-538) probes j0, j0, j0+1, j0+4, ... (mod cap) from
// j0 = signed FNV-1a of the low 4 key bytes, floor-modulo cap, and stops at the first slot whose count is 0 or whose key
// matches.  The slots are filled in rounds: in round s every unplaced entry bids for its s-th probe slot if no earlier
// round took it (atomicMin of the key into `okeys`, which starts all-ones), the smallest key wins, the losers move on.
// A taken slot is never vacated, so every probe slot before a key's own is occupied and pointer() finds it; the image
// depends only on the set of entries.  The short-record sentinel 2^64-1 equals the all-ones bid marker: it takes its
// first probe slot before the bidding starts.  Taken slots are marked by a count >= 1 (`ocnts`); the unclaimed ones get
// key 0 back at the end, as the host writes them.  Round 1 probes j0 again, which round 0 took: it is skipped.
//
// Compression.  One CTA encodes one chunk of a member (deflate.cuh) from shared memory into a worst-case-sized staging
// slot; a one-CTA scan turns the slab's chunk sizes into offsets and chains the chunk CRC-32s (pg_crc_combine); a copy
// kernel compacts the slots.  The caller walks the member in slabs and overlaps the D2H copy and the file write.
#include "common.cuh"
#include "deflate.cuh"

#define PG_DEF_THREADS 256
#define PG_OAK_MAX_ROUNDS 4096
#define PG_OAK_BATCH 8            // rounds enqueued between two reads of the remaining count

namespace {

__device__ __forceinline__ int64_t oak_slot0(uint64_t key, int64_t cap) {
    uint64_t a = 0xcbf29ce484222325ull, v = key;
    for (int i = 0; i < 4; i++) { a ^= (v & 0xff); a *= 0x100000001b3ull; v >>= 8; }
    int64_t j = (int64_t)a % cap;
    return j < 0 ? j + cap : j;
}
// the s-th probe slot of pointer() for s != 1
__device__ __forceinline__ int64_t oak_probe(uint64_t key, int64_t cap, int64_t s) {
    const int64_t j0 = oak_slot0(key, cap);
    if (s == 0) return j0;
    const int64_t t = s - 1;
    return (int64_t)(((uint64_t)j0 + (uint64_t)((t * t) % cap)) % (uint64_t)cap);
}

__global__ void k_oak_seed(const uint64_t *__restrict__ keys, const uint16_t *__restrict__ vals, const uint8_t *__restrict__ cnts,
                           int64_t n, int64_t cap, uint64_t *okeys, uint16_t *ovals, uint8_t *ocnts, int64_t *work,
                           unsigned long long *count) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t k = keys[i];
        if (k == ~0ull) {                                   // the sentinel: first, into an empty table
            const int64_t j = oak_slot0(k, cap);
            okeys[j] = k; ovals[j] = vals[i]; ocnts[j] = cnts[i] ? cnts[i] : 1;
        } else {
            work[atomicAdd(count, 1ull)] = i;
        }
    }
}

__global__ void k_oak_bid(const uint64_t *__restrict__ keys, int64_t cap, uint64_t *okeys, const uint8_t *__restrict__ ocnts,
                          const int64_t *__restrict__ work, const unsigned long long *count, int64_t s) {
    const int64_t m = (int64_t)*count;
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < m; w += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t k = keys[work[w]];
        const int64_t j = oak_probe(k, cap, s);
        if (ocnts[j] == 0) atomicMin((unsigned long long *)&okeys[j], (unsigned long long)k);
    }
}

__global__ void k_oak_claim(const uint64_t *__restrict__ keys, const uint16_t *__restrict__ vals, const uint8_t *__restrict__ cnts,
                            int64_t cap, const uint64_t *__restrict__ okeys, uint16_t *ovals, uint8_t *ocnts,
                            const int64_t *__restrict__ work, const unsigned long long *count, int64_t *next,
                            unsigned long long *next_count, int64_t s) {
    const int64_t m = (int64_t)*count;
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < m; w += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = work[w];
        const uint64_t k = keys[i];
        const int64_t j = oak_probe(k, cap, s);
        if (okeys[j] == k) { ovals[j] = vals[i]; ocnts[j] = cnts[i] ? cnts[i] : 1; }
        else next[atomicAdd(next_count, 1ull)] = i;
    }
}

__global__ void k_oak_finish(uint64_t *okeys, const uint8_t *__restrict__ ocnts, int64_t cap) {
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < cap; j += (int64_t)gridDim.x * blockDim.x)
        if (ocnts[j] == 0) okeys[j] = 0;
}

struct DefHeader {
    uint8_t b[PG_DEFLATE_HDR_MAX];
};

__global__ void __launch_bounds__(PG_DEF_THREADS)
k_def_chunks(DefHeader hdr, int64_t hdr_len, const uint8_t *__restrict__ data, int64_t total, int64_t chunk, int64_t first,
             uint8_t *staging, int64_t slot_bytes, int64_t *sizes, uint32_t *crcs) {
    extern __shared__ __align__(16) uint8_t smem[];
    PgDeflateWs *ws = (PgDeflateWs *)smem;
    PgInflateWs *iws = (PgInflateWs *)(smem + ((sizeof(PgDeflateWs) + 15) & ~(size_t)15));
    uint32_t *crc_tab = (uint32_t *)((uint8_t *)iws + ((sizeof(PgInflateWs) + 15) & ~(size_t)15));
    uint8_t *in = (uint8_t *)(crc_tab + 256);
    const int64_t c = first + blockIdx.x;
    const int64_t p0 = c * chunk;
    const int64_t n = total - p0 < chunk ? total - p0 : chunk;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) crc_tab[i] = pg_crc_entry(i);
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        const int64_t p = p0 + i;
        in[i] = p < hdr_len ? hdr.b[p] : data[p - hdr_len];
    }
    __syncthreads();
    const int64_t size = pg_deflate_chunk(in, n, p0 + n == total, staging + (int64_t)blockIdx.x * slot_bytes, ws,
                                          PgDefLanes{(int)threadIdx.x, (int)blockDim.x});
    if (threadIdx.x < 32) {
        const uint32_t crc = pg_crc32_lanes(in, n, crc_tab, iws, PgLanes{(int)threadIdx.x, 32});
        if (threadIdx.x == 0) { sizes[blockIdx.x] = size; crcs[blockIdx.x] = crc; }
    }
}

size_t def_smem(int64_t chunk) {
    return ((sizeof(PgDeflateWs) + 15) & ~(size_t)15) + ((sizeof(PgInflateWs) + 15) & ~(size_t)15) + 1024 + (size_t)chunk;
}

// sizes[0, m) -> exclusive offsets, sizes[m] = total; state[0]: running CRC-32 of the member, chained over the chunks;
// state[1] = the slab's compressed bytes
__global__ void __launch_bounds__(1024)
k_def_scan(int64_t *sizes, const uint32_t *__restrict__ crcs, int64_t m, int64_t first, int64_t chunk, int64_t total,
           int64_t *state) {
    __shared__ int64_t part[1024];
    const int t = threadIdx.x;
    const int64_t per = (m + blockDim.x - 1) / blockDim.x;
    const int64_t a = t * per < m ? t * per : m, b = a + per < m ? a + per : m;
    int64_t s = 0;
    for (int64_t i = a; i < b; i++) s += sizes[i];
    part[t] = s;
    __syncthreads();
    if (t == 0) {
        int64_t acc = 0;
        for (int i = 0; i < (int)blockDim.x; i++) { const int64_t v = part[i]; part[i] = acc; acc += v; }
        state[1] = acc;
        // chunks have `chunk` bytes except the member's last: one shift operator serves all the full ones
        uint32_t crc = (uint32_t)state[0];
        const uint32_t shift = pg_crc_x8n(chunk);
        for (int64_t i = 0; i < m; i++) {
            const int64_t p0 = (first + i) * chunk, len = total - p0 < chunk ? total - p0 : chunk;
            crc = (len == chunk ? pg_crc_mulmod(shift, crc) : pg_crc_mulmod(pg_crc_x8n(len), crc)) ^ crcs[i];
        }
        state[0] = (int64_t)crc;
    }
    __syncthreads();
    int64_t acc = part[t];
    for (int64_t i = a; i < b; i++) { const int64_t v = sizes[i]; sizes[i] = acc; acc += v; }
    if (t == 0) sizes[m] = state[1];
}

__global__ void k_def_copy(const uint8_t *__restrict__ staging, int64_t slot_bytes, const int64_t *__restrict__ offs,
                           uint8_t *out) {
    const int64_t c = blockIdx.x;
    const int64_t o = offs[c], n = offs[c + 1] - o;
    const uint8_t *src = staging + c * slot_bytes;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) out[o + i] = src[i];
}

int grid_for(int64_t n, int threads) {
    const int64_t cap = (int64_t)pg_num_sms() * 8;
    int64_t g = (n + threads - 1) / threads;
    return (int)(g < 1 ? 1 : g > cap ? cap : g);
}

}  // namespace

extern "C" int64_t pg_oakht_place_workspace_bytes(int64_t n) { return 2 * (n > 0 ? n : 0) * 8 + 64; }

extern "C" int pg_oakht_place(const uint64_t *d_keys, const uint16_t *d_vals, const uint8_t *d_cnts, int64_t n, int64_t cap,
                              uint64_t *d_okeys, uint16_t *d_ovals, uint8_t *d_ocnts, void *d_ws, int64_t ws_bytes,
                              pg_stream_t stream_) {
    if (n < 0 || cap < 1 || n > cap || !d_okeys || !d_ovals || !d_ocnts || (n && (!d_keys || !d_vals || !d_cnts || !d_ws)))
        return pg_fail(PG_ERR_INVALID, "pg_oakht_place: bad arguments");
    if (ws_bytes < pg_oakht_place_workspace_bytes(n))
        return pg_fail(PG_ERR_WORKSPACE, "pg_oakht_place: workspace of %lld bytes, %lld needed", (long long)ws_bytes,
                       (long long)pg_oakht_place_workspace_bytes(n));
    cudaStream_t s = (cudaStream_t)stream_;
    PG_CUDA(cudaMemsetAsync(d_okeys, 0xFF, (size_t)cap * 8, s));
    PG_CUDA(cudaMemsetAsync(d_ovals, 0, (size_t)cap * 2, s));
    PG_CUDA(cudaMemsetAsync(d_ocnts, 0, (size_t)cap, s));
    unsigned long long *counts = (unsigned long long *)d_ws;            // [0], [1]: the two work lists' lengths
    int64_t *work[2] = {(int64_t *)((char *)d_ws + 64), (int64_t *)((char *)d_ws + 64) + n};
    PG_CUDA(cudaMemsetAsync(counts, 0, 16, s));
    if (n) k_oak_seed<<<grid_for(n, 256), 256, 0, s>>>(d_keys, d_vals, d_cnts, n, cap, d_okeys, d_ovals, d_ocnts, work[0], counts);
    PG_CUDA(cudaGetLastError());
    int64_t left = n, rounds = 0, s_probe = 0;
    int cur = 0;
    while (left > 0) {
        if (rounds >= PG_OAK_MAX_ROUNDS)
            return pg_fail(PG_ERR_CAPACITY, "pg_oakht_place: probe sequence exhausted (%lld entries unplaced after %d rounds)",
                           (long long)left, PG_OAK_MAX_ROUNDS);
        const int g = grid_for(left, 256);
        for (int r = 0; r < PG_OAK_BATCH && rounds < PG_OAK_MAX_ROUNDS; r++, rounds++) {
            PG_CUDA(cudaMemsetAsync(counts + (cur ^ 1), 0, 8, s));
            k_oak_bid<<<g, 256, 0, s>>>(d_keys, cap, d_okeys, d_ocnts, work[cur], counts + cur, s_probe);
            k_oak_claim<<<g, 256, 0, s>>>(d_keys, d_vals, d_cnts, cap, d_okeys, d_ovals, d_ocnts, work[cur], counts + cur,
                                          work[cur ^ 1], counts + (cur ^ 1), s_probe);
            PG_CUDA(cudaGetLastError());
            cur ^= 1;
            s_probe = s_probe == 0 ? 2 : s_probe + 1;
        }
        unsigned long long h = 0;
        PG_CUDA(cudaMemcpyAsync(&h, counts + cur, 8, cudaMemcpyDeviceToHost, s));
        PG_CUDA(cudaStreamSynchronize(s));
        left = (int64_t)h;
    }
    k_oak_finish<<<grid_for(cap, 256), 256, 0, s>>>(d_okeys, d_ocnts, cap);
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}

extern "C" int64_t pg_deflate_slot_bytes(int64_t chunk_bytes) { return ((chunk_bytes + 8) + 15) / 16 * 16; }

extern "C" int pg_deflate_chunks(const uint8_t *hdr, int64_t hdr_len, const uint8_t *d_data, int64_t data_len,
                                 int64_t chunk_bytes, int64_t first_chunk, int64_t n_chunks, uint8_t *d_staging,
                                 int64_t slot_bytes, int64_t *d_sizes, uint32_t *d_crcs, pg_stream_t stream) {
    const int64_t total = hdr_len + data_len;
    const int64_t all = total ? (total + chunk_bytes - 1) / chunk_bytes : 1;
    if (chunk_bytes < 1 || chunk_bytes > PG_DEF_MAX_CHUNK || hdr_len < 0 || hdr_len > PG_DEFLATE_HDR_MAX || data_len < 0 ||
        (hdr_len && !hdr) || (data_len && !d_data) || first_chunk < 0 || n_chunks < 0 || first_chunk + n_chunks > all ||
        n_chunks > 0x7FFFFFFF || slot_bytes < pg_deflate_slot_bytes(chunk_bytes) || slot_bytes % 16 || !d_staging || !d_sizes || !d_crcs)
        return pg_fail(PG_ERR_INVALID, "pg_deflate_chunks: bad arguments");
    if (n_chunks == 0) return PG_OK;
    DefHeader h;
    memset(&h, 0, sizeof h);
    if (hdr_len) memcpy(h.b, hdr, (size_t)hdr_len);
    const size_t smem = def_smem(chunk_bytes);
    PG_CUDA(cudaFuncSetAttribute(k_def_chunks, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_def_chunks<<<(unsigned)n_chunks, PG_DEF_THREADS, smem, (cudaStream_t)stream>>>(h, hdr_len, d_data, total, chunk_bytes, first_chunk,
                                                                                    d_staging, slot_bytes, d_sizes, d_crcs);
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}

extern "C" int pg_deflate_compact(const uint8_t *d_staging, int64_t slot_bytes, int64_t *d_sizes, const uint32_t *d_crcs,
                                  int64_t first_chunk, int64_t n_chunks, int64_t chunk_bytes, int64_t total_bytes, uint8_t *d_out,
                                  int64_t *d_state, pg_stream_t stream) {
    if (!d_staging || !d_sizes || !d_crcs || !d_out || !d_state || n_chunks < 1 || n_chunks > 0x7FFFFFFF || chunk_bytes < 1 ||
        chunk_bytes > PG_DEF_MAX_CHUNK || first_chunk < 0 || total_bytes < 0)
        return pg_fail(PG_ERR_INVALID, "pg_deflate_compact: bad arguments");
    cudaStream_t s = (cudaStream_t)stream;
    k_def_scan<<<1, 1024, 0, s>>>(d_sizes, d_crcs, n_chunks, first_chunk, chunk_bytes, total_bytes, d_state);
    k_def_copy<<<(unsigned)n_chunks, 256, 0, s>>>(d_staging, slot_bytes, d_sizes, d_out);
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}
