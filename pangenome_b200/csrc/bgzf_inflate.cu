// bgzf_inflate.cu - BGZF input: the member index (host) and the inflate kernel (sm_100a).
//
// A BGZF file is a chain of gzip members of at most 64 KiB output each; every member is a self-contained raw-DEFLATE
// stream whose compressed size (BSIZE) and output size (ISIZE) sit in its header and trailer.  The host walks the
// headers only (pg_host_bgzf_index: a few bytes per 64 KiB), the compressed file crosses PCIe as it is, and ONE launch
// inflates every member straight into the buffer K1 (pg_fasta_scan_pack) reads.
//
// Kernel shape: one warp per member, WARPS warps per CTA, the member's Huffman tables and scratch in shared memory
// (PgInflateWs, about 3.7 KB per warp).  DEFLATE decoding is a serial chain - the position of symbol i+1 is known only
// once symbol i is decoded - so parallelism comes from members: a 1 GB file has ~16 000, several per SM.  Inside the
// warp every lane runs the same decoder on the same bits (inflate.cuh), which keeps the warp converged without a
// shuffle per symbol; the lanes share the work without a serial dependency (look-up table fills, match and stored
// copies, the CRC-32 of the output).  Lane 0 writes literals.
#include "common.cuh"
#include "inflate.cuh"

#define PG_BGZF_WARPS 4

namespace {

__global__ void k_bgzf_status_init(int64_t *status) {
    status[0] = 0;
    status[1] = INT64_MAX;
}

__global__ void __launch_bounds__(PG_BGZF_WARPS * 32)
k_bgzf_inflate(const uint8_t *__restrict__ gz, int64_t gz_bytes, const int64_t *__restrict__ member_off,
               const int64_t *__restrict__ out_off, int64_t n_members, uint8_t *out, int64_t out_bytes, int64_t *status) {
    __shared__ PgInflateWs ws[PG_BGZF_WARPS];
    __shared__ uint32_t crc_tab[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) crc_tab[i] = pg_crc_entry(i);
    __syncthreads();
    const int warp = threadIdx.x >> 5;
    const int64_t m = (int64_t)blockIdx.x * PG_BGZF_WARPS + warp;
    if (m >= n_members) return;
    PgLanes L{(int)(threadIdx.x & 31), 32};
    const int64_t mb = member_off[m], me = member_off[m + 1];
    const int64_t ob = out_off[m], oe = out_off[m + 1];
    int err;
    if (mb < 0 || me < mb || me > gz_bytes || ob < 0 || oe < ob || oe > out_bytes)
        err = PG_INF_ERR_HEADER;                       // the caller's window does not lie inside the buffers
    else
        err = pg_bgzf_member(gz + mb, me - mb, out + ob, oe - ob, crc_tab, &ws[warp], L);
    if (err && L.lane == 0) {
        atomicAdd((unsigned long long *)&status[0], 1ull);
        atomicMin((long long *)&status[1], (long long)((m << 8) | err));
    }
}

inline uint32_t le16(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }

// size of the BGZF member at gz[pos], 0 when the bytes there are not a BGZF header (or the header runs past the end)
int64_t bgzf_member_size(const uint8_t *gz, int64_t nbytes, int64_t pos) {
    if (nbytes - pos < 12) return 0;
    const uint8_t *h = gz + pos;
    if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || h[3] != 4) return 0;
    const int64_t xlen = le16(h + 10);
    if (nbytes - pos < 12 + xlen) return 0;
    for (int64_t x = 12; x + 4 <= 12 + xlen;) {
        const int64_t slen = le16(h + x + 2);
        if (h[x] == 'B' && h[x + 1] == 'C' && slen == 2 && x + 6 <= 12 + xlen) return (int64_t)le16(h + x + 4) + 1;
        x += 4 + slen;
    }
    return 0;
}

}  // namespace

extern "C" int pg_host_bgzf_index(const uint8_t *gz, int64_t nbytes, int64_t *member_off, int64_t *out_off, int64_t cap,
                                  int64_t *counts) {
    if (nbytes < 0 || cap < 0 || !counts || (nbytes && !gz) || (cap && (!member_off || !out_off)))
        return pg_fail(PG_ERR_INVALID, "pg_host_bgzf_index: bad arguments");
    int64_t pos = 0, n = 0, total = 0;
    if (nbytes == 0 || bgzf_member_size(gz, nbytes, 0) == 0)
        return pg_fail(PG_ERR_NOT_BGZF, "pg_host_bgzf_index: the input does not start with a BGZF member");
    while (pos < nbytes) {
        const int64_t size = bgzf_member_size(gz, nbytes, pos);
        if (size == 0)
            return pg_fail(PG_ERR_INVALID, "pg_host_bgzf_index: no BGZF member header at byte %lld (member %lld)",
                           (long long)pos, (long long)n);
        const int64_t xlen = le16(gz + pos + 10);
        if (size < 12 + xlen + 8)
            return pg_fail(PG_ERR_INVALID, "pg_host_bgzf_index: BSIZE of the member at byte %lld is smaller than its header",
                           (long long)pos);
        if (size > nbytes - pos)
            return pg_fail(PG_ERR_INVALID, "pg_host_bgzf_index: the member at byte %lld is truncated (BSIZE %lld, %lld bytes left)",
                           (long long)pos, (long long)size, (long long)(nbytes - pos));
        const int64_t isize = (int64_t)pg_le32(gz + pos + size - 4);
        if (isize > 65536)
            return pg_fail(PG_ERR_INVALID, "pg_host_bgzf_index: the member at byte %lld claims %lld output bytes (BGZF: at most 65536)",
                           (long long)pos, (long long)isize);
        if (n < cap) { member_off[n] = pos; out_off[n] = total; }
        total += isize;
        pos += size;
        n++;
    }
    if (n <= cap) { member_off[n] = nbytes; out_off[n] = total; }
    counts[0] = n;
    counts[1] = total;
    return PG_OK;
}

extern "C" int pg_bgzf_inflate(const uint8_t *d_gz, int64_t gz_bytes, const int64_t *d_member_off, const int64_t *d_out_off,
                               int64_t n_members, uint8_t *d_out, int64_t out_bytes, int64_t *d_status, pg_stream_t stream) {
    if (n_members < 0 || gz_bytes < 0 || out_bytes < 0 || !d_status || (n_members && (!d_gz || !d_member_off || !d_out_off)))
        return pg_fail(PG_ERR_INVALID, "pg_bgzf_inflate: bad arguments");
    cudaStream_t s = (cudaStream_t)stream;
    k_bgzf_status_init<<<1, 1, 0, s>>>(d_status);
    PG_CUDA(cudaGetLastError());
    if (n_members == 0) return PG_OK;
    const int64_t blocks = (n_members + PG_BGZF_WARPS - 1) / PG_BGZF_WARPS;
    if (blocks > 0x7FFFFFFF) return pg_fail(PG_ERR_INVALID, "pg_bgzf_inflate: too many members");
    k_bgzf_inflate<<<(unsigned)blocks, PG_BGZF_WARPS * 32, 0, s>>>(d_gz, gz_bytes, d_member_off, d_out_off, n_members, d_out,
                                                                   out_bytes, d_status);
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}
