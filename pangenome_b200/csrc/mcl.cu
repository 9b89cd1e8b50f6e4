// mcl.cu - K7m: Markov clustering of the rdBG edge graph (opt-in replacement of the external `mcl` run,
// kmer_numba.py:1911).  The arithmetic is specified in include/pgdbg.h and DESIGN.md §3; every float32 operation
// here is an explicitly rounded intrinsic (nvcc would otherwise contract a*b+c into an FMA) and every sum runs left
// to right in the specified order, so oracle/mcl.c reproduces the matrices bit for bit.
//
//   plan      thread per column: product count, staging size min(products, S), list of large columns
//   expand    warp per column (<= PG_MCL_WARP_PRODUCTS products, shared-memory accumulator) or CTA per column
//             (shared accumulator up to PG_MCL_SMEM_SLOTS slots, else a global slab per CTA); both run mcl_column:
//               1. accumulate: for k in column j in ascending order, the group adds M[i,k]*M[k,j] for the rows i of
//                  column k into a hash keyed by row - rows of one column k are distinct, so each accumulator is
//                  touched once per k and the group synchronises between k: every sum runs in ascending k;
//               2. select: counts over the accumulator find the threshold key (value bits, then row) of the
//                  min(S, #entries >= theta) largest entries by binary search - no sort of the full column;
//               3. order the kept entries by row (rank counting, <= S entries), inflate, one thread normalises;
//   compact   scan of the kept counts -> next column pointers, warp per column copy
//   components atomic-hooking union-find over the stored entries (the smaller index becomes the root)
#include <cooperative_groups.h>
#include "common.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int SCAN_T = 1024;
constexpr int MCL_T = 256;
constexpr int WARPS = MCL_T / 32;
constexpr int S = PG_MCL_SELECT_S;
constexpr int WARP_P = PG_MCL_WARP_PRODUCTS;
constexpr int WARP_SLOTS = 2 * WARP_P;

// ---- int64 exclusive scan (n + 1 outputs, the total last); in == out allowed --------------------------------
__device__ long long block_incl_scan(long long v, long long *s_warp) {
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int o = 1; o < 32; o <<= 1) { long long y = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += y; }
    if (lane == 31) s_warp[w] = v;
    __syncthreads();
    if (w == 0) {
        long long t = lane < (int)(blockDim.x >> 5) ? s_warp[lane] : 0;
        for (int o = 1; o < 32; o <<= 1) { long long y = __shfl_up_sync(0xffffffffu, t, o); if (lane >= o) t += y; }
        s_warp[lane] = t;
    }
    __syncthreads();
    if (w > 0) v += s_warp[w - 1];
    __syncthreads();
    return v;
}
__global__ void __launch_bounds__(SCAN_T) k_scan_sums(const int64_t *in, int64_t n, int64_t *bsum) {
    __shared__ long long s[32];
    int64_t i = blockIdx.x * (int64_t)SCAN_T + threadIdx.x;
    long long v = block_incl_scan(i < n ? in[i] : 0, s);
    if (threadIdx.x == SCAN_T - 1) bsum[blockIdx.x] = v;
}
__global__ void __launch_bounds__(SCAN_T) k_scan_top(int64_t *bsum, int64_t nb) {
    __shared__ long long s[32];
    __shared__ long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int64_t base = 0; base < nb; base += SCAN_T) {
        int64_t i = base + threadIdx.x;
        long long v = i < nb ? bsum[i] : 0;
        long long incl = block_incl_scan(v, s);
        long long c = carry;
        if (i < nb) bsum[i] = c + incl - v;
        __syncthreads();
        if (threadIdx.x == SCAN_T - 1) carry = c + incl;
        __syncthreads();
    }
}
__global__ void __launch_bounds__(SCAN_T) k_scan_apply(const int64_t *in, int64_t n, const int64_t *bsum, int64_t *out) {
    __shared__ long long s[32];
    int64_t i = blockIdx.x * (int64_t)SCAN_T + threadIdx.x;
    long long v = i < n ? in[i] : 0;
    long long incl = block_incl_scan(v, s) + bsum[blockIdx.x];
    if (i < n) out[i] = incl - v;
    if (i == n - 1) out[n] = incl;
}
int scan_excl(const int64_t *in, int64_t n, int64_t *out, void *ws, int64_t ws_bytes, cudaStream_t st) {
    if (ws_bytes < pg_mcl_scan_workspace_bytes(n)) return pg_fail(PG_ERR_WORKSPACE, "mcl scan: workspace too small");
    if (n == 0) { PG_CUDA(cudaMemsetAsync(out, 0, 8, st)); return PG_OK; }
    int64_t nb = (n + SCAN_T - 1) / SCAN_T;
    int64_t *bsum = reinterpret_cast<int64_t *>(ws);
    k_scan_sums<<<(unsigned)nb, SCAN_T, 0, st>>>(in, n, bsum);
    k_scan_top<<<1, SCAN_T, 0, st>>>(bsum, nb);
    k_scan_apply<<<(unsigned)nb, SCAN_T, 0, st>>>(in, n, bsum, out);
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}

// ---- the specified float32 arithmetic ------------------------------------------------------------------------
struct Inflate {
    float r;
    int whole;      // floor(r) when r is a multiple of 1/2, else 0 (powf)
    bool half;
    __device__ __forceinline__ float operator()(float x) const {
        if (whole == 0) return powf(x, r);
        float p = x;
        for (int i = 1; i < whole; i++) p = __fmul_rn(p, x);
        return half ? __fmul_rn(p, __fsqrt_rn(x)) : p;
    }
};

// one thread: divide the column by its sum (ascending row), return chaos = max / sum of squares - 1
__device__ float column_finish(float *v, int64_t K) {
    if (K == 0) return 0.f;
    float sum = 0.f;
    for (int64_t e = 0; e < K; e++) sum = __fadd_rn(sum, v[e]);
    float mx = 0.f, sq = 0.f;
    for (int64_t e = 0; e < K; e++) {
        float x = __fdiv_rn(v[e], sum);
        v[e] = x;
        mx = fmaxf(mx, x);
        sq = __fadd_rn(sq, __fmul_rn(x, x));
    }
    return __fsub_rn(__fdiv_rn(mx, sq), 1.f);
}

__device__ __forceinline__ void stats_column(int64_t *stats, float chaos, int64_t K) {
    atomicMax(reinterpret_cast<unsigned long long *>(stats + PG_MCL_STAT_CHAOS), (unsigned long long)__float_as_uint(fmaxf(chaos, 0.f)));
    atomicAdd(reinterpret_cast<unsigned long long *>(stats + PG_MCL_STAT_NNZ), (unsigned long long)K);
}

// group-wide sum of one int per thread through a shared word
template <class G>
__device__ __forceinline__ int gsum(G &g, int v, int *word) {
    if (g.thread_rank() == 0) *word = 0;
    g.sync();
    if (v) atomicAdd(word, v);
    g.sync();
    int r = *word;
    g.sync();
    return r;
}

__device__ __forceinline__ unsigned row_hash(int32_t i) { return (uint32_t)i * 0x9E3779B1u; }

// keep an accumulator entry iff (value bits, -row) >= (tb, -tr)
__device__ __forceinline__ bool keeps(float v, int32_t row, uint32_t tb, int32_t tr) {
    uint32_t b = __float_as_uint(v);
    return b > tb || (b == tb && row <= tr);
}

struct ColumnBufs {
    int32_t *hkey; float *hval; int hcap;      // accumulator (power-of-two slots)
    int32_t *krow; float *kval;                // kept entries, unordered
    int32_t *srow; float *sval;                // kept entries by row
    int *word;                                 // 2 ints of shared scratch
};

template <class G>
__device__ void mcl_column(G &g, int64_t j, const int64_t *__restrict__ cp, const int32_t *__restrict__ rows,
                           const float *__restrict__ vals, const ColumnBufs &b, const Inflate &pw, const int64_t *__restrict__ stage_off,
                           int32_t *__restrict__ out_rows, float *__restrict__ out_vals, int64_t *__restrict__ kept, int64_t *stats) {
    const int tid = g.thread_rank(), nt = g.num_threads();
    const unsigned mask = (unsigned)b.hcap - 1u;
    for (int s = tid; s < b.hcap; s += nt) { b.hkey[s] = -1; b.hval[s] = 0.f; }
    g.sync();
    // 1. expansion, ascending k
    for (int64_t p = cp[j]; p < cp[j + 1]; p++) {
        int32_t k = rows[p];
        float mkj = vals[p];
        for (int64_t q = cp[k] + tid; q < cp[k + 1]; q += nt) {
            int32_t i = rows[q];
            float prod = __fmul_rn(vals[q], mkj);
            unsigned s = row_hash(i) & mask;
            for (;;) {
                int32_t old = atomicCAS(b.hkey + s, -1, i);
                if (old == -1 || old == i) break;
                s = (s + 1) & mask;
            }
            b.hval[s] = __fadd_rn(b.hval[s], prod);
        }
        g.sync();
    }
    // 2. selection: want = min(S, #entries >= theta), or 1 when no entry reaches theta
    int c_all = 0, c_theta = 0;
    for (int s = tid; s < b.hcap; s += nt)
        if (b.hkey[s] >= 0) { c_all++; c_theta += b.hval[s] >= PG_MCL_PRUNE_THETA; }
    c_all = gsum(g, c_all, b.word);
    c_theta = gsum(g, c_theta, b.word);
    if (c_all == 0) { if (tid == 0) kept[j] = 0; return; }
    int want = c_theta == 0 ? 1 : (c_theta < S ? c_theta : S);
    uint32_t tb = 0;
    int32_t tr = 0x7fffffff;
    if (want == c_theta) {
        tb = __float_as_uint(PG_MCL_PRUNE_THETA);
    } else if (want < c_all) {
        // largest tb with #(bits >= tb) >= want, then the smallest tr with #(bits == tb, row <= tr) >= want - #(bits > tb)
        uint32_t lo = 0, hi = 0x7f800000u;
        while (lo < hi) {
            uint32_t mid = lo + (hi - lo + 1) / 2;
            int c = 0;
            for (int s = tid; s < b.hcap; s += nt) c += b.hkey[s] >= 0 && __float_as_uint(b.hval[s]) >= mid;
            if (gsum(g, c, b.word) >= want) lo = mid; else hi = mid - 1;
        }
        tb = lo;
        int c = 0;
        for (int s = tid; s < b.hcap; s += nt) c += b.hkey[s] >= 0 && __float_as_uint(b.hval[s]) > tb;
        int q = want - gsum(g, c, b.word);
        int32_t rlo = 0, rhi = 0x7fffffff;
        while (rlo < rhi) {
            int32_t mid = rlo + (rhi - rlo) / 2;
            c = 0;
            for (int s = tid; s < b.hcap; s += nt) c += b.hkey[s] >= 0 && b.hkey[s] <= mid && __float_as_uint(b.hval[s]) == tb;
            if (gsum(g, c, b.word) >= q) rhi = mid; else rlo = mid + 1;
        }
        tr = rlo;
    }
    // 3. compact the kept entries, order them by row, inflate, normalise
    if (tid == 0) b.word[1] = 0;
    g.sync();
    for (int s = tid; s < b.hcap; s += nt) {
        int32_t i = b.hkey[s];
        if (i >= 0 && keeps(b.hval[s], i, tb, tr)) {
            int at = atomicAdd(b.word + 1, 1);
            b.krow[at] = i; b.kval[at] = b.hval[s];
        }
    }
    g.sync();
    const int K = b.word[1];
    for (int e = tid; e < K; e += nt) {
        int32_t i = b.krow[e];
        int r = 0;
        for (int f = 0; f < K; f++) r += b.krow[f] < i;
        b.srow[r] = i; b.sval[r] = pw(b.kval[e]);
    }
    g.sync();
    if (tid == 0) {
        float chaos = column_finish(b.sval, K);
        kept[j] = K;
        stats_column(stats, chaos, K);
    }
    g.sync();
    const int64_t off = stage_off[j];
    for (int e = tid; e < K; e += nt) { out_rows[off + e] = b.srow[e]; out_vals[off + e] = b.sval[e]; }
}

__device__ __forceinline__ int pow2_at_least(int64_t x) {
    int c = 2;
    while (c < x) c <<= 1;
    return c;
}

__global__ void __launch_bounds__(MCL_T) k_mcl_warp(const int64_t *__restrict__ cp, const int32_t *__restrict__ rows, const float *__restrict__ vals,
                                                    int64_t n, const int64_t *__restrict__ prod, const int64_t *__restrict__ stage_off, Inflate pw,
                                                    int32_t *__restrict__ out_rows, float *__restrict__ out_vals, int64_t *__restrict__ kept, int64_t *stats) {
    __shared__ int32_t hk[WARPS][WARP_SLOTS];
    __shared__ float hv[WARPS][WARP_SLOTS];
    __shared__ int32_t kr[WARPS][WARP_P], sr[WARPS][WARP_P];
    __shared__ float kv[WARPS][WARP_P], sv[WARPS][WARP_P];
    __shared__ int word[WARPS][2];
    auto tile = cg::tiled_partition<32>(cg::this_thread_block());
    const int w = threadIdx.x >> 5;
    const int64_t j = blockIdx.x * (int64_t)WARPS + w;
    if (j >= n) return;
    const int64_t P = prod[j];
    if (P > WARP_P) return;                                    // the CTA path takes it
    ColumnBufs b{hk[w], hv[w], pow2_at_least(2 * P), kr[w], kv[w], sr[w], sv[w], word[w]};
    mcl_column(tile, j, cp, rows, vals, b, pw, stage_off, out_rows, out_vals, kept, stats);
}

__global__ void __launch_bounds__(MCL_T) k_mcl_cta(const int64_t *__restrict__ cp, const int32_t *__restrict__ rows, const float *__restrict__ vals,
                                                   int64_t n, const int64_t *__restrict__ prod, const int64_t *__restrict__ stage_off,
                                                   const int32_t *__restrict__ large, int64_t n_large, Inflate pw,
                                                   int32_t *__restrict__ out_rows, float *__restrict__ out_vals, int64_t *__restrict__ kept, int64_t *stats,
                                                   int32_t *slab_keys, float *slab_vals, int64_t slab_slots) {
    __shared__ int32_t hk[PG_MCL_SMEM_SLOTS];
    __shared__ float hv[PG_MCL_SMEM_SLOTS];
    __shared__ int32_t kr[S], sr[S];
    __shared__ float kv[S], sv[S];
    __shared__ int word[2];
    auto block = cg::this_thread_block();
    for (int64_t t = blockIdx.x; t < n_large; t += gridDim.x) {
        const int64_t j = large[t];
        const int64_t P = prod[j];
        const int hcap = pow2_at_least(2 * (P < n ? P : n));
        ColumnBufs b{hk, hv, hcap, kr, kv, sr, sv, word};
        if (hcap > PG_MCL_SMEM_SLOTS) { b.hkey = slab_keys + blockIdx.x * slab_slots; b.hval = slab_vals + blockIdx.x * slab_slots; }
        mcl_column(block, j, cp, rows, vals, b, pw, stage_off, out_rows, out_vals, kept, stats);
        block.sync();
    }
}

__global__ void k_mcl_plan(const int64_t *__restrict__ cp, const int32_t *__restrict__ rows, int64_t n, int64_t *__restrict__ prod,
                           int64_t *__restrict__ stage_cap, int32_t *__restrict__ large, int64_t *stats) {
    int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    long long p = 0;
    if (j < n) {
        for (int64_t q = cp[j]; q < cp[j + 1]; q++) { int32_t k = rows[q]; p += cp[k + 1] - cp[k]; }
        prod[j] = p;
        stage_cap[j] = p < S ? p : S;
        if (p > WARP_P) large[atomicAdd(reinterpret_cast<unsigned long long *>(stats + PG_MCL_STAT_LARGE), 1ull)] = (int32_t)j;
    }
    long long sum = p, mx = p;
    for (int o = 16; o; o >>= 1) {
        sum += __shfl_down_sync(0xffffffffu, sum, o);
        long long y = __shfl_down_sync(0xffffffffu, mx, o);
        mx = y > mx ? y : mx;
    }
    if ((threadIdx.x & 31) == 0 && sum) {
        atomicAdd(reinterpret_cast<unsigned long long *>(stats + PG_MCL_STAT_PRODUCTS), (unsigned long long)sum);
        atomicMax(reinterpret_cast<unsigned long long *>(stats + PG_MCL_STAT_MAXPROD), (unsigned long long)mx);
    }
}

__global__ void k_mcl_normalise(const int64_t *__restrict__ cp, float *vals, int64_t n, int64_t *stats) {
    int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j >= n) return;
    int64_t K = cp[j + 1] - cp[j];
    stats_column(stats, column_finish(vals + cp[j], K), K);
}

__global__ void __launch_bounds__(MCL_T) k_mcl_compact(const int64_t *__restrict__ stage_off, const int32_t *__restrict__ srows, const float *__restrict__ svals,
                                                       const int64_t *__restrict__ kept, int64_t n, const int64_t *__restrict__ cp_out,
                                                       int32_t *__restrict__ rows_out, float *__restrict__ vals_out) {
    const int64_t j = blockIdx.x * (int64_t)WARPS + (threadIdx.x >> 5);
    if (j >= n) return;
    const int64_t src = stage_off[j], dst = cp_out[j], K = kept[j];
    for (int64_t e = threadIdx.x & 31; e < K; e += 32) { rows_out[dst + e] = srows[src + e]; vals_out[dst + e] = svals[src + e]; }
}

__device__ __forceinline__ int32_t uf_root(int32_t *parent, int32_t x) {
    int32_t p = parent[x];
    while (p != x) { int32_t gp = parent[p]; if (gp != p) parent[x] = gp; x = p; p = gp; }   // path halving (benign race)
    return x;
}
__global__ void k_mcl_uf_init(int32_t *parent, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) parent[i] = (int32_t)i;
}
__global__ void k_mcl_union(const int64_t *__restrict__ cp, const int32_t *__restrict__ rows, int64_t n, int32_t *parent) {
    int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j >= n) return;
    for (int64_t q = cp[j]; q < cp[j + 1]; q++) {
        int32_t a = (int32_t)j, b = rows[q];
        for (;;) {
            a = uf_root(parent, a); b = uf_root(parent, b);
            if (a == b) break;
            if (a < b) { int32_t t = a; a = b; b = t; }                 // hook the larger root under the smaller
            if (atomicCAS(parent + a, a, b) == a) break;
        }
    }
}
__global__ void k_mcl_flatten(int32_t *parent, int64_t n) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    int32_t r = (int32_t)i;
    while (parent[r] != r) r = parent[r];
    parent[i] = r;
}

inline unsigned nblocks(int64_t n, int t) { return (unsigned)(n > 0 ? (n + t - 1) / t : 1); }

int check_csc(const int64_t *cp, const int32_t *rows, int64_t n, const char *who) {
    if (!cp || n < 0 || n >= (1ll << 31) || (n > 0 && !rows)) return pg_fail(PG_ERR_INVALID, "%s: bad matrix arguments", who);
    return PG_OK;
}

}  // namespace

extern "C" int64_t pg_mcl_scan_workspace_bytes(int64_t n) { return (n / SCAN_T + 2) * 8 + 256; }

extern "C" int64_t pg_mcl_slab_slots(int64_t max_products, int64_t n) {
    int64_t m = max_products < n ? max_products : n, c = 2;
    while (c < 2 * m) c <<= 1;
    return c;
}

extern "C" int pg_mcl_normalise(const int64_t *d_colptr, const int32_t *d_rows, float *d_vals, int64_t n, int64_t *d_stats,
                                pg_stream_t stream_) {
    int rc = check_csc(d_colptr, d_rows, n, "pg_mcl_normalise"); if (rc) return rc;
    if (!d_stats || (n > 0 && !d_vals)) return pg_fail(PG_ERR_INVALID, "pg_mcl_normalise: bad arguments");
    if (n == 0) return PG_OK;
    k_mcl_normalise<<<nblocks(n, 256), 256, 0, (cudaStream_t)stream_>>>(d_colptr, d_vals, n, d_stats);
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}

extern "C" int pg_mcl_plan(const int64_t *d_colptr, const int32_t *d_rows, int64_t n, int64_t *d_prod, int64_t *d_stage_off,
                           int32_t *d_large, int64_t *d_stats, void *d_scan_ws, int64_t scan_ws_bytes, pg_stream_t stream_) {
    int rc = check_csc(d_colptr, d_rows, n, "pg_mcl_plan"); if (rc) return rc;
    if (!d_prod || !d_stage_off || !d_large || !d_stats || !d_scan_ws) return pg_fail(PG_ERR_INVALID, "pg_mcl_plan: bad arguments");
    cudaStream_t st = (cudaStream_t)stream_;
    if (n > 0) k_mcl_plan<<<nblocks(n, 256), 256, 0, st>>>(d_colptr, d_rows, n, d_prod, d_stage_off, d_large, d_stats);
    PG_CUDA(cudaGetLastError());
    return scan_excl(d_stage_off, n, d_stage_off, d_scan_ws, scan_ws_bytes, st);
}

extern "C" int pg_mcl_expand(const int64_t *d_colptr, const int32_t *d_rows, const float *d_vals, int64_t n, const int64_t *d_prod,
                             const int64_t *d_stage_off, const int32_t *d_large, int64_t n_large, int64_t max_products, float inflation,
                             int32_t *d_stage_rows, float *d_stage_vals, int64_t *d_kept, int64_t *d_stats, void *d_ws, int64_t ws_bytes,
                             int n_ctas, pg_stream_t stream_) {
    int rc = check_csc(d_colptr, d_rows, n, "pg_mcl_expand"); if (rc) return rc;
    if (!d_vals || !d_prod || !d_stage_off || !d_kept || !d_stats || n_large < 0 || n_large > n || (n_large > 0 && !d_large) ||
        !(inflation > 1.f) || !(inflation < 64.f))
        return pg_fail(PG_ERR_INVALID, "pg_mcl_expand: bad arguments (inflation must be in (1, 64))");
    if (n == 0) return PG_OK;
    if (!d_stage_rows || !d_stage_vals) return pg_fail(PG_ERR_INVALID, "pg_mcl_expand: null staging buffers");
    Inflate pw;
    pw.r = inflation;
    float twice = inflation * 2.f;
    pw.whole = (twice == floorf(twice)) ? (int)floorf(inflation) : 0;
    pw.half = pw.whole && (twice != 2.f * floorf(inflation));
    cudaStream_t st = (cudaStream_t)stream_;
    k_mcl_warp<<<nblocks(n, WARPS), MCL_T, 0, st>>>(d_colptr, d_rows, d_vals, n, d_prod, d_stage_off, pw, d_stage_rows, d_stage_vals, d_kept, d_stats);
    PG_CUDA(cudaGetLastError());
    if (n_large > 0) {
        int64_t slab = pg_mcl_slab_slots(max_products, n);
        if (slab > PG_MCL_SMEM_SLOTS) {
            if (n_ctas < 1 || !d_ws || ws_bytes < (int64_t)n_ctas * slab * 8)
                return pg_fail(PG_ERR_WORKSPACE, "pg_mcl_expand: workspace too small for %d CTAs of %lld slots", n_ctas, (long long)slab);
        } else if (n_ctas < 1) {
            return pg_fail(PG_ERR_INVALID, "pg_mcl_expand: n_ctas < 1");
        }
        int32_t *keys = reinterpret_cast<int32_t *>(d_ws);
        float *vals = keys ? reinterpret_cast<float *>(keys + (int64_t)n_ctas * slab) : nullptr;
        int64_t grid = n_large < n_ctas ? n_large : n_ctas;
        k_mcl_cta<<<(unsigned)grid, MCL_T, 0, st>>>(d_colptr, d_rows, d_vals, n, d_prod, d_stage_off, d_large, n_large, pw, d_stage_rows,
                                                   d_stage_vals, d_kept, d_stats, keys, vals, slab);
        PG_CUDA(cudaGetLastError());
    }
    return PG_OK;
}

extern "C" int pg_mcl_compact(const int64_t *d_stage_off, const int32_t *d_stage_rows, const float *d_stage_vals, const int64_t *d_kept,
                              int64_t n, int64_t *d_colptr_out, int32_t *d_rows_out, float *d_vals_out, void *d_scan_ws,
                              int64_t scan_ws_bytes, pg_stream_t stream_) {
    if (n < 0 || !d_stage_off || !d_kept || !d_colptr_out || !d_scan_ws) return pg_fail(PG_ERR_INVALID, "pg_mcl_compact: bad arguments");
    cudaStream_t st = (cudaStream_t)stream_;
    int rc = scan_excl(d_kept, n, d_colptr_out, d_scan_ws, scan_ws_bytes, st); if (rc) return rc;
    if (n == 0) return PG_OK;
    if (!d_stage_rows || !d_stage_vals || !d_rows_out || !d_vals_out) return pg_fail(PG_ERR_INVALID, "pg_mcl_compact: null buffers");
    k_mcl_compact<<<nblocks(n, WARPS), MCL_T, 0, st>>>(d_stage_off, d_stage_rows, d_stage_vals, d_kept, n, d_colptr_out, d_rows_out, d_vals_out);
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}

extern "C" int pg_mcl_components(const int64_t *d_colptr, const int32_t *d_rows, int64_t n, int32_t *d_root, pg_stream_t stream_) {
    int rc = check_csc(d_colptr, d_rows, n, "pg_mcl_components"); if (rc) return rc;
    if (!d_root && n > 0) return pg_fail(PG_ERR_INVALID, "pg_mcl_components: null output");
    if (n == 0) return PG_OK;
    cudaStream_t st = (cudaStream_t)stream_;
    k_mcl_uf_init<<<nblocks(n, 256), 256, 0, st>>>(d_root, n);
    k_mcl_union<<<nblocks(n, 256), 256, 0, st>>>(d_colptr, d_rows, n, d_root);
    k_mcl_flatten<<<nblocks(n, 256), 256, 0, st>>>(d_root, n);
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}
