/* mcl.c - CPU oracle of the Markov clustering stage (pangenome_b200/csrc/mcl.cu) - TEST INFRASTRUCTURE ONLY.
 *
 * A plain restatement of the definition in include/pgdbg.h / DESIGN.md §3 with the same float32 operations in
 * the same order: build with `gcc -O2 -ffp-contract=off` so that no a*b+c becomes an FMA.
 *
 *   A     : edges with w >= max(min_weight, 1), symmetrised, duplicates merged by max; A[j,j] = max_i A[i,j]
 *           (1 for a node with no edge); M = column-normalise(A)
 *   step  : M <- normalise(inflate_r(prune(M.M)))
 *   prune : keep the min(S, #entries >= theta) largest entries (value descending, row ascending); a column
 *           with no entry >= theta keeps its largest entry
 *   chaos : max over columns of max(0, max_i M[i,j] / sum_i M[i,j]^2 - 1), after normalisation
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define THETA 1e-4f
#define SEL_S 1024

typedef struct {
    int64_t n, nnz;
    int64_t *cp;
    int32_t *rows;
    float *vals;
    float chaos;
    int64_t products;
} mclo;

typedef struct { int64_t col; int32_t row; float v; } ent;

static int cmp_colrow(const void *a, const void *b) {
    const ent *x = a, *y = b;
    if (x->col != y->col) return x->col < y->col ? -1 : 1;
    return x->row < y->row ? -1 : x->row > y->row;
}
static int cmp_valdesc_rowasc(const void *a, const void *b) {
    const ent *x = a, *y = b;
    if (x->v != y->v) return x->v > y->v ? -1 : 1;
    return x->row < y->row ? -1 : x->row > y->row;
}
static int cmp_row(const void *a, const void *b) {
    const ent *x = a, *y = b;
    return x->row < y->row ? -1 : x->row > y->row;
}

/* divide by the sum (ascending row), return chaos */
static float column_finish(float *v, int64_t K) {
    if (K == 0) return 0.f;
    float sum = 0.f, mx = 0.f, sq = 0.f;
    for (int64_t e = 0; e < K; e++) sum = sum + v[e];
    for (int64_t e = 0; e < K; e++) {
        float x = v[e] / sum;
        v[e] = x;
        mx = fmaxf(mx, x);
        sq = sq + x * x;
    }
    return mx / sq - 1.f;
}

static float normalise_all(mclo *m) {
    float chaos = 0.f;
    for (int64_t j = 0; j < m->n; j++) {
        float c = column_finish(m->vals + m->cp[j], m->cp[j + 1] - m->cp[j]);
        if (c > chaos) chaos = c;
    }
    return chaos;
}

void *mclo_new(int64_t n, int64_t m_edges, const int64_t *src, const int64_t *dst, const int64_t *w, int64_t min_weight) {
    mclo *m = calloc(1, sizeof(mclo));
    m->n = n;
    ent *e = malloc(sizeof(ent) * (size_t)(2 * m_edges + n + 1));
    float *colmax = calloc((size_t)n + 1, sizeof(float));
    int64_t ne = 0;
    for (int64_t t = 0; t < m_edges; t++) {
        if (w[t] < min_weight || w[t] < 1) continue;
        float v = (float)w[t];
        e[ne++] = (ent){dst[t], (int32_t)src[t], v};
        e[ne++] = (ent){src[t], (int32_t)dst[t], v};
        if (v > colmax[src[t]]) colmax[src[t]] = v;
        if (v > colmax[dst[t]]) colmax[dst[t]] = v;
    }
    for (int64_t j = 0; j < n; j++) e[ne++] = (ent){j, (int32_t)j, colmax[j] > 0.f ? colmax[j] : 1.f};
    qsort(e, (size_t)ne, sizeof(ent), cmp_colrow);
    m->cp = calloc((size_t)n + 1, sizeof(int64_t));
    m->rows = malloc(sizeof(int32_t) * (size_t)(ne + 1));
    m->vals = malloc(sizeof(float) * (size_t)(ne + 1));
    int64_t nnz = 0;
    for (int64_t t = 0; t < ne; t++) {
        if (nnz && e[t].col == e[t - 1].col && e[t].row == e[t - 1].row) {
            if (e[t].v > m->vals[nnz - 1]) m->vals[nnz - 1] = e[t].v;
            continue;
        }
        m->rows[nnz] = e[t].row;
        m->vals[nnz] = e[t].v;
        m->cp[e[t].col + 1]++;
        nnz++;
    }
    for (int64_t j = 0; j < n; j++) m->cp[j + 1] += m->cp[j];
    m->nnz = nnz;
    free(e);
    free(colmax);
    m->chaos = normalise_all(m);
    return m;
}

static float inflate(float x, double r, int whole, int half) {
    if (!whole) return powf(x, (float)r);
    float p = x;
    for (int i = 1; i < whole; i++) p = p * x;
    return half ? p * sqrtf(x) : p;
}

void mclo_iterate(void *h, double r) {
    mclo *m = h;
    int64_t n = m->n;
    float rf = (float)r, twice = rf * 2.f;
    int whole = twice == floorf(twice) ? (int)floorf(rf) : 0;
    int half = whole && twice != 2.f * floorf(rf);
    float *acc = calloc((size_t)n + 1, sizeof(float));
    char *mark = calloc((size_t)n + 1, 1);
    ent *list = malloc(sizeof(ent) * ((size_t)n + 1));
    int64_t *cp = calloc((size_t)n + 1, sizeof(int64_t));
    int64_t cap = m->nnz + 16, nnz = 0;
    int32_t *rows = malloc(sizeof(int32_t) * (size_t)cap);
    float *vals = malloc(sizeof(float) * (size_t)cap);
    float chaos = 0.f;
    m->products = 0;
    for (int64_t j = 0; j < n; j++) {
        int64_t cnt = 0;
        for (int64_t p = m->cp[j]; p < m->cp[j + 1]; p++) {
            int32_t k = m->rows[p];
            float mkj = m->vals[p];
            m->products += m->cp[k + 1] - m->cp[k];
            for (int64_t q = m->cp[k]; q < m->cp[k + 1]; q++) {
                int32_t i = m->rows[q];
                if (!mark[i]) { mark[i] = 1; acc[i] = 0.f; list[cnt++].row = i; }
                acc[i] = acc[i] + m->vals[q] * mkj;
            }
        }
        int64_t c_theta = 0;
        for (int64_t t = 0; t < cnt; t++) {
            list[t].v = acc[list[t].row];
            mark[list[t].row] = 0;
            c_theta += list[t].v >= THETA;
        }
        int64_t want = c_theta == 0 ? 1 : (c_theta < SEL_S ? c_theta : SEL_S);
        if (want > cnt) want = cnt;
        if (want < cnt) qsort(list, (size_t)cnt, sizeof(ent), cmp_valdesc_rowasc);
        qsort(list, (size_t)want, sizeof(ent), cmp_row);
        if (nnz + want > cap) {
            cap = 2 * (nnz + want);
            rows = realloc(rows, sizeof(int32_t) * (size_t)cap);
            vals = realloc(vals, sizeof(float) * (size_t)cap);
        }
        for (int64_t t = 0; t < want; t++) { rows[nnz + t] = list[t].row; vals[nnz + t] = inflate(list[t].v, r, whole, half); }
        float c = column_finish(vals + nnz, want);
        if (c > chaos) chaos = c;
        nnz += want;
        cp[j + 1] = nnz;
    }
    free(acc); free(mark); free(list);
    free(m->cp); free(m->rows); free(m->vals);
    m->cp = cp; m->rows = rows; m->vals = vals; m->nnz = nnz; m->chaos = chaos;
}

static int32_t find(int32_t *p, int32_t x) {
    while (p[x] != x) { p[x] = p[p[x]]; x = p[x]; }
    return x;
}

/* root = smallest node index of the component of the undirected graph of the stored entries */
void mclo_components(void *h, int32_t *root) {
    mclo *m = h;
    for (int64_t i = 0; i < m->n; i++) root[i] = (int32_t)i;
    for (int64_t j = 0; j < m->n; j++)
        for (int64_t q = m->cp[j]; q < m->cp[j + 1]; q++) {
            int32_t a = find(root, (int32_t)j), b = find(root, m->rows[q]);
            if (a != b) { if (a < b) root[b] = a; else root[a] = b; }
        }
    for (int64_t i = 0; i < m->n; i++) root[i] = find(root, (int32_t)i);
}

int64_t mclo_n(void *h) { return ((mclo *)h)->n; }
int64_t mclo_nnz(void *h) { return ((mclo *)h)->nnz; }
int64_t mclo_products(void *h) { return ((mclo *)h)->products; }
float mclo_chaos(void *h) { return ((mclo *)h)->chaos; }
int64_t *mclo_colptr(void *h) { return ((mclo *)h)->cp; }
int32_t *mclo_rows(void *h) { return ((mclo *)h)->rows; }
float *mclo_vals(void *h) { return ((mclo *)h)->vals; }
void mclo_free(void *h) {
    mclo *m = h;
    if (!m) return;
    free(m->cp); free(m->rows); free(m->vals); free(m);
}
