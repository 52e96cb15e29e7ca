/*
 * cobweb_oracle.c -- CPU restatement of the reference's Cobweb hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product package may import, link or call this
 * file; only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs use it, and only as the checker or the timed CPU baseline.
 *
 * Every function cites the reference file:line it restates (paths relative to
 * /root/reference).  Pinned by tests/test_oracle_golden.py against fixtures produced by
 * running the reference itself (tests/golden/make_golden.py).
 *
 * Arithmetic contract (shared with the CUDA engine so that decisions are bit-identical):
 *   - every elementwise operation is a single IEEE-754 binary32 operation, in the order the
 *     reference's torch expressions evaluate them, with no FMA contraction
 *     (compile with -ffp-contract=off);
 *   - log() is co_logf() below (pure binary32 + integer ops, <1 ulp), not libm;
 *   - a reduction over the D attributes ("tensor.sum()") is a balanced pairwise sum in
 *     binary64 over groups of four consecutive terms, rounded once to binary32.  torch's own
 *     CPU sum is a vector-width-dependent cascade in binary32 and therefore not reproducible
 *     across machines; the pairwise-double sum is within a few binary32 ulps of it.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define CO_OP_BEST 0
#define CO_OP_NEW 1
#define CO_OP_MERGE 2
#define CO_OP_SPLIT 3
#define CO_OP_LEAF 4
#define CO_OP_FRINGE 5

typedef struct {
    float count;
    int parent;
    int nchild, capchild;
    int *child;
    int nsent;
    int alive;
} co_node;

typedef struct {
    int D;
    int use_info, use_kl, acuity_cutoff;
    int greedy; /* COBWEB_GREEDY_MODE (src/utils/constants.py:1) */
    float prior_var;
    int n, cap; /* node slots used / allocated */
    int root;
    co_node *nd;
    float *mean, *m2; /* [cap, D] */
    /* scratch rows */
    float *pm, *pv, *plv; /* parent-with-x  mean / var / log var */
    float *qm, *qv, *qlv; /* parent-as-is   mean / var / log var */
    float *t1, *t2, *t3, *t4;
    double *g;
    long n_score_calls; /* compute_score evaluations (SURVEY 8d work counter) */
    long n_rows_read;
    /* guided replay (co_ifit_guided): decisions recorded from the reference are applied, the
     * oracle's own choice and its margin to the applied one are reported */
    const signed char *g_op;
    const int *g_b1, *g_b2;
    long g_pos, g_n;
    long g_rank_disagree, g_op_disagree;
    float g_rank_margin, g_op_margin; /* largest margin among disagreements */
    float *g_pus;                     /* [g_n, 4] oracle pu of best/new/merge/split (NaN absent) */
} co_tree;

/* ------------------------------------------------------------------ scalar helpers */

static inline uint32_t f2u(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
static inline float u2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }

/* Natural logarithm in binary32 (argument reduction to [sqrt(1/2), sqrt(2)), s = f/(2+f),
 * degree-4 even polynomial in s^2; the classic fdlibm logf scheme).  Stands in for
 * torch.log on fp32 tensors (src/cobweb/CobwebTorchTree.py:350, CobwebTorchNode.py:102). */
float co_logf(float x) {
    const float ln2_hi = 6.9313812256e-01f, ln2_lo = 9.0580006145e-06f;
    const float Lg1 = 0.66666662693f, Lg2 = 0.40000972152f, Lg3 = 0.28498786688f, Lg4 = 0.24279078841f;
    uint32_t ix = f2u(x);
    int k = 0;
    if (ix < 0x00800000u || ix >= 0x7f800000u) {
        if ((ix << 1) == 0) return -INFINITY;
        if (ix >> 31) return NAN;
        if (ix >= 0x7f800000u) return x;
        x = x * 33554432.0f; /* subnormal: scale by 2^25 */
        k = -25;
        ix = f2u(x);
    }
    ix += 0x3f800000u - 0x3f3504f3u;
    k += (int)(ix >> 23) - 0x7f;
    ix = (ix & 0x007fffffu) + 0x3f3504f3u;
    x = u2f(ix);
    float f = x - 1.0f;
    float s = f / (2.0f + f);
    float z = s * s;
    float w = z * z;
    float t1 = w * (Lg2 + w * Lg4);
    float t2 = z * (Lg1 + w * Lg3);
    float R = t2 + t1;
    float hfsq = (0.5f * f) * f;
    float dk = (float)k;
    return ((((s * (hfsq + R)) + (dk * ln2_lo)) - hfsq) + f) + (dk * ln2_hi);
}

/* tensor.sum() over D attributes: see the arithmetic contract in the file header. */
static float co_sum(co_tree *t, const float *v) {
    int D = t->D, G = (D + 3) / 4, Gp = 1;
    while (Gp < G) Gp <<= 1;
    double *g = t->g;
    for (int j = 0; j < Gp; j++) {
        double s = 0.0;
        if (j < G) {
            int b = 4 * j;
            s = (double)v[b];
            if (b + 1 < D) s += (double)v[b + 1];
            if (b + 2 < D) s += (double)v[b + 2];
            if (b + 3 < D) s += (double)v[b + 3];
        }
        g[j] = s;
    }
    for (int w = Gp; w > 1; w >>= 1)
        for (int j = 0; j < w / 2; j++) g[j] = g[2 * j] + g[2 * j + 1];
    return (float)g[0];
}

float co_sum_public(int D, const float *v) {
    co_tree t;
    t.D = D;
    int G = (D + 3) / 4, Gp = 1;
    while (Gp < G) Gp <<= 1;
    t.g = (double *)malloc(sizeof(double) * Gp);
    float r = co_sum(&t, v);
    free(t.g);
    return r;
}

/* ------------------------------------------------------------------ tree storage */

co_tree *co_create(int D, float prior_var, int use_info, int use_kl, int acuity_cutoff) {
    co_tree *t = (co_tree *)calloc(1, sizeof(co_tree));
    t->D = D;
    t->prior_var = prior_var;
    t->use_info = use_info;
    t->use_kl = use_kl;
    t->acuity_cutoff = acuity_cutoff;
    t->cap = 1024;
    t->nd = (co_node *)calloc(t->cap, sizeof(co_node));
    t->mean = (float *)calloc((size_t)t->cap * D, sizeof(float));
    t->m2 = (float *)calloc((size_t)t->cap * D, sizeof(float));
    float **rows[] = {&t->pm, &t->pv, &t->plv, &t->qm, &t->qv, &t->qlv, &t->t1, &t->t2, &t->t3, &t->t4};
    for (unsigned i = 0; i < sizeof(rows) / sizeof(rows[0]); i++) *rows[i] = (float *)calloc(D, sizeof(float));
    int G = (D + 3) / 4, Gp = 1;
    while (Gp < G) Gp <<= 1;
    t->g = (double *)calloc(Gp, sizeof(double));
    /* CobwebTorchTree.clear(): an empty root (CobwebTorchTree.py:43-50) */
    t->n = 1;
    t->root = 0;
    t->nd[0].parent = -1;
    t->nd[0].alive = 1;
    return t;
}

void co_free(co_tree *t) {
    if (!t) return;
    for (int i = 0; i < t->n; i++) free(t->nd[i].child);
    free(t->nd); free(t->mean); free(t->m2);
    free(t->pm); free(t->pv); free(t->plv); free(t->qm); free(t->qv); free(t->qlv);
    free(t->t1); free(t->t2); free(t->t3); free(t->t4); free(t->g);
    free(t);
}

/* CobwebTorchNode.__init__ without otherNode (CobwebTorchNode.py:31-47): zero statistics */
static int new_node(co_tree *t) {
    if (t->n == t->cap) {
        int nc = t->cap * 2;
        t->nd = (co_node *)realloc(t->nd, sizeof(co_node) * nc);
        memset(t->nd + t->cap, 0, sizeof(co_node) * (nc - t->cap));
        t->mean = (float *)realloc(t->mean, sizeof(float) * (size_t)nc * t->D);
        t->m2 = (float *)realloc(t->m2, sizeof(float) * (size_t)nc * t->D);
        t->cap = nc;
    }
    int i = t->n++;
    memset(&t->nd[i], 0, sizeof(co_node));
    t->nd[i].parent = -1;
    t->nd[i].alive = 1;
    memset(t->mean + (size_t)i * t->D, 0, sizeof(float) * t->D);
    memset(t->m2 + (size_t)i * t->D, 0, sizeof(float) * t->D);
    return i;
}

static void child_append(co_tree *t, int p, int c) {
    co_node *n = &t->nd[p];
    if (n->nchild == n->capchild) {
        n->capchild = n->capchild ? 2 * n->capchild : 4;
        n->child = (int *)realloc(n->child, sizeof(int) * n->capchild);
    }
    n->child[n->nchild++] = c;
}

/* list.remove(): first occurrence, order of the rest preserved */
static void child_remove(co_tree *t, int p, int c) {
    co_node *n = &t->nd[p];
    int j = 0;
    while (j < n->nchild && n->child[j] != c) j++;
    for (; j + 1 < n->nchild; j++) n->child[j] = n->child[j + 1];
    n->nchild--;
}

#define MEAN(t, i) ((t)->mean + (size_t)(i) * (t)->D)
#define M2(t, i) ((t)->m2 + (size_t)(i) * (t)->D)

/* ------------------------------------------------------------------ node statistics */

/* CobwebTorchTree.compute_var (CobwebTorchTree.py:336-342) */
static inline float co_var(const co_tree *t, float m2, float count) {
    float v = m2 / count;
    if (t->acuity_cutoff) return v < t->prior_var ? t->prior_var : v; /* torch.clamp(min=) */
    return v + t->prior_var;
}

/* CobwebTorchNode.increment_counts (CobwebTorchNode.py:57-68) */
static void increment_counts(co_tree *t, int i, const float *x) {
    float *mu = MEAN(t, i), *m2 = M2(t, i);
    t->nd[i].count = t->nd[i].count + 1.0f;
    float n = t->nd[i].count;
    for (int d = 0; d < t->D; d++) {
        float delta = x[d] - mu[d];
        mu[d] = mu[d] + delta / n;
        m2[d] = m2[d] + delta * (x[d] - mu[d]);
    }
}

/* CobwebTorchNode.update_counts_from_node (CobwebTorchNode.py:70-85) */
static void update_counts_from_node(co_tree *t, int self, int other) {
    float *ms = MEAN(t, self), *qs = M2(t, self);
    const float *mo = MEAN(t, other), *qo = M2(t, other);
    float ns = t->nd[self].count, no = t->nd[other].count;
    float k = (ns * no) / (ns + no);
    float tot = ns + no;
    for (int d = 0; d < t->D; d++) {
        float delta = mo[d] - ms[d];
        qs[d] = (qs[d] + qo[d]) + (delta * delta) * k;
        ms[d] = (ns * ms[d] + no * mo[d]) / tot;
    }
    t->nd[self].count = ns + no;
}

/* mean_var (CobwebTorchNode.py:211): mean row pointer + variance into vout */
static void mean_var(co_tree *t, int i, float *vout) {
    const float *m2 = M2(t, i);
    float n = t->nd[i].count;
    for (int d = 0; d < t->D; d++) vout[d] = co_var(t, m2[d], n);
    t->n_rows_read++;
}

/* mean_var_insert (CobwebTorchNode.py:214-222) */
static void mean_var_insert(co_tree *t, int i, const float *x, float *mout, float *vout) {
    const float *mu = MEAN(t, i), *m2 = M2(t, i);
    float n = t->nd[i].count + 1.0f;
    for (int d = 0; d < t->D; d++) {
        float delta = x[d] - mu[d];
        float mean = mu[d] + delta / n;
        float q = m2[d] + delta * (x[d] - mean);
        mout[d] = mean;
        vout[d] = co_var(t, q, n);
    }
}

/* mean_var_merge (CobwebTorchNode.py:224-239) */
static void mean_var_merge(co_tree *t, int a, int b, const float *x, float *mout, float *vout) {
    const float *ma = MEAN(t, a), *qa = M2(t, a), *mb = MEAN(t, b), *qb = M2(t, b);
    float na = t->nd[a].count, nb = t->nd[b].count;
    float k = (na * nb) / (na + nb);
    float tot = na + nb;
    float cnt = tot + 1.0f;
    for (int d = 0; d < t->D; d++) {
        float delta = mb[d] - ma[d];
        float q = (qa[d] + qb[d]) + (delta * delta) * k;
        float mean = (na * ma[d] + nb * mb[d]) / tot;
        float dl = x[d] - mean;
        mean = mean + dl / cnt;
        q = q + dl * (x[d] - mean);
        mout[d] = mean;
        vout[d] = co_var(t, q, cnt);
    }
}

/* CobwebTorchTree.compute_score (CobwebTorchTree.py:344-364).  lv2 = log(var2) is passed in
 * because every caller scores many children against the same parent. */
static float compute_score(co_tree *t, const float *mu1, const float *var1, const float *mu2,
                           const float *var2, const float *lv2) {
    int D = t->D;
    float *a = t->t3, *b = t->t4;
    t->n_score_calls++;
    if (t->use_info) {
        for (int d = 0; d < D; d++) a[d] = lv2[d] - co_logf(var1[d]);
        if (!t->use_kl) return 0.5f * co_sum(t, a);
        for (int d = 0; d < D; d++) {
            float df = mu1[d] - mu2[d];
            b[d] = (var1[d] + df * df) / var2[d];
        }
        float score = co_sum(t, a);
        score = score + co_sum(t, b);
        score = score - (float)D;
        return score / 2.0f;
    }
    const float c = 2.0f * sqrtf(3.14159274101257324f); /* 2 * torch.sqrt(pi_tensor) */
    for (int d = 0; d < D; d++) {
        a[d] = 1.0f / (c * sqrtf(var1[d]));
        b[d] = 1.0f / (c * sqrtf(var2[d]));
    }
    float score = -co_sum(t, a);
    return score + co_sum(t, b);
}

float co_compute_score(co_tree *t, const float *mu1, const float *var1, const float *mu2, const float *var2) {
    float *lv = (float *)malloc(sizeof(float) * t->D);
    for (int d = 0; d < t->D; d++) lv[d] = co_logf(var2[d]);
    float r = compute_score(t, mu1, var1, mu2, var2, lv);
    free(lv);
    return r;
}

/* CobwebTorchNode.is_exact_match (CobwebTorchNode.py:652-666); torch.isclose defaults
 * rtol=1e-5, atol=1e-8: close = (a == b) | (isfinite(|a-b|) & (|a-b| <= atol + |rtol*b|)) */
static int isclose32(float a, float b) {
    if (a == b) return 1;
    float err = fabsf(a - b);
    float allowed = 1e-8f + fabsf(1e-5f * b);
    return isfinite(err) && err <= allowed;
}

static int is_exact_match(co_tree *t, int i, const float *x) {
    const float *mu = MEAN(t, i), *m2 = M2(t, i);
    float n = t->nd[i].count;
    for (int d = 0; d < t->D; d++)
        if (!isclose32(sqrtf(m2[d] / n), 0.0f)) return 0;
    for (int d = 0; d < t->D; d++)
        if (!isclose32(x[d], mu[d])) return 0;
    return 1;
}

/* ------------------------------------------------------------------ ifit */

typedef struct {
    int best1, best2;
    float best1_pu;
} two_best;

/* Everything get_best_operation needs at one internal node, in one pass.
 * two_best_children (CobwebTorchNode.py:374-420), pu_for_insert (:422-460),
 * pu_for_new_child (:482-515), pu_for_merge (:550-591), pu_for_split (:611-650),
 * get_best_operation (:287-372).  Returns the op code; *b1, *b2 receive best1/best2. */
static int best_operation(co_tree *t, int cur, const float *x, int *b1out, int *b2out) {
    co_node *P = &t->nd[cur];
    int C = P->nchild, D = t->D;
    float N = P->count;
    float N1 = N + 1.0f;
    float *s_as_is = (float *)malloc(sizeof(float) * C * 2);
    float *s_ins = s_as_is + C;

    /* parent after inserting x: mean_var_insert on self (:391, :445, :499, :573) */
    mean_var_insert(t, cur, x, t->pm, t->pv);
    for (int d = 0; d < D; d++) t->plv[d] = co_logf(t->pv[d]);

    int best1 = -1, best2 = -1;
    float g1 = 0, g2 = 0;
    for (int j = 0; j < C; j++) {
        int c = P->child[j];
        float nc = t->nd[c].count;
        mean_var_insert(t, c, x, t->t1, t->t2);
        s_ins[j] = compute_score(t, t->t1, t->t2, t->pm, t->pv, t->plv);
        float gain = ((nc + 1.0f) / N1) * s_ins[j];
        mean_var(t, c, t->t2);
        s_as_is[j] = compute_score(t, MEAN(t, c), t->t2, t->pm, t->pv, t->plv);
        gain = gain - (nc / N1) * s_as_is[j];
        /* sort(reverse=True) on (gain, count, random()) -- ties beyond count: first child wins */
        if (best1 < 0 || gain > g1 || (gain == g1 && nc > t->nd[P->child[best1]].count)) {
            best2 = best1; g2 = g1;
            best1 = j; g1 = gain;
        } else if (best2 < 0 || gain > g2 || (gain == g2 && nc > t->nd[P->child[best2]].count)) {
            best2 = j; g2 = gain;
        }
    }

    int guided = t->g_op && t->g_pos < t->g_n;
    if (guided) {
        int f1 = t->g_b1[t->g_pos], f2 = t->g_b2[t->g_pos];
        float *gains = (float *)malloc(sizeof(float) * C);
        for (int j = 0; j < C; j++) {
            float nc = t->nd[P->child[j]].count;
            gains[j] = ((nc + 1.0f) / N1) * s_ins[j] - (nc / N1) * s_as_is[j];
        }
        float m = 0.0f;
        if (f1 != best1) m = gains[best1] - gains[f1];
        else if (f2 != best2 && f2 >= 0 && best2 >= 0) m = gains[best2] - gains[f2];
        if (f1 != best1 || f2 != best2) {
            t->g_rank_disagree++;
            if (m > t->g_rank_margin) t->g_rank_margin = m;
        }
        best1 = f1;
        best2 = f2;
        free(gains);
    }

    /* pu_for_insert(best1) */
    float pu_best = 0.0f;
    for (int j = 0; j < C; j++) {
        float nc = t->nd[P->child[j]].count;
        if (j == best1) pu_best = pu_best + ((nc + 1.0f) / N1) * s_ins[j];
        else pu_best = pu_best + (nc / N1) * s_as_is[j];
    }
    pu_best = pu_best / (float)C;

    /* pu_for_new_child */
    float pu_new = 0.0f;
    for (int j = 0; j < C; j++) pu_new = pu_new + (t->nd[P->child[j]].count / N1) * s_as_is[j];
    for (int d = 0; d < D; d++) t->t2[d] = 0.0f + t->prior_var; /* mean_var_new (:204-209) */
    pu_new = pu_new + (1.0f / N1) * compute_score(t, x, t->t2, t->pm, t->pv, t->plv);
    pu_new = pu_new / (float)(C + 1);

    int op = CO_OP_BEST;
    float top = pu_best;
    float pus[4] = {pu_best, pu_new, NAN, NAN};
    if (pu_new > top) { top = pu_new; op = CO_OP_NEW; }

    if (C > 2 && best2 >= 0) {
        int c1 = P->child[best1], c2 = P->child[best2];
        float pu = 0.0f;
        for (int j = 0; j < C; j++) {
            if (j == best1 || j == best2) continue;
            pu = pu + (t->nd[P->child[j]].count / N1) * s_as_is[j];
        }
        float p = ((t->nd[c1].count + t->nd[c2].count) + 1.0f) / N1;
        mean_var_merge(t, c1, c2, x, t->t1, t->t2);
        pu = pu + p * compute_score(t, t->t1, t->t2, t->pm, t->pv, t->plv);
        pu = pu / (float)(C - 1);
        pus[2] = pu;
        if (pu > top) { top = pu; op = CO_OP_MERGE; }
    }

    int c1 = P->child[best1];
    int G = t->nd[c1].nchild;
    if (G > 0) {
        /* parent WITHOUT x (:630) */
        mean_var(t, cur, t->qv);
        for (int d = 0; d < D; d++) t->qlv[d] = co_logf(t->qv[d]);
        const float *qm = MEAN(t, cur);
        float pu = 0.0f;
        for (int j = 0; j < C; j++) {
            if (j == best1) continue;
            int c = P->child[j];
            mean_var(t, c, t->t2);
            pu = pu + (t->nd[c].count / N) * compute_score(t, MEAN(t, c), t->t2, qm, t->qv, t->qlv);
        }
        for (int j = 0; j < G; j++) {
            int g = t->nd[c1].child[j];
            mean_var(t, g, t->t2);
            pu = pu + (t->nd[g].count / N) * compute_score(t, MEAN(t, g), t->t2, qm, t->qv, t->qlv);
        }
        pu = pu / (float)(C - 1 + G);
        pus[3] = pu;
        if (pu > top) { top = pu; op = CO_OP_SPLIT; }
    }
    if (guided) {
        int fop = t->g_op[t->g_pos];
        if (t->g_pus) memcpy(t->g_pus + 4 * t->g_pos, pus, sizeof(pus));
        if (fop != op) {
            float m = top - pus[fop];
            t->g_op_disagree++;
            if (!(m <= t->g_op_margin)) t->g_op_margin = m; /* NaN (absent candidate) sticks */
            op = fop;
        }
        t->g_pos++;
    }
    *b1out = c1;
    *b2out = best2 >= 0 ? P->child[best2] : -1;
    free(s_as_is);
    return op;
}

/* CobwebTorchNode.create_new_child (CobwebTorchNode.py:462-480) */
static int create_new_child(co_tree *t, int p, const float *x) {
    int c = new_node(t);
    t->nd[c].parent = p;
    increment_counts(t, c, x);
    child_append(t, p, c);
    return c;
}

/* CobwebTorchTree.cobweb (CobwebTorchTree.py:143-233) for one instance. */
static int cobweb_one(co_tree *t, const float *x, signed char *trace, long *ntrace, long trace_cap) {
#define TR(code) do { if (trace && *ntrace < trace_cap) trace[*ntrace] = (signed char)(code); (*ntrace)++; } while (0)
    int cur = t->root;
    for (;;) {
        co_node *n = &t->nd[cur];
        if (n->nchild == 0 && (is_exact_match(t, cur, x) || n->count == 0.0f)) {
            increment_counts(t, cur, x);
            TR(CO_OP_LEAF);
            return cur;
        }
        if (n->nchild == 0) {
            /* fringe split (:190-204): copy-construct a parent from the leaf */
            int nw = new_node(t);
            int par = t->nd[cur].parent;
            t->nd[nw].parent = par;
            update_counts_from_node(t, nw, cur);
            t->nd[cur].parent = nw;
            child_append(t, nw, cur);
            if (par >= 0) {
                child_remove(t, par, cur);
                child_append(t, par, nw);
            } else {
                t->root = nw;
            }
            increment_counts(t, nw, x);
            TR(CO_OP_FRINGE);
            return create_new_child(t, nw, x);
        }
        int b1 = -1, b2 = -1;
        /* CobwebTorchTree.py:209-213: in greedy mode the action is "new" whatever two_best_children returns */
        int op = t->greedy ? CO_OP_NEW : best_operation(t, cur, x, &b1, &b2);
        TR(op);
        if (op == CO_OP_BEST) {
            increment_counts(t, cur, x);
            cur = b1;
        } else if (op == CO_OP_NEW) {
            increment_counts(t, cur, x);
            return create_new_child(t, cur, x);
        } else if (op == CO_OP_MERGE) {
            /* CobwebTorchNode.merge (CobwebTorchNode.py:517-548) */
            increment_counts(t, cur, x);
            int nw = new_node(t);
            t->nd[nw].parent = cur;
            update_counts_from_node(t, nw, b1);
            update_counts_from_node(t, nw, b2);
            t->nd[b1].parent = nw;
            t->nd[b2].parent = nw;
            child_append(t, nw, b1);
            child_append(t, nw, b2);
            child_remove(t, cur, b1);
            child_remove(t, cur, b2);
            child_append(t, cur, nw);
            cur = nw;
        } else {
            /* CobwebTorchNode.split (CobwebTorchNode.py:593-609); no increment, retry same node */
            child_remove(t, cur, b1);
            for (int j = 0; j < t->nd[b1].nchild; j++) {
                int g = t->nd[b1].child[j];
                t->nd[g].parent = cur;
                child_append(t, cur, g);
            }
            t->nd[b1].nchild = 0;
            t->nd[b1].alive = 0;
        }
    }
#undef TR
}

/* CobwebTorchTree.ifit per row (CobwebTorchTree.py:123) + the wrapper's bookkeeping
 * leaf.sentence_id.append(i) (CobwebWrapper.py:73-77) when tag_sentences != 0.
 * trace_off[i]..trace_off[i+1] delimit insert i's op codes in trace (may be NULL). */
long co_ifit(co_tree *t, const float *X, long n, int *leaf_out, signed char *trace, long *trace_off,
             long trace_cap, int tag_sentences) {
    long nt = 0;
    for (long i = 0; i < n; i++) {
        if (trace_off) trace_off[i] = nt;
        int leaf = cobweb_one(t, X + (size_t)i * t->D, trace, &nt, trace_cap);
        if (tag_sentences) t->nd[leaf].nsent++;
        if (leaf_out) leaf_out[i] = leaf;
    }
    if (trace_off) trace_off[n] = nt;
    return nt;
}

/* co_ifit with the internal-node decisions (op, best1, best2 as child-list positions) taken
 * from a recorded reference run instead of the oracle's own arg-max.  The oracle still
 * evaluates every candidate; stats[0..3] = #ranking disagreements, #op disagreements, largest
 * gain margin and largest pu margin among the disagreements.  Used to show that wherever the
 * oracle would have chosen differently from the reference, the two candidates were within
 * fp32 summation noise of each other. */
long co_ifit_guided(co_tree *t, const float *X, long n, int *leaf_out, const signed char *g_op, const int *g_b1,
                    const int *g_b2, long g_n, float *pus_out, double *stats, int tag_sentences) {
    t->g_op = g_op; t->g_b1 = g_b1; t->g_b2 = g_b2; t->g_n = g_n; t->g_pos = 0;
    t->g_rank_disagree = t->g_op_disagree = 0;
    t->g_rank_margin = t->g_op_margin = 0.0f;
    t->g_pus = pus_out;
    co_ifit(t, X, n, leaf_out, NULL, NULL, 0, tag_sentences);
    stats[0] = (double)t->g_rank_disagree;
    stats[1] = (double)t->g_op_disagree;
    stats[2] = t->g_rank_margin;
    stats[3] = t->g_op_margin;
    long used = t->g_pos;
    t->g_op = NULL;
    return used;
}

/* ------------------------------------------------------------------ export / import */

int co_num_slots(const co_tree *t) { return t->n; }
int co_root(const co_tree *t) { return t->root; }
long co_score_calls(const co_tree *t) { return t->n_score_calls; }

int co_num_nodes(const co_tree *t) {
    int c = 0;
    for (int i = 0; i < t->n; i++) c += t->nd[i].alive;
    return c;
}

/* BFS order, children in list order: the numbering build_prediction_index uses
 * (CobwebWrapper.py:107-132).  order[b] = node slot; returns #nodes. */
int co_bfs(const co_tree *t, int *order, int *parent_bfs, float *count, int *nchild, int *nsent, int *depth) {
    int *pos = (int *)malloc(sizeof(int) * t->n);
    int head = 0, tail = 0;
    order[tail] = t->root;
    parent_bfs[tail] = -1;
    if (depth) depth[tail] = 0;
    tail++;
    while (head < tail) {
        int i = order[head];
        pos[i] = head;
        const co_node *n = &t->nd[i];
        if (count) count[head] = n->count;
        if (nchild) nchild[head] = n->nchild;
        if (nsent) nsent[head] = n->nsent;
        for (int j = 0; j < n->nchild; j++) {
            order[tail] = n->child[j];
            parent_bfs[tail] = head;
            if (depth) depth[tail] = depth[head] + 1;
            tail++;
        }
        head++;
    }
    free(pos);
    return tail;
}

void co_get_rows(const co_tree *t, const int *slots, int n, float *mean_out, float *m2_out) {
    for (int i = 0; i < n; i++) {
        if (mean_out) memcpy(mean_out + (size_t)i * t->D, MEAN(t, slots[i]), sizeof(float) * t->D);
        if (m2_out) memcpy(m2_out + (size_t)i * t->D, M2(t, slots[i]), sizeof(float) * t->D);
    }
}

/* Replace the tree by nodes given in an order where parent[i] < i and siblings appear in
 * child-list order (e.g. a BFS or pre-order dump of an engine-built store). */
void co_load(co_tree *t, int n, const int *parent, const float *count, const int *nsent, const float *mean,
             const float *m2) {
    for (int i = 0; i < t->n; i++) { free(t->nd[i].child); t->nd[i].child = NULL; }
    t->n = 0;
    for (int i = 0; i < n; i++) {
        int s = new_node(t);
        t->nd[s].count = count[i];
        t->nd[s].parent = parent[i];
        t->nd[s].nsent = nsent ? nsent[i] : 0;
        memcpy(MEAN(t, s), mean + (size_t)i * t->D, sizeof(float) * t->D);
        memcpy(M2(t, s), m2 + (size_t)i * t->D, sizeof(float) * t->D);
        if (parent[i] >= 0) child_append(t, parent[i], s);
    }
    t->root = 0;
}

/* ------------------------------------------------------------------ best-first categorize */

/* CobwebTorchNode.log_prob (CobwebTorchNode.py:100-104) */
static float log_prob(co_tree *t, int i, const float *x, float *tmp) {
    const float *mu = MEAN(t, i), *m2 = M2(t, i);
    float n = t->nd[i].count;
    const float half_log_2pi = 0.5f * 1.83787703514099121f; /* 0.5 * torch.log(2 * pi_tensor) */
    for (int d = 0; d < t->D; d++) {
        float var = co_var(t, m2[d], n);
        float df = x[d] - mu[d];
        tmp[d] = (0.5f * co_logf(var) + half_log_2pi) + (0.5f * (df * df)) / var;
    }
    t->n_rows_read++;
    return -co_sum(t, tmp);
}

float co_log_prob(co_tree *t, int node, const float *x) {
    float *tmp = (float *)malloc(sizeof(float) * t->D);
    float r = log_prob(t, node, x, tmp);
    free(tmp);
    return r;
}

typedef struct {
    float neg, par;
    long seq;
    int node;
} hitem;

static inline int hless(const hitem *a, const hitem *b) {
    if (a->neg != b->neg) return a->neg < b->neg;
    if (a->par != b->par) return a->par < b->par;
    return a->seq < b->seq;
}

/* CobwebTorchTree._cobweb_categorize (CobwebTorchTree.py:235-289) for nq queries.
 * out_leaves[q*k + j] = j-th retrieved node slot (-1 past out_nfound[q]); when k == 0
 * ("retrieve_k=None") only out_best is meaningful: best-scoring popped node, or the last
 * popped node if !use_best.  heap ties (never seen on continuous data) pop in push order. */
void co_categorize(co_tree *t, const float *Q, long nq, int k, long max_nodes, int greedy, int use_best,
                   int *out_leaves, int *out_nfound, int *out_best, long *out_lp_calls) {
    float *tmp = (float *)malloc(sizeof(float) * t->D);
    long hcap = 1024;
    hitem *h = (hitem *)malloc(sizeof(hitem) * hcap);
    for (long q = 0; q < nq; q++) {
        const float *x = Q + (size_t)q * t->D;
        long hn = 0, seq = 0, visited = 0, calls = 0;
        int found = 0, best = t->root, curr = t->root;
        float best_score = -INFINITY;
        h[hn++] = (hitem){-log_prob(t, t->root, x, tmp), 0.0f, seq++, t->root};
        calls++;
        while (hn > 0) {
            hitem top = h[0];
            h[0] = h[--hn];
            for (long i = 0;;) { /* sift down */
                long l = 2 * i + 1, r = l + 1, m = i;
                if (l < hn && hless(&h[l], &h[m])) m = l;
                if (r < hn && hless(&h[r], &h[m])) m = r;
                if (m == i) break;
                hitem sw = h[i]; h[i] = h[m]; h[m] = sw;
                i = m;
            }
            curr = top.node;
            float score = -top.neg;
            visited++;
            if (score > best_score) { best = curr; best_score = score; }
            if (greedy) hn = 0;
            if (visited >= max_nodes) break;
            if (t->nd[curr].nsent > 0) {
                if (k > 0 && found < k) out_leaves[q * k + found] = curr;
                found++;
            }
            if (k > 0 && found == k) break;
            const co_node *n = &t->nd[curr];
            for (int j = 0; j < n->nchild; j++) {
                if (hn == hcap) { hcap *= 2; h = (hitem *)realloc(h, sizeof(hitem) * hcap); }
                hitem it = {-log_prob(t, n->child[j], x, tmp), score, seq++, n->child[j]};
                calls++;
                long i = hn++;
                h[i] = it;
                while (i > 0) { /* sift up */
                    long p = (i - 1) / 2;
                    if (!hless(&h[i], &h[p])) break;
                    hitem sw = h[i]; h[i] = h[p]; h[p] = sw;
                    i = p;
                }
            }
        }
        if (k > 0) {
            for (int j = found < k ? found : k; j < k; j++) out_leaves[q * k + j] = -1;
            if (out_nfound) out_nfound[q] = found < k ? found : k;
        }
        if (out_best) out_best[q] = use_best ? best : curr;
        if (out_lp_calls) out_lp_calls[q] = calls;
    }
    free(h);
    free(tmp);
}

/* ------------------------------------------------------------------ dense ("fast") predict */

/* Node matrices of build_prediction_index (CobwebWrapper.py:186-203): var = compute_var or
 * prior for empty nodes; plus sum_d log var, the query-independent half of the score. */
void co_index_stats(co_tree *t, const int *order, int n, float *means, float *vars, float *sumlog) {
    float *lv = (float *)malloc(sizeof(float) * t->D);
    for (int b = 0; b < n; b++) {
        int i = order[b];
        const float *m2 = M2(t, i);
        float cnt = t->nd[i].count;
        float *v = vars + (size_t)b * t->D;
        memcpy(means + (size_t)b * t->D, MEAN(t, i), sizeof(float) * t->D);
        for (int d = 0; d < t->D; d++) {
            v[d] = cnt > 0.0f ? co_var(t, m2[d], cnt) : t->prior_var;
            lv[d] = co_logf(v[d]);
        }
        sumlog[b] = co_sum(t, lv);
    }
    free(lv);
}

/* The sparse path product leaf = P @ node_scores (CobwebWrapper.py:241, 290): torch.sparse.mm
 * on CPU accumulates each row's non-zeros in column order (root first) with a fused
 * multiply-add in binary32 -- verified bit-for-bit against the reference's own node scores in
 * tests/test_oracle_golden.py.  path_idx[l*maxlen + j] = node index or -1; path_w = w/len. */
void co_leaf_scores(long nq, int nn, const float *node_scores, long nl, int maxlen, const int *path_idx,
                    const float *path_w, float *leaf_scores) {
#pragma omp parallel for schedule(static)
    for (long q = 0; q < nq; q++) {
        const float *s = node_scores + (size_t)q * nn;
        for (long l = 0; l < nl; l++) {
            float acc = 0.0f;
            for (int j = 0; j < maxlen; j++) {
                int b = path_idx[l * maxlen + j];
                if (b < 0) break;
                acc = fmaf(path_w[l * maxlen + j], s[b], acc);
            }
            leaf_scores[(size_t)q * nl + l] = acc;
        }
    }
}

/* cobweb_predict_indexed / cobweb_rank_scores node term (CobwebWrapper.py:230-236, 283-287):
 * s_n = -0.5 * (sum_d log V + sum_d (x - M)^2 / V) for every node, then the sparse path
 * product (:241) via co_leaf_scores. */
void co_dense_scores(int D, long nq, const float *Q, int nn, const float *means, const float *vars,
                     const float *sumlog, long nl, int maxlen, const int *path_idx, const float *path_w,
                     float *node_scores, float *leaf_scores) {
#pragma omp parallel
    {
        co_tree tt;
        tt.D = D;
        int G = (D + 3) / 4, Gp = 1;
        while (Gp < G) Gp <<= 1;
        tt.g = (double *)malloc(sizeof(double) * Gp);
        float *tmp = (float *)malloc(sizeof(float) * D);
#pragma omp for collapse(2) schedule(static)
        for (long q = 0; q < nq; q++) {
            for (int b = 0; b < nn; b++) {
                const float *x = Q + (size_t)q * D, *m = means + (size_t)b * D, *v = vars + (size_t)b * D;
                for (int d = 0; d < D; d++) {
                    float df = x[d] - m[d];
                    tmp[d] = (df * df) / v[d];
                }
                node_scores[(size_t)q * nn + b] = -0.5f * (sumlog[b] + co_sum(&tt, tmp));
            }
        }
        free(tmp);
        free(tt.g);
    }
    if (leaf_scores) co_leaf_scores(nq, nn, node_scores, nl, maxlen, path_idx, path_w, leaf_scores);
}

/* Operands of the engine's FP32 form (dense_operands in the CUDA sources): r = 1 / sqrt(var), mb = -(mean * r),
 * each a single binary32 operation, so that (x - mean)^2 / var = (x * r + mb)^2. */
void co_fp32_operands(int D, int nn, const float *means, const float *vars, float *r, float *mb) {
    for (size_t i = 0; i < (size_t)nn * D; i++) {
        r[i] = 1.0f / sqrtf(vars[i]);
        mb[i] = -(means[i] * r[i]);
    }
}

/* out[i] = fmaf(a[i], b[i], c[i]): the fused multiply-add co_fp32_node_scores uses, exposed so the tests can check it
 * against exact rational arithmetic. */
void co_fmaf_array(long n, const float *a, const float *b, const float *c, float *out) {
    for (long i = 0; i < n; i++) out[i] = fmaf(a[i], b[i], c[i]);
}

/* Node scores of the engine's FP32 form bit for bit (dense_score_kernel / small_scores_kernel): per (query, node) one
 * chain over d ascending, u = fma(x, r, mb); acc = fma(u, u, acc) from acc = +0, then -0.5 * (sumlog + acc).  libm
 * fmaf is correctly rounded, as the device's FFMA is. */
void co_fp32_node_scores(int D, long nq, const float *Q, int nn, const float *means, const float *vars,
                         const float *sumlog, float *node_scores) {
    float *r = (float *)malloc(sizeof(float) * (size_t)nn * D);
    float *mb = (float *)malloc(sizeof(float) * (size_t)nn * D);
    co_fp32_operands(D, nn, means, vars, r, mb);
#pragma omp parallel for collapse(2) schedule(static)
    for (long q = 0; q < nq; q++) {
        for (int b = 0; b < nn; b++) {
            const float *x = Q + (size_t)q * D, *rb = r + (size_t)b * D, *mbb = mb + (size_t)b * D;
            float acc = 0.0f;
            for (int d = 0; d < D; d++) {
                const float u = fmaf(x[d], rb[d], mbb[d]);
                acc = fmaf(u, u, acc);
            }
            node_scores[(size_t)q * nn + b] = -0.5f * (sumlog[b] + acc);
        }
    }
    free(r);
    free(mb);
}

/* Throughput-oriented variant of the same scores for the CPU baseline (bench.py): plain
 * binary32 accumulation, vectorisable, one pass per query over the node matrices like the
 * reference's broadcast expression.  Not used for parity. */
void co_dense_scores_fast(int D, long nq, const float *Q, int nn, const float *means, const float *vars,
                          const float *sumlog, float *node_scores) {
#pragma omp parallel for collapse(2) schedule(static)
    for (long q = 0; q < nq; q++) {
        for (int b = 0; b < nn; b++) {
            const float *x = Q + (size_t)q * D, *m = means + (size_t)b * D, *v = vars + (size_t)b * D;
            float acc = 0.0f;
#pragma omp simd reduction(+ : acc)
            for (int d = 0; d < D; d++) {
                float df = x[d] - m[d];
                acc += (df * df) / v[d];
            }
            node_scores[(size_t)q * nn + b] = -0.5f * (sumlog[b] + acc);
        }
    }
}

/* top-k of a score row, descending, ties -> lower index (torch.topk, CobwebWrapper.py:256) */
void co_topk(const float *scores, long n, int k, int *idx_out, float *val_out) {
    for (int j = 0; j < k; j++) { idx_out[j] = -1; val_out[j] = -INFINITY; }
    for (long i = 0; i < n; i++) {
        float s = scores[i];
        if (idx_out[k - 1] >= 0 && !(s > val_out[k - 1])) continue;
        int j = k - 1;
        while (j > 0 && (idx_out[j - 1] < 0 || s > val_out[j - 1])) {
            idx_out[j] = idx_out[j - 1];
            val_out[j] = val_out[j - 1];
            j--;
        }
        idx_out[j] = (int)i;
        val_out[j] = s;
    }
}

/* Threads of the dense baseline loops (bench.py sets them explicitly: torchrun exports OMP_NUM_THREADS=1).
 * Returns the thread count in effect (1 without OpenMP). */
int co_set_threads(int n) {
#ifdef _OPENMP
    if (n > 0) omp_set_num_threads(n);
    return omp_get_max_threads();
#else
    (void)n;
    return 1;
#endif
}

/* COBWEB_GREEDY_MODE switch of the reference (a module constant there, src/utils/constants.py:1). */
void co_set_greedy(co_tree *t, int greedy) { t->greedy = greedy; }
