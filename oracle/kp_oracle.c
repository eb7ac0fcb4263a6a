/*
 * kp_oracle.c — CPU restatement of kmerPaPa's optimal pattern-partition DP.
 *
 * THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may load it.  The product path
 * (kmerpapa_b200/) never links, imports or calls anything in oracle/.
 *
 * What it restates (paths relative to the reference checkout, /root/reference):
 *   src/kmerpapa/pattern_utils.py:5-19     IUPAC letter -> nucleotide list ("code")
 *   src/kmerpapa/pattern_utils.py:48-57    two-way splits per letter ("complements") and their order
 *   src/kmerpapa/pattern_utils.py:86-100   digit order per general letter ("perm_code")
 *   src/kmerpapa/pattern_utils.py:237-257  dense mixed-radix pattern index (position 0 least significant)
 *   src/kmerpapa/algorithms/bottum_up_array_w_numba.py:26-29   level-0 score (scipy xlogy/xlog1py)
 *   src/kmerpapa/algorithms/bottum_up_array_w_numba.py:31-64   handle_pattern (single DP)
 *   src/kmerpapa/algorithms/bottum_up_array_w_numba.py:17-24   backtrack (left child first)
 *   src/kmerpapa/algorithms/bottum_up_array_penalty_plus_pseudo_CV.py:15-20  level-0 train/test
 *   src/kmerpapa/algorithms/bottum_up_array_penalty_plus_pseudo_CV.py:26-78  handle_pattern (CV, one fold)
 *
 * Third-party arithmetic the reference leans on and that is NOT under /root/reference:
 *   - glibc 2.39 log() (numba lowers math.log/np.log to the C library): restated below as
 *     kpo_log(), the exact IEEE operation sequence of __log_fma with glibc's own coefficient
 *     table (oracle/kpo_log_data.h, extracted by tools/extract_glibc_log_data.py).
 *     tests/test_oracle.py pins kpo_log() bit-for-bit against the system log().
 *   - scipy 1.18.1 special.xlogy / xlog1py (level 0 only): x*log(y) and x*cephes_log1p(y);
 *     cephes log1p restated below, pinned bit-for-bit against scipy in tests/test_oracle.py.
 *
 * Parity status: PINNED.  The reference has no golden vectors for this path (its tests only
 * cover index bijections and fold sums), so the oracle is pinned against outputs of the
 * unmodified reference itself, generated in the build container by tests/golden/make_golden.py
 * (full score/count/backtrack tables on small general patterns, and the CLI outputs of
 * BASELINE configs 1 and 2).
 *
 * Order of evaluation: the reference walks patterns level by level; a pattern only reads
 * patterns with a smaller dense index (every split lowers one digit), so any topological order
 * gives identical tables.  Here: blocks of the index space (high digits fixed) are processed
 * by block level, blocks of one level in parallel (OpenMP), ascending index inside a block.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "kpo_log_data.h"

#define KPO_MAXK 32

/* ------------------------------------------------------------------------------------------- */
/* glibc log(), FMA variant, restated                                                           */
/* ------------------------------------------------------------------------------------------- */
static const double kLn2hi = KP_LOG_LN2HI, kLn2lo = KP_LOG_LN2LO;
static const double kA[5] = KP_LOG_A_INIT;
static const double kB[11] = KP_LOG_B_INIT;
static const double kTab[256] = KP_LOG_TAB_INIT;

static inline uint64_t as_u64(double x) { uint64_t u; memcpy(&u, &x, 8); return u; }
static inline double as_f64(uint64_t u) { double x; memcpy(&x, &u, 8); return x; }
#define FMA(a, b, c) __builtin_fma((a), (b), (c))

double kpo_log(double x)
{
    uint64_t ix = as_u64(x);
    uint32_t top = (uint32_t)(ix >> 48);
    if (ix - 0x3fee000000000000ULL < 0x0003090000000000ULL) {
        /* 1 - 2^-4 <= x < 1 + 0x1.09p-4: polynomial in r = x - 1 with a split-hi/lo head */
        if (ix == 0x3ff0000000000000ULL) return 0.0;
        double r = x - 1.0;
        double r2 = r * r;
        double r3 = r * r2;
        double t2 = FMA(r, kB[2], kB[1]);
        double t3 = FMA(r, kB[5], kB[4]);
        double t5 = FMA(r, kB[8], kB[7]);
        t2 = FMA(r2, kB[3], t2);
        t3 = FMA(r2, kB[6], t3);
        double t1 = FMA(r2, kB[9], t5);
        t1 = FMA(r3, kB[10], t1);
        t1 = FMA(t1, r3, t3);
        t1 = FMA(t1, r3, t2);
        double rw = FMA(r, 0x1p27, r);
        double rhi = FMA(-0x1p27, r, rw);
        double rlo = r - rhi;
        double rhi2 = rhi * rhi;
        double hi = FMA(rhi2, kB[0], r);
        double t8 = r - hi;
        double rr = r + rhi;
        double lo = FMA(rhi2, kB[0], t8);
        double t = kB[0] * rlo;
        lo = FMA(t, rr, lo);
        double y = FMA(t1, r3, lo);
        return hi + y;
    }
    if ((uint32_t)(top - 0x10) > 0x7fdfu) {
        if (ix * 2 == 0) return -INFINITY;
        if (ix == 0x7ff0000000000000ULL) return x;
        if ((top & 0x8000u) || (top & 0x7ff0u) == 0x7ff0u) return NAN;
        ix = as_u64(x * 0x1p52);
        ix -= 52ULL << 52;
    }
    uint64_t tmp = ix - 0x3fe6000000000000ULL;
    int i = (int)((tmp >> 45) & 127);
    int64_t k = (int64_t)tmp >> 52;
    uint64_t iz = ix - (tmp & 0xfff0000000000000ULL);
    double invc = kTab[2 * i], logc = kTab[2 * i + 1];
    double z = as_f64(iz);
    double kd = (double)k;
    double w = FMA(kd, kLn2hi, logc);
    double r = FMA(z, invc, -1.0);
    double q5 = FMA(r, kA[2], kA[1]);
    double hi = r + w;
    double r2 = r * r;
    double lo = w - hi;
    lo = lo + r;
    lo = FMA(kd, kLn2lo, lo);
    double r3 = r * r2;
    double q1 = FMA(r, kA[4], kA[3]);
    lo = FMA(r2, kA[0], lo);
    q1 = FMA(q1, r2, q5);
    double y = FMA(r3, q1, lo);
    return y + hi;
}

/* cephes log1p as shipped in scipy.special (xsf/cephes/unity.h) — used by xlog1py at level 0 */
static const double kLP[7] = {
    4.5270000862445199635215E-5, 4.9854102823193375972212E-1, 6.5787325942061044846969E0,
    2.9911919328553073277375E1,  6.0949667980987787057556E1,  5.7112963590585538103336E1,
    2.0039553499201281259648E1,
};
static const double kLQ[6] = {
    1.5062909083469192043167E1, 8.3047565967967209469434E1, 2.2176239823732856465394E2,
    3.0909872225312059774938E2, 2.1642788614495947685003E2, 6.0118660497603843919306E1,
};

double kpo_log1p(double x)
{
    double z = 1.0 + x;
    if (z < 0.70710678118654752440 || z > 1.41421356237309504880) return kpo_log(z);
    z = x * x;
    double num = kLP[0];
    for (int i = 1; i <= 6; i++) num = num * x + kLP[i];
    double den = x + kLQ[0];
    for (int i = 1; i < 6; i++) den = den * x + kLQ[i];
    z = -0.5 * z + x * (z * num / den);
    return x + z;
}

double kpo_xlogy(double x, double y) { return (x == 0.0 && !isnan(y)) ? 0.0 : x * kpo_log(y); }
double kpo_xlog1py(double x, double y) { return (x == 0.0 && !isnan(y)) ? 0.0 : x * kpo_log1p(y); }

/* number of inputs where the restated log differs (bitwise) from the C library's log() */
int64_t kpo_log_mismatches(const double *x, int64_t n)
{
    int64_t bad = 0;
    for (int64_t i = 0; i < n; i++) {
        double a = kpo_log(x[i]), b = log(x[i]);
        if (as_u64(a) != as_u64(b) && !(isnan(a) && isnan(b))) bad++;
    }
    return bad;
}

void kpo_log_array(const double *x, double *y, int64_t n) { for (int64_t i = 0; i < n; i++) y[i] = kpo_log(x[i]); }
void kpo_log1p_array(const double *x, double *y, int64_t n) { for (int64_t i = 0; i < n; i++) y[i] = kpo_log1p(x[i]); }

/* ------------------------------------------------------------------------------------------- */
/* IUPAC tables                                                                                 */
/* ------------------------------------------------------------------------------------------- */
/* digit order of the sub-letters of each general letter (pattern_utils.py:86-100) */
static const char *perm_of(char g)
{
    switch (g) {
    case 'A': return "A"; case 'C': return "C"; case 'G': return "G"; case 'T': return "T";
    case 'R': return "AGR"; case 'Y': return "CTY"; case 'S': return "GCS";
    case 'W': return "ATW"; case 'K': return "GTK"; case 'M': return "ACM";
    case 'B': return "CGTSYKB"; case 'D': return "AGTRWKD";
    case 'H': return "ACTMWYH"; case 'V': return "ACGMRSV";
    case 'N': return "ACGTRYSWKMBDHVN";
    }
    return NULL;
}
/* two-way splits (c1,c2) of a letter, in scan order (pattern_utils.py:48-57); pairs "c1c2" */
static const char *splits_of(char x)
{
    switch (x) {
    case 'R': return "AG"; case 'Y': return "CT"; case 'S': return "GC";
    case 'W': return "AT"; case 'K': return "GT"; case 'M': return "AC";
    case 'V': return "ASCRGM"; case 'H': return "AYCWTM";
    case 'D': return "AKGWTR"; case 'B': return "CKGYTS";
    case 'N': return "SWKMRYABCDGHTV";
    }
    return "";
}
static int nletters(char x)
{
    switch (x) {
    case 'A': case 'C': case 'G': case 'T': return 1;
    case 'R': case 'Y': case 'S': case 'W': case 'K': case 'M': return 2;
    case 'B': case 'D': case 'H': case 'V': return 3;
    case 'N': return 4;
    }
    return 0;
}

typedef struct {
    int k;
    int radix[KPO_MAXK];
    int nbase[KPO_MAXK];
    uint64_t w[KPO_MAXK + 1];  /* pattern index weights */
    uint64_t kw[KPO_MAXK + 1]; /* k-mer index weights */
    uint8_t lev[KPO_MAXK][15];
    uint8_t nsplit[KPO_MAXK][15];
    int8_t c1[KPO_MAXK][15][7], c2[KPO_MAXK][15][7]; /* child digits */
    char letter[KPO_MAXK][15];
    uint64_t npat, nkmer;
    int total_level;
} kpo_plan;

static int plan_init(kpo_plan *P, const char *gen_pat)
{
    memset(P, 0, sizeof *P);
    int k = (int)strlen(gen_pat);
    if (k < 1 || k > KPO_MAXK) return -1;
    P->k = k;
    uint64_t w = 1, kw = 1;
    for (int i = 0; i < k; i++) {
        const char *perm = perm_of(gen_pat[i]);
        if (!perm) return -2;
        int r = (int)strlen(perm);
        P->radix[i] = r;
        P->nbase[i] = nletters(gen_pat[i]);
        P->w[i] = w;
        P->kw[i] = kw;
        P->total_level += P->nbase[i] - 1;
        for (int d = 0; d < r; d++) {
            char x = perm[d];
            P->letter[i][d] = x;
            P->lev[i][d] = (uint8_t)(nletters(x) - 1);
            const char *sp = splits_of(x);
            int ns = (int)strlen(sp) / 2;
            P->nsplit[i][d] = (uint8_t)ns;
            for (int j = 0; j < ns; j++) {
                const char *p1 = strchr(perm, sp[2 * j]), *p2 = strchr(perm, sp[2 * j + 1]);
                if (!p1 || !p2) return -3;
                P->c1[i][d][j] = (int8_t)(p1 - perm);
                P->c2[i][d][j] = (int8_t)(p2 - perm);
            }
        }
        if (w > UINT64_MAX / (uint64_t)r) return -4;
        w *= (uint64_t)r;
        kw *= (uint64_t)P->nbase[i];
    }
    P->w[k] = w;
    P->kw[k] = kw;
    P->npat = w;
    P->nkmer = kw;
    return 0;
}

int kpo_plan_info(const char *gen_pat, uint64_t *npat, uint64_t *nkmer, int *total_level)
{
    kpo_plan P;
    int rc = plan_init(&P, gen_pat);
    if (rc) return rc;
    *npat = P.npat; *nkmer = P.nkmer; *total_level = P.total_level;
    return 0;
}

/* k-mer index (position 0 fastest, bases in the reference's `code` order) -> pattern index */
static uint64_t kmer_to_pat(const kpo_plan *P, uint64_t kidx)
{
    uint64_t pat = 0;
    for (int i = 0; i < P->k; i++) {
        uint64_t b = kidx % (uint64_t)P->nbase[i];
        kidx /= (uint64_t)P->nbase[i];
        pat += b * P->w[i]; /* singleton letters come first in perm order, same order as `code` */
    }
    return pat;
}

int kpo_kmer_patnums(const char *gen_pat, uint64_t *out)
{
    kpo_plan P;
    int rc = plan_init(&P, gen_pat);
    if (rc) return rc;
    for (uint64_t x = 0; x < P.nkmer; x++) out[x] = kmer_to_pat(&P, x);
    return 0;
}

int kpo_num2pattern(const char *gen_pat, uint64_t num, char *out)
{
    kpo_plan P;
    int rc = plan_init(&P, gen_pat);
    if (rc) return rc;
    for (int i = 0; i < P.k; i++) {
        out[i] = P.letter[i][num % (uint64_t)P.radix[i]];
        num /= (uint64_t)P.radix[i];
    }
    out[P.k] = 0;
    return 0;
}

/* ------------------------------------------------------------------------------------------- */
/* blocking for the parallel sweep                                                              */
/* ------------------------------------------------------------------------------------------- */
typedef struct {
    int hstart;         /* positions >= hstart are "high" (fixed per block) */
    uint64_t bw;        /* patterns per block */
    uint64_t nblocks;
    int nblevels;
    uint64_t *order;    /* block ids sorted by block level */
    uint64_t *lvl_off;  /* nblevels+1 offsets into order */
} kpo_blocks;

static int blocks_init(const kpo_plan *P, kpo_blocks *B)
{
    int h = P->k;
    if (P->npat > (1u << 20)) {
        h = 0;
        for (int i = 0; i < P->k; i++) if (P->w[i] <= (1u << 20)) h = i;
    }
    B->hstart = h;
    B->bw = P->w[h];
    B->nblocks = P->npat / B->bw;
    int maxl = 0;
    for (int i = h; i < P->k; i++) maxl += P->nbase[i] - 1;
    B->nblevels = maxl + 1;
    B->order = (uint64_t *)malloc(sizeof(uint64_t) * B->nblocks);
    B->lvl_off = (uint64_t *)calloc((size_t)B->nblevels + 1, sizeof(uint64_t));
    uint8_t *bl = (uint8_t *)malloc(B->nblocks);
    if (!B->order || !B->lvl_off || !bl) return -1;
    for (uint64_t b = 0; b < B->nblocks; b++) {
        uint64_t x = b; int l = 0;
        for (int i = h; i < P->k; i++) { l += P->lev[i][x % (uint64_t)P->radix[i]]; x /= (uint64_t)P->radix[i]; }
        bl[b] = (uint8_t)l;
        B->lvl_off[l + 1]++;
    }
    for (int l = 0; l < B->nblevels; l++) B->lvl_off[l + 1] += B->lvl_off[l];
    uint64_t *cur = (uint64_t *)malloc(sizeof(uint64_t) * (size_t)B->nblevels);
    memcpy(cur, B->lvl_off, sizeof(uint64_t) * (size_t)B->nblevels);
    for (uint64_t b = 0; b < B->nblocks; b++) B->order[cur[bl[b]]++] = b;
    free(cur); free(bl);
    return 0;
}
static void blocks_free(kpo_blocks *B) { free(B->order); free(B->lvl_off); }

/* ------------------------------------------------------------------------------------------- */
/* single DP  (bottum_up_array_w_numba.py)                                                      */
/* ------------------------------------------------------------------------------------------- */
typedef struct {
    const kpo_plan *P;
    double alpha, beta, penalty;
    float *score;      /* [npat] */
    uint64_t *M, *U;   /* [npat] */
    uint8_t *split;    /* [npat] i*8+j of the winning split, 0xFF = pattern kept whole */
} single_ctx;

static inline double self_score(double alpha, double beta, double penalty, uint64_t M, uint64_t U, double *logp_out, double *log1mp_out)
{
    /* w_numba.py:56-61: p, then s = penalty (+ (-2M)log p) (+ (-2U)log(1-p)); all float64, no FMA */
    double p = ((double)M + alpha) / ((((double)(M + U)) + alpha) + beta);
    double s = penalty;
    double logp = 0.0, log1mp = 0.0;
    if (logp_out) { logp = kpo_log(p); log1mp = kpo_log(1.0 - p); *logp_out = logp; *log1mp_out = log1mp; }
    if (M > 0) { if (!logp_out) logp = kpo_log(p); s = s + ((-2.0 * (double)M) * logp); }
    if (U > 0) { if (!logp_out) log1mp = kpo_log(1.0 - p); s = s + ((-2.0 * (double)U) * log1mp); }
    return s;
}

static void single_block(const single_ctx *C, const kpo_blocks *B, uint64_t block)
{
    const kpo_plan *P = C->P;
    int k = P->k;
    int dig[KPO_MAXK];
    uint64_t base = block * B->bw;
    { uint64_t x = base; for (int i = 0; i < k; i++) { dig[i] = (int)(x % (uint64_t)P->radix[i]); x /= (uint64_t)P->radix[i]; } }
    for (uint64_t off = 0; off < B->bw; off++) {
        uint64_t pat = base + off;
        int level = 0;
        for (int i = 0; i < k; i++) level += P->lev[i][dig[i]];
        if (level > 0) {
            float best = INFINITY;
            uint8_t code = 0xFF;
            int first = 1;
            for (int i = 0; i < k; i++) {
                int d = dig[i];
                int ns = P->nsplit[i][d];
                for (int j = 0; j < ns; j++) {
                    uint64_t p1 = pat - (uint64_t)(d - P->c1[i][d][j]) * P->w[i];
                    uint64_t p2 = pat - (uint64_t)(d - P->c2[i][d][j]) * P->w[i];
                    float cand = C->score[p1] + C->score[p2];          /* float32 add (w_numba.py:46) */
                    if (cand < best) { best = cand; code = (uint8_t)(i * 8 + j); }
                    if (first) { C->M[pat] = C->M[p1] + C->M[p2]; C->U[pat] = C->U[p1] + C->U[p2]; first = 0; }
                }
            }
            double s = self_score(C->alpha, C->beta, C->penalty, C->M[pat], C->U[pat], NULL, NULL);
            if (s < (double)best) { best = (float)s; code = 0xFF; }  /* float64 compare, float32 store (:62-63) */
            C->score[pat] = best;
            C->split[pat] = code;
        }
        /* odometer */
        for (int i = 0; i < k; i++) { if (++dig[i] < P->radix[i]) break; dig[i] = 0; }
    }
}

/* level-0 score, w_numba.py:26-29 (Python floats + scipy) */
double kpo_leaf_score(double alpha, double beta, double penalty, uint64_t M, uint64_t U)
{
    double p = ((double)M + alpha) / ((((double)(M + U)) + alpha) + beta);
    return -2.0 * (kpo_xlogy((double)M, p) + kpo_xlog1py((double)U, -p)) + penalty;
}

/* level >= 1 self-score of n items (w_numba.py:56-61), each with its own alpha, beta and penalty */
void kpo_self_score_array(const double *alpha, const double *beta, const double *penalty, const uint64_t *M, const uint64_t *U,
                          double *out, int64_t n)
{
    for (int64_t i = 0; i < n; i++) out[i] = self_score(alpha[i], beta[i], penalty[i], M[i], U[i], NULL, NULL);
}

/*
 * kmerM/kmerU: counts per k-mer in k-mer index order.  leaf_score: optional level-0 scores
 * (float32, k-mer index order) computed by the caller with scipy; NULL -> kpo_leaf_score().
 * Outputs are full tables in the reference's dense numbering.
 */
int kpo_single_dp(const char *gen_pat, const uint64_t *kmerM, const uint64_t *kmerU, const float *leaf_score,
                  double alpha, double beta, double penalty,
                  float *score, uint64_t *M, uint64_t *U, uint8_t *split, int nthreads)
{
    kpo_plan P;
    int rc = plan_init(&P, gen_pat);
    if (rc) return rc;
    kpo_blocks B;
    if (blocks_init(&P, &B)) return -10;
    for (uint64_t x = 0; x < P.nkmer; x++) {
        uint64_t pat = kmer_to_pat(&P, x);
        M[pat] = kmerM[x]; U[pat] = kmerU[x];
        score[pat] = leaf_score ? leaf_score[x] : (float)kpo_leaf_score(alpha, beta, penalty, kmerM[x], kmerU[x]);
        split[pat] = 0xFF;
    }
    single_ctx C = { &P, alpha, beta, penalty, score, M, U, split };
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
    for (int l = 0; l < B.nblevels; l++) {
        int64_t lo = (int64_t)B.lvl_off[l], hi = (int64_t)B.lvl_off[l + 1];
#pragma omp parallel for schedule(dynamic, 1)
        for (int64_t t = lo; t < hi; t++) single_block(&C, &B, B.order[t]);
    }
    blocks_free(&B);
    return 0;
}

/* backtrack (w_numba.py:17-24): DFS, c1 subtree first; writes dense indices of the partition */
int64_t kpo_backtrack(const char *gen_pat, const uint8_t *split, uint64_t *out, int64_t cap)
{
    kpo_plan P;
    if (plan_init(&P, gen_pat)) return -1;
    int64_t n = 0, sp = 0, scap = 1024;
    uint64_t *stack = (uint64_t *)malloc(sizeof(uint64_t) * (size_t)scap);
    stack[sp++] = P.npat - 1;
    while (sp > 0) {
        uint64_t pat = stack[--sp];
        uint8_t code = split[pat];
        if (code == 0xFF) { if (n < cap) out[n] = pat; n++; continue; }
        int i = code >> 3, j = code & 7;
        int d = (int)((pat / P.w[i]) % (uint64_t)P.radix[i]);
        uint64_t p1 = pat - (uint64_t)(d - P.c1[i][d][j]) * P.w[i];
        uint64_t p2 = pat - (uint64_t)(d - P.c2[i][d][j]) * P.w[i];
        if (sp + 2 > scap) { scap *= 2; stack = (uint64_t *)realloc(stack, sizeof(uint64_t) * (size_t)scap); }
        stack[sp++] = p2; /* right child popped after the whole left subtree */
        stack[sp++] = p1;
    }
    free(stack);
    return n;
}

/* ------------------------------------------------------------------------------------------- */
/* CV, one fold = one job  (bottum_up_array_penalty_plus_pseudo_CV.py)                          */
/* ------------------------------------------------------------------------------------------- */
typedef struct {
    const kpo_plan *P;
    double alpha, beta, penalty;
    float *train, *test;          /* [npat] */
    uint64_t *Mtr, *Utr, *Mte, *Ute; /* [npat] train and held-out counts */
} cv_ctx;

static void cv_block(const cv_ctx *C, const kpo_blocks *B, uint64_t block)
{
    const kpo_plan *P = C->P;
    int k = P->k;
    int dig[KPO_MAXK];
    uint64_t base = block * B->bw;
    { uint64_t x = base; for (int i = 0; i < k; i++) { dig[i] = (int)(x % (uint64_t)P->radix[i]); x /= (uint64_t)P->radix[i]; } }
    for (uint64_t off = 0; off < B->bw; off++) {
        uint64_t pat = base + off;
        int level = 0;
        for (int i = 0; i < k; i++) level += P->lev[i][dig[i]];
        if (level > 0) {
            float btrain = INFINITY, btest = 0.0f; /* test_score_mem is np.empty; only read after a win */
            int first = 1;
            for (int i = 0; i < k; i++) {
                int d = dig[i];
                int ns = P->nsplit[i][d];
                for (int j = 0; j < ns; j++) {
                    uint64_t p1 = pat - (uint64_t)(d - P->c1[i][d][j]) * P->w[i];
                    uint64_t p2 = pat - (uint64_t)(d - P->c2[i][d][j]) * P->w[i];
                    float ntrain = C->train[p1] + C->train[p2];
                    float ntest = C->test[p1] + C->test[p2];
                    if (ntrain < btrain) { btrain = ntrain; btest = ntest; }   /* _CV.py:48-51 */
                    if (first) {
                        /* held-out rows add; train = sum over folds - held-out is linear, so it adds too */
                        C->Mte[pat] = C->Mte[p1] + C->Mte[p2]; C->Ute[pat] = C->Ute[p1] + C->Ute[p2];
                        C->Mtr[pat] = C->Mtr[p1] + C->Mtr[p2]; C->Utr[pat] = C->Utr[p1] + C->Utr[p2];
                        first = 0;
                    }
                }
            }
            double logp, log1mp;
            double s = self_score(C->alpha, C->beta, C->penalty, C->Mtr[pat], C->Utr[pat], &logp, &log1mp);
            if (s < (double)btrain) {                                          /* _CV.py:71-78 */
                btrain = (float)s;
                double t = 0.0;
                if (C->Mte[pat] > 0) t = t + ((-2.0 * (double)C->Mte[pat]) * logp);
                if (C->Ute[pat] > 0) t = t + ((-2.0 * (double)C->Ute[pat]) * log1mp);
                btest = (float)t;
            }
            C->train[pat] = btrain;
            C->test[pat] = btest;
        }
        for (int i = 0; i < k; i++) { if (++dig[i] < P->radix[i]) break; dig[i] = 0; }
    }
}

/* level 0 of one fold, _CV.py:15-20 */
void kpo_cv_leaf(double alpha, double beta, double penalty, uint64_t Mtr, uint64_t Utr, uint64_t Mte, uint64_t Ute,
                 double *train, double *test)
{
    double p = ((double)Mtr + alpha) / ((((double)(Mtr + Utr)) + alpha) + beta);
    *train = -2.0 * (kpo_xlogy((double)Mtr, p) + kpo_xlog1py((double)Utr, -p)) + penalty;
    *test = -2.0 * (kpo_xlogy((double)Mte, p) + kpo_xlog1py((double)Ute, -p));
}

/*
 * One (fold, alpha, penalty) job.  kmerMtot/kmerUtot: all-fold totals per k-mer; kmerMte/kmerUte:
 * this fold's held-out counts per k-mer.  leaf_train/leaf_test: optional float32 level-0 values
 * from scipy (k-mer order).  train/test: full float32 tables out; work arrays are allocated here.
 */
int kpo_cv_job(const char *gen_pat, const uint64_t *kmerMtot, const uint64_t *kmerUtot,
               const uint64_t *kmerMte, const uint64_t *kmerUte,
               const float *leaf_train, const float *leaf_test,
               double alpha, double beta, double penalty, float *train, float *test, int nthreads)
{
    kpo_plan P;
    int rc = plan_init(&P, gen_pat);
    if (rc) return rc;
    kpo_blocks B;
    if (blocks_init(&P, &B)) return -10;
    uint64_t *cnt = (uint64_t *)malloc(sizeof(uint64_t) * 4 * P.npat);
    if (!cnt) { blocks_free(&B); return -11; }
    cv_ctx C = { &P, alpha, beta, penalty, train, test, cnt, cnt + P.npat, cnt + 2 * P.npat, cnt + 3 * P.npat };
    for (uint64_t x = 0; x < P.nkmer; x++) {
        uint64_t pat = kmer_to_pat(&P, x);
        C.Mte[pat] = kmerMte[x]; C.Ute[pat] = kmerUte[x];
        C.Mtr[pat] = kmerMtot[x] - kmerMte[x]; C.Utr[pat] = kmerUtot[x] - kmerUte[x];
        if (leaf_train) { train[pat] = leaf_train[x]; test[pat] = leaf_test[x]; }
        else {
            double a, b;
            kpo_cv_leaf(alpha, beta, penalty, C.Mtr[pat], C.Utr[pat], C.Mte[pat], C.Ute[pat], &a, &b);
            train[pat] = (float)a; test[pat] = (float)b;
        }
    }
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
    for (int l = 0; l < B.nblevels; l++) {
        int64_t lo = (int64_t)B.lvl_off[l], hi = (int64_t)B.lvl_off[l + 1];
#pragma omp parallel for schedule(dynamic, 1)
        for (int64_t t = lo; t < hi; t++) cv_block(&C, &B, B.order[t]);
    }
    free(cnt);
    blocks_free(&B);
    return 0;
}

int kpo_max_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
